"""BASELINE config 4: end-to-end MI training step with the critic / loss swapped for the fused kernels.

Mirrors the loop body of ``MultiModalManager.train`` (mutual_info_img_txt/main_utils.py:184-236) on
synthetic data: a 6-stage residual image encoder on 1x256x256 inputs (768-d embedding, the shape of
``ResNet256_6_2_1``, model.py:272-370), a BERT-base text encoder over 128-token ids (pooled output +
dropout, model.py:54-105; ``transformers.BertModel``, random init — no checkpoint, no network), three
optimizers as main_utils.py:152-172, and the three-call critic sequence (main_utils.py:220-226).
The encoders are stand-ins of the reference's shapes (they are out of scope, SURVEY 2 rows 5-7); the
point is the critic slot:

    --critic fused   mi_b200.FusedCritic + dv_bound_loss on the PairBatch handle  (this repo)
    --critic mlp     mi_b200.FusedMLPCritic(768, (1024, 512)): the reference's OWN mi_discriminator (main_utils.py:77), fused
    --critic mlp_pairs  the same nn.Sequential on the explicit pair tensor (what the reference executes, torch ops)
    --critic mlp_sharded  FusedMLPCritic through sharded_mi_loss: at N > 1 the loss of the GLOBAL batch (every rank's rows
                     against every rank's texts), not per-rank batches
    --critic pairs   the same separable critic on the explicit [B + N_neg, 2D] pair tensor (torch ops;
                     the reference's formulation with the O(B^2) loop replaced by one gather)

    python examples/train_step_config4.py --critic fused --batch 256 --steps 5
    torchrun --nproc-per-node N examples/train_step_config4.py ...      # DDP encoders + sharded critic
"""
import argparse
import os
import sys
import time

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mi_b200  # noqa: E402


class Block(nn.Module):
    def __init__(self, cin, cout, stride):
        super().__init__()
        self.c1 = nn.Conv2d(cin, cout, 3, stride, 1, bias=False)
        self.b1 = nn.BatchNorm2d(cout)
        self.c2 = nn.Conv2d(cout, cout, 3, 1, 1, bias=False)
        self.b2 = nn.BatchNorm2d(cout)
        self.down = None
        if stride != 1 or cin != cout:
            self.down = nn.Sequential(nn.Conv2d(cin, cout, 1, stride, bias=False), nn.BatchNorm2d(cout))

    def forward(self, x):
        idt = x if self.down is None else self.down(x)
        y = torch.relu(self.b1(self.c1(x)))
        return torch.relu(self.b2(self.c2(y)) + idt)


class ImageEncoder(nn.Module):
    """1x256x256 -> 768: stem 8 ch, six stride-2 stages (8,16,32,64,128,192), 2x2 average pool."""

    def __init__(self, blocks=(2, 2, 2, 2, 2, 2)):
        super().__init__()
        self.stem = nn.Sequential(nn.Conv2d(1, 8, 3, 1, 1, bias=False), nn.BatchNorm2d(8), nn.ReLU())
        chans, layers, cin = (8, 16, 32, 64, 128, 192), [], 8
        for c, n in zip(chans, blocks):
            for k in range(n):
                layers.append(Block(cin, c, 2 if k == 0 else 1))
                cin = c
        self.body = nn.Sequential(*layers)
        self.pool = nn.AvgPool2d(2)

    def forward(self, x):
        return torch.flatten(self.pool(self.body(self.stem(x))), 1)


class TextEncoder(nn.Module):
    def __init__(self, layers=12):
        super().__init__()
        from transformers import BertConfig, BertModel
        self.bert = BertModel(BertConfig(num_hidden_layers=layers))
        self.drop = nn.Dropout(0.1)

    def forward(self, ids, mask, seg):
        return self.drop(self.bert(input_ids=ids, attention_mask=mask, token_type_ids=seg).pooler_output)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--critic", default="fused", choices=["fused", "pairs", "mlp", "mlp_pairs", "mlp_sharded"])
    ap.add_argument("--estimator", default="dv")
    ap.add_argument("--batch", type=int, default=256, help="per GPU")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--seq", type=int, default=128)
    ap.add_argument("--bert-layers", type=int, default=12)
    ap.add_argument("--throughput-steps", type=int, default=10,
                    help="after the instrumented steps: this many steps WITHOUT any host synchronisation inside the step "
                         "(the loss of step n is read while step n+1 runs: deferred logging instead of main_utils.py:233's "
                         "per-step .item())")
    a = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)
    img_enc, txt_enc = ImageEncoder().to(dev), TextEncoder(a.bert_layers).to(dev)
    if a.critic in ("mlp", "mlp_pairs", "mlp_sharded"):             # the mi_discriminator slot (main_utils.py:77)
        critic = mi_b200.FusedMLPCritic(768, (1024, 512), precision="fast").to(dev)
    else:
        critic = mi_b200.FusedCritic(768, "bilinear").to(dev)
    if world > 1:
        from torch.nn.parallel import DistributedDataParallel as DDP
        img_enc, txt_enc = DDP(img_enc, device_ids=[local]), DDP(txt_enc, device_ids=[local])
    img_opt = torch.optim.Adam(img_enc.parameters(), lr=1e-4)       # main_utils.py:152-153
    mi_opt = torch.optim.Adam(critic.parameters(), lr=1e-4)
    txt_opt = torch.optim.AdamW(txt_enc.parameters(), lr=1e-4)      # main_utils.py:166-168
    sched = torch.optim.lr_scheduler.LambdaLR(txt_opt, lambda s: min(1.0, (s + 1) / 10))
    mi_critic = mi_b200.select_estimator(a.estimator)               # main_utils.py:141-144
    B = a.batch
    g = torch.Generator().manual_seed(1 + rank)
    times, crit_times = [], []
    for step in range(a.steps + 2):
        img = torch.rand(B, 1, 256, 256, generator=g).to(dev)
        ids = torch.randint(1000, 30000, (B, a.seq), generator=g).to(dev)
        mask, seg = torch.ones_like(ids), torch.zeros_like(ids)
        study = torch.arange(B) + rank * B
        study[1::16] = study[0::16][: len(study[1::16])]              # some studies have two images
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        img_opt.zero_grad(); txt_opt.zero_grad(); mi_opt.zero_grad()
        emb_img, emb_txt = img_enc(img), txt_enc(ids, mask, seg)     # main_utils.py:218-219
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        if world > 1 and a.critic in ("fused", "pairs", "mlp_sharded"):     # global batch over the ranks (both critics)
            loss = mi_b200.sharded_mi_loss(emb_img, emb_txt, critic, study, a.estimator)
        elif a.critic in ("fused", "mlp", "mlp_sharded"):             # (N > 1 with --critic mlp: per-rank batches, as the reference's DDP)
            mi_input = mi_b200.create_mi_pairs(emb_img, emb_txt, study.tolist(), dev)      # :220-221
            loss = mi_critic(critic(mi_input), B, dev)                                     # :222-224
        else:
            mi_input = mi_b200.create_mi_pairs_tensor(emb_img, emb_txt, study.tolist(), dev)
            loss = mi_critic(critic(mi_input), B, dev)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        loss.sum().backward()                                        # :226
        mi_opt.step(); img_opt.step(); txt_opt.step(); sched.step()  # :227-230
        lv = loss.sum().item()                                       # :233
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        if step >= 2:
            times.append(t3 - t0); crit_times.append(t2 - t1)
        if rank == 0:
            print(f"step {step}: loss {lv:.5f}  step {1e3 * (t3 - t0):.1f} ms  (encoders fwd {1e3 * (t1 - t0):.1f}, "
                  f"critic+loss fwd(+fused bwd) {1e3 * (t2 - t1):.2f})", flush=True)
    # ---- throughput: the same step with NO host synchronisation inside it (SURVEY 8f-4: the reference's three per-step syncs —
    # mi_critics.py:10 H2D of log N, main_utils.py:233 loss.item(), and the adapter's optional no-negatives check — are gone;
    # the sharded critic's only host read is its guard count, which waits for the score tiles, not for the step)
    tput = None
    if a.throughput_steps > 0:
        critic.check_negatives = False
        img = torch.rand(B, 1, 256, 256, generator=g).to(dev)
        ids = torch.randint(1000, 30000, (B, a.seq), generator=g).to(dev)
        mask, seg = torch.ones_like(ids), torch.zeros_like(ids)
        study = torch.arange(B) + rank * B
        study_list = study.tolist()
        pending, logged = None, []
        loss_pin = [torch.zeros(1).pin_memory() for _ in range(2)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for step in range(a.throughput_steps):
            img_opt.zero_grad(); txt_opt.zero_grad(); mi_opt.zero_grad()
            emb_img, emb_txt = img_enc(img), txt_enc(ids, mask, seg)
            if world > 1 and a.critic in ("fused", "pairs", "mlp_sharded"):
                loss = mi_b200.sharded_mi_loss(emb_img, emb_txt, critic, study, a.estimator)
            elif a.critic in ("fused", "mlp", "mlp_sharded"):
                loss = mi_critic(critic(mi_b200.create_mi_pairs(emb_img, emb_txt, study_list, dev)), B, dev)
            else:
                loss = mi_critic(critic(mi_b200.create_mi_pairs_tensor(emb_img, emb_txt, study_list, dev)), B, dev)
            loss.sum().backward()
            mi_opt.step(); img_opt.step(); txt_opt.step(); sched.step()
            if pending is not None:                      # the PREVIOUS step's loss: (nearly) there already, no stall of this step
                pending[1].synchronize()
                logged.append(float(pending[0]))
            slot = loss_pin[step & 1]
            slot.copy_(loss.detach().reshape(-1)[:1], non_blocking=True)
            ev = torch.cuda.Event(); ev.record()
            pending = (slot, ev)
        torch.cuda.synchronize()
        tput = (time.perf_counter() - t0) / a.throughput_steps
    if rank == 0:
        print(f"RESULT critic={a.critic} world={world} batch/gpu={B} global_pairs={(B * world) ** 2} "
              f"step_ms={1e3 * sum(times) / len(times):.1f} critic_ms={1e3 * sum(crit_times) / len(crit_times):.2f} "
              f"samples/s={B * world * len(times) / sum(times):.0f}"
              + ("" if tput is None else f"  | no-sync loop: step_ms={1e3 * tput:.1f} samples/s={B * world / tput:.0f}"), flush=True)


if __name__ == "__main__":
    main()
