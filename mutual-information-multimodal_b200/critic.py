"""Host-side mirror of the reference's critic / loss API.

The reference's hot path is three calls inside ``MultiModalManager.train``
(mutual_info_img_txt/main_utils.py:220-226)::

    mi_input  = self.create_mi_pairs(embedding_img, embedding_txt, study_id, device)
    mi_output = self.mi_discriminator(mi_input)
    loss      = mi_critic(mi_output, args.batch_size, device)     # dv_bound_loss | infonce_bound_loss
    loss.backward()

The same three calls work here with the same names, argument meaning and result shapes, but nothing
B^2-sized is ever built on the host side:

* ``create_mi_pairs`` returns a ``PairBatch`` handle (embeddings + study ids) instead of the
  ``[B + N_neg, 2D]`` tensor of main_utils.py:93-108;
* ``FusedCritic`` (an ``nn.Module`` that owns ``W`` / the temperature, so ``.parameters()`` and
  ``.to(device)`` behave like the ``make_mlp`` critic of main_utils.py:77) maps it to a ``ScoreHandle``;
* ``dv_bound_loss`` / ``infonce_bound_loss`` (mi_critics.py:3-12, :14-23) accept that handle and
  launch the fused CUDA path (forward statistics + gradient passes) through the C ABI; gradients
  reach ``embedding_img`` / ``embedding_txt`` / ``W`` through a ``torch.autograd.Function``.

Passing a plain logits tensor to the loss functions keeps the reference's exact tensor semantics
(for critics that are not fused, e.g. the original MLP).
"""
from __future__ import annotations

import math
from typing import Optional, Sequence, Union

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops


def _dense_ids(study_id) -> torch.Tensor:
    """Exact study_id -> dense int32 (equal ids <=> equal codes); main_utils.py:105 compares the
    ids for inequality only, so any injective relabelling preserves the mask."""
    if torch.is_tensor(study_id):
        if study_id.dtype in (torch.int32,) and study_id.dim() == 1:
            return study_id
        _, inv = torch.unique(study_id.reshape(-1), return_inverse=True)
        return inv.to(torch.int32)
    table = {}
    return torch.tensor([table.setdefault(s, len(table)) for s in study_id], dtype=torch.int32)


class PairBatch:
    """What ``create_mi_pairs`` returns: the batch of image / text embeddings and their study ids.
    Positives are the B matched rows, negatives every (i, j), i != j, study_id[i] != study_id[j]
    (main_utils.py:93-108) — enumerated by index arithmetic inside the kernels, never stored."""

    def __init__(self, embedding_img: torch.Tensor, embedding_txt: torch.Tensor, sid: torch.Tensor):
        if embedding_img.shape != embedding_txt.shape or embedding_img.dim() != 2:
            raise ValueError("embedding_img and embedding_txt must both be [B, D]")
        if sid.numel() != embedding_img.shape[0]:
            raise ValueError("len(study_id) must equal the batch size")
        self.embedding_img = embedding_img
        self.embedding_txt = embedding_txt
        self.sid = sid

    @property
    def batch_size(self) -> int:
        return self.embedding_img.shape[0]

    def __len__(self) -> int:      # the reference's pair tensor has B + N_neg rows; we only know B cheaply
        return self.batch_size


def create_mi_pairs(embedding_img: torch.Tensor, embedding_txt: torch.Tensor,
                    study_id: Union[Sequence, torch.Tensor], device=None) -> PairBatch:
    """Drop-in for ``MultiModalManager.create_mi_pairs`` (main_utils.py:80-110)."""
    sid = _dense_ids(study_id)
    dev = embedding_img.device if device is None else torch.device(device)
    return PairBatch(embedding_img, embedding_txt, sid.to(dev, non_blocking=True))


def create_mi_pairs_tensor(embedding_img: torch.Tensor, embedding_txt: torch.Tensor,
                           study_id: Union[Sequence, torch.Tensor], device=None) -> torch.Tensor:
    """The reference's explicit ``[B + N_neg, 2D]`` pair tensor in the reference's row order
    (main_utils.py:93-108: B matched rows, then gap-major negatives (i, (i+gap+1) mod B) with different
    study ids) built by index arithmetic and ONE gather instead of the O(B^2) ``torch.cat`` loop
    (SURVEY 8f-2).  For critics that are not fused (e.g. the original ``make_mlp``) at small B; differentiable."""
    B = embedding_img.shape[0]
    dev = embedding_img.device
    sid = _dense_ids(study_id).to(dev)
    pos = torch.cat((embedding_img, embedding_txt), 1)
    if B < 2:
        return pos
    i = torch.arange(B, device=dev).expand(B - 1, B)
    j = (i + torch.arange(1, B, device=dev)[:, None]) % B
    keep = (sid[i] != sid[j]).reshape(-1)
    ii, jj = i.reshape(-1)[keep], j.reshape(-1)[keep]
    return torch.cat((pos, torch.cat((embedding_img[ii], embedding_txt[jj]), 1)), 0)


class ScoreHandle:
    """Lazy stand-in for the ``[N, 1]`` logits tensor (``mi_output``, main_utils.py:222)."""

    def __init__(self, pairs: PairBatch, critic):
        self.pairs = pairs
        self.critic = critic

    @property
    def shape(self):
        return (self.pairs.batch_size,)


class _FusedCriticLoss(torch.autograd.Function):
    """loss = estimator(S), S = inv_tau * X W Y^T — forward statistics and the gradient passes run
    in one call (gradients are produced with the loss, scaled by grad_output in backward)."""

    @staticmethod
    def forward(ctx, X, Y, W, sid, estimator, precision, inv_tau, check_negatives):
        need = any(t is not None and t.requires_grad for t in (X, Y, W))
        # (a tripped single-pass guard is handled INSIDE the library: exact repeat behind a device-side predicate)
        out, dX, dY, dW = ops.critic_loss_fwd_bwd(X, Y, W, sid, estimator, precision, inv_tau, need_grads=need)
        if check_negatives and float(out[3].item()) == 0.0:
            # one host sync, opt-out with check_negatives=False (then the loss is nan / -inf like the reference's:
            # dv -> tensor([nan]), infonce -> tensor(-inf), mi_critics.py:9-10 with no negatives)
            raise ops.MIError("no negative pairs in the batch (every study_id is equal): the reference "
                              "returns nan (dv) / -inf (infonce) here; the fused path refuses instead")
        ctx.grads = (dX, dY, dW)
        ctx.dtypes = (X.dtype, Y.dtype, None if W is None else W.dtype)
        ctx.stats = out
        return out[0].to(torch.float32)

    @staticmethod
    def backward(ctx, grad_out):
        dX, dY, dW = ctx.grads
        tx, ty, tw = ctx.dtypes
        g = grad_out.to(torch.float32)
        gx = None if dX is None else (dX * g).to(tx)
        gy = None if dY is None else (dY * g).to(ty)
        gw = None if dW is None else (dW * g).to(tw)
        return gx, gy, gw, None, None, None, None, None


class _ShardedFusedCriticLoss(torch.autograd.Function):
    """Data-parallel form: every rank passes its row shard; the loss is the GLOBAL-batch estimator
    (identical on all ranks), gradients are returned for the local rows and dW is already summed."""

    @staticmethod
    def forward(ctx, X, Y, W, sid, estimator, precision, inv_tau, group, grad_scale):
        from . import dist as mdist
        need = any(t is not None and t.requires_grad for t in (X, Y, W))
        out, dX, dY, dW = mdist.sharded_critic_loss_fwd_bwd(X, Y, W, sid, estimator, precision, inv_tau,
                                                           need_grads=need, group=group)
        ctx.grads = (dX, dY, dW)
        ctx.dtypes = (X.dtype, Y.dtype, None if W is None else W.dtype)
        ctx.grad_scale = grad_scale
        ctx.stats = out
        return out["loss"].to(torch.float32)

    @staticmethod
    def backward(ctx, grad_out):
        dX, dY, dW = ctx.grads
        tx, ty, tw = ctx.dtypes
        g = grad_out.to(torch.float32)
        ge = g * ctx.grad_scale          # encoder grads: DDP averages over ranks, the global loss needs the sum
        gx = None if dX is None else (dX * ge).to(tx)
        gy = None if dY is None else (dY * ge).to(ty)
        gw = None if dW is None else (dW * g).to(tw)
        return gx, gy, gw, None, None, None, None, None, None


class _ShardedFusedMLPCriticLoss(torch.autograd.Function):
    """Data-parallel form of the concat-MLP critic: every rank passes its row shard; the loss is the GLOBAL-batch
    estimator (identical on all ranks), embedding gradients are those of the local rows, the six parameter gradients are
    already summed over ranks (the gradient of the global loss)."""

    @staticmethod
    def forward(ctx, X, Y, W1, b1, W2, b2, W3, b3, sid, estimator, precision, group, grad_scale):
        from . import dist as mdist
        tensors = (X, Y, W1, b1, W2, b2, W3, b3)
        need = any(t.requires_grad for t in tensors)
        out, dX, dY, grads = mdist.sharded_mlp_critic_loss_fwd_bwd(X, Y, (W1, b1, W2, b2, W3, b3), sid, estimator, precision,
                                                                   need_grads=need, group=group)
        ctx.grads = None if dX is None else (dX, dY) + tuple(grads[n] for n in mdist.MLP_GRAD_NAMES)
        ctx.dtypes = tuple(t.dtype for t in tensors)
        ctx.grad_scale = grad_scale
        ctx.stats = out
        return out["loss"].to(torch.float32)

    @staticmethod
    def backward(ctx, grad_out):
        if ctx.grads is None:
            return (None,) * 13
        g = grad_out.to(torch.float32)
        ge = g * ctx.grad_scale          # encoder grads: DDP averages over ranks, the global loss needs the sum
        scales = (ge, ge) + (g,) * 6
        outs = tuple((t * s).to(dt) for t, s, dt in zip(ctx.grads, scales, ctx.dtypes))
        return outs + (None,) * 5


def sharded_mi_loss(embedding_img, embedding_txt, critic: "FusedCritic", study_id, estimator: str = "dv",
                    group=None, ddp_mean_correction: bool = True) -> torch.Tensor:
    """Global-batch MI loss when every rank holds a row shard of the batch (SURVEY 8e / 8f-4).
    ``study_id`` is this rank's integer id tensor (raw int64 ids are relabelled consistently across ranks).
    With ``ddp_mean_correction`` the embedding gradients are multiplied by the world size so that
    DistributedDataParallel's gradient averaging of the encoders yields the gradient of the global loss; parameter
    gradients are those of the global loss, not scaled.  ``critic`` is a ``FusedCritic`` or a ``FusedMLPCritic``."""
    import torch.distributed as tdist
    ops.reject_separable_only(estimator, "the batch-sharded loss")
    world = tdist.get_world_size(group) if tdist.is_available() and tdist.is_initialized() else 1
    sid = study_id if torch.is_tensor(study_id) else torch.tensor([int(s) for s in study_id], dtype=torch.int64)
    sid = sid.to(embedding_img.device)
    scale = float(world) if ddp_mean_correction else 1.0
    if isinstance(critic, FusedMLPCritic):
        c = critic
        return _ShardedFusedMLPCriticLoss.apply(embedding_img, embedding_txt, c[0].weight, c[0].bias, c[2].weight, c[2].bias,
                                                c[4].weight, c[4].bias, sid, estimator, c.precision, group, scale)
    return _ShardedFusedCriticLoss.apply(embedding_img, embedding_txt, critic.W, sid, estimator, critic.precision,
                                         critic.inv_tau, group, scale)


class FusedCritic(nn.Module):
    """Separable critic f(x, y) = inv_tau * x^T W y in the ``mi_discriminator`` slot
    (main_utils.py:77,222).  ``critic='dot'`` has no parameters (W = I); ``'bilinear'`` owns W [D, D].

    Called with a ``PairBatch`` it returns a ``ScoreHandle`` (fused path).  Called with an explicit
    ``[N, 2D]`` pair tensor (the reference's ``mi_input``) it evaluates the same critic row by row with
    torch ops and returns ``[N, 1]`` logits — the compatibility path for small batches.

    The fused loss call never synchronises with the host (the reference adds two syncs per step on this path:
    mi_critics.py:10 and main_utils.py:233).  A batch without any negative pair gives ``nan`` (dv) / ``-inf`` (infonce)
    exactly like the reference; ``check_negatives=True`` turns that into an ``MIError`` at the price of one host read.
    """

    def __init__(self, dim: int, critic: str = "bilinear", temperature: Optional[float] = None,
                 precision: str = "fast", check_negatives: bool = False):
        super().__init__()
        if critic not in ("dot", "bilinear"):
            raise ValueError("critic must be 'dot' or 'bilinear'")
        ops._precision(precision)          # "fast" / "strict" ("fp32" is the MLP critic's only): raises before any launch
        self.dim = dim
        self.critic = critic
        self.precision = precision
        self.check_negatives = check_negatives
        self.inv_tau = 1.0 / (temperature if temperature is not None else (math.sqrt(dim) if critic == "dot" else 1.0))
        if critic == "bilinear":
            w = torch.eye(dim) / math.sqrt(dim)
            self.W = nn.Parameter(w)
        else:
            self.register_parameter("W", None)

    def forward(self, mi_input):
        if isinstance(mi_input, PairBatch):
            return ScoreHandle(mi_input, self)
        rows = mi_input
        D = self.dim
        t = rows[:, :D] if self.W is None else rows[:, :D] @ self.W.to(rows.dtype)
        return (t * rows[:, D:]).sum(1, keepdim=True) * self.inv_tau


class _FusedMLPCriticLoss(torch.autograd.Function):
    """loss = estimator(S), S[i,j] = make_mlp(2D,[H1,H2])([x_i ; y_j]) for every pair — one library call
    produces the loss and the gradients of both embeddings and all six MLP tensors."""

    @staticmethod
    def forward(ctx, X, Y, W1, b1, W2, b2, W3, b3, sid, estimator, precision, check_negatives):
        tensors = (X, Y, W1, b1, W2, b2, W3, b3)
        need = any(t.requires_grad for t in tensors)
        out, _, grads = ops.mlp_critic_loss_fwd_bwd(X, Y, (W1, b1, W2, b2, W3, b3), sid, estimator, precision, need_grads=need)
        if check_negatives and float(out.cpu()[3]) == 0.0:
            raise ops.MIError("no negative pairs in the batch (every study_id is equal): the reference "
                              "returns nan (dv) / -inf (infonce) here; the fused path refuses instead")
        ctx.grads = grads
        ctx.dtypes = tuple(t.dtype for t in tensors)
        ctx.stats = out
        return out[0].to(torch.float32)

    @staticmethod
    def backward(ctx, grad_out):
        g = grad_out.to(torch.float32)
        if ctx.grads is None:
            return (None,) * 12
        names = ("dX", "dY", "dW1", "db1", "dW2", "db2", "dW3", "db3")
        outs = tuple((ctx.grads[n] * g).to(dt) for n, dt in zip(names, ctx.dtypes))
        return outs + (None, None, None, None)


class FusedMLPCritic(nn.Sequential):
    """The reference's own critic, ``make_mlp(2 * dim, hidden_dims)`` (model.py:18-32; main_utils.py:77 builds
    ``make_mlp(1536, [1024, 512])``), as a drop-in for the ``mi_discriminator`` slot: the SAME ``nn.Sequential``
    (``Linear, ReLU, Linear, ReLU, Linear`` — identical parameter names ``0.weight … 4.bias``, identical default
    initialisation, so a reference checkpoint loads with ``load_state_dict``).

    Called with the explicit ``[N, 2D]`` pair tensor it IS the reference module (torch ops).  Called with a
    ``PairBatch`` (what this package's ``create_mi_pairs`` returns) it yields a ``ScoreHandle`` and the loss
    functions run the fused CUDA path: layer 1 is evaluated once per image and once per text
    (``W1 [x;y] = W1x x + W1y y``), layers 2-3 on tensor cores for all B^2 pairs, the pair tensor is never built."""

    def __init__(self, dim: int = 768, hidden_dims=(1024, 512), precision: str = "strict", check_negatives: bool = False):
        if len(hidden_dims) != 2:
            raise ValueError("the fused path implements the reference's two-hidden-layer critic")
        h1, h2 = int(hidden_dims[0]), int(hidden_dims[1])
        ops._mlp_precision(precision)      # "fast", "strict" or "fp32" (three bf16 pieces per operand)
        super().__init__(nn.Linear(2 * dim, h1), nn.ReLU(), nn.Linear(h1, h2), nn.ReLU(), nn.Linear(h2, 1))
        self.dim = dim
        self.precision = precision
        self.check_negatives = check_negatives

    def forward(self, mi_input):
        if isinstance(mi_input, PairBatch):
            return ScoreHandle(mi_input, self)
        return super().forward(mi_input)


def mi_estimator_loss(handle: ScoreHandle, estimator: str) -> torch.Tensor:
    p, c = handle.pairs, handle.critic
    if isinstance(c, FusedMLPCritic):
        ops.reject_separable_only(estimator, "the concat-MLP critic (FusedMLPCritic)")
        return _FusedMLPCriticLoss.apply(p.embedding_img, p.embedding_txt, c[0].weight, c[0].bias, c[2].weight, c[2].bias,
                                         c[4].weight, c[4].bias, p.sid, estimator, c.precision, c.check_negatives)
    return _FusedCriticLoss.apply(p.embedding_img, p.embedding_txt, c.W, p.sid, estimator, c.precision,
                                  c.inv_tau, c.check_negatives)


def dv_bound_loss(discriminator_logits, pos_size, device=None):
    """mi_critics.py:3-12.  Returns a 1-element tensor of shape [1] like the reference does for
    ``[N, 1]`` logits."""
    if isinstance(discriminator_logits, ScoreHandle):
        if pos_size != discriminator_logits.pairs.batch_size:
            raise ValueError("pos_size must equal the batch size (main_utils.py:224 passes args.batch_size)")
        return mi_estimator_loss(discriminator_logits, "dv").reshape(1)
    logits = discriminator_logits
    size = logits.shape[0]
    pos_energy = torch.mean(logits[:pos_size])
    lse = torch.logsumexp(logits[pos_size:], dim=0)
    neg_energy = lse - torch.log(torch.tensor(size - pos_size).float()).to(logits.device)   # fp32 log N (mi_critics.py:10)
    return neg_energy - pos_energy


def infonce_bound_loss(discriminator_logits, pos_size, device=None):
    """mi_critics.py:14-23 (the reference's "infonce": DV without the log N_neg term).  0-d result."""
    if isinstance(discriminator_logits, ScoreHandle):
        if pos_size != discriminator_logits.pairs.batch_size:
            raise ValueError("pos_size must equal the batch size (main_utils.py:224 passes args.batch_size)")
        return mi_estimator_loss(discriminator_logits, "infonce")
    logits = discriminator_logits
    pos_energy = torch.mean(logits[:pos_size])
    lse = torch.logsumexp(logits[pos_size:], dim=0)
    return torch.mean(lse) - pos_energy


def infonce_row_loss(handle: ScoreHandle, pos_size=None, device=None):
    """True row-wise InfoNCE (north star; no counterpart in the reference)."""
    return mi_estimator_loss(handle, "infonce_row")


def infonce_sym_loss(handle: ScoreHandle, pos_size=None, device=None):
    """Symmetric (row + column) InfoNCE (north star; no counterpart in the reference)."""
    return mi_estimator_loss(handle, "infonce_sym")


def js_bound_loss(discriminator_logits, pos_size, device=None):
    """Jensen-Shannon bound (Deep InfoMax / f-GAN; no counterpart in the reference), minimised:
    ``mean_{negatives} softplus(S) + mean_i softplus(-S_ii)``.  A ``ScoreHandle`` runs the fused path; a plain logits
    tensor (positives first, then negatives, as ``create_mi_pairs_tensor`` orders them) is computed with torch ops.  0-d."""
    if isinstance(discriminator_logits, ScoreHandle):
        if pos_size != discriminator_logits.pairs.batch_size:
            raise ValueError("pos_size must equal the batch size (main_utils.py:224 passes args.batch_size)")
        return mi_estimator_loss(discriminator_logits, "js")
    logits = discriminator_logits
    pos, neg = logits[:pos_size], logits[pos_size:]
    return torch.mean(F.softplus(neg)) + torch.mean(F.softplus(-pos))


def nwj_bound_loss(discriminator_logits, pos_size, device=None):
    """NWJ bound (Nguyen-Wainwright-Jordan, "MINE-f"; no counterpart in the reference), minimised:
    ``e^{-1} mean_{negatives} e^{S} - mean_i S_ii = e^{LSE - ln N_neg - 1} - pos_mean`` (ln N_neg in fp64).
    ``ScoreHandle`` -> fused path; plain logits (positives first) -> torch ops.  0-d."""
    if isinstance(discriminator_logits, ScoreHandle):
        if pos_size != discriminator_logits.pairs.batch_size:
            raise ValueError("pos_size must equal the batch size (main_utils.py:224 passes args.batch_size)")
        return mi_estimator_loss(discriminator_logits, "nwj")
    logits = discriminator_logits
    pos, neg = logits[:pos_size], logits[pos_size:]
    n_neg = neg.numel()
    ln_n = math.log(n_neg) if n_neg > 0 else -math.inf
    return torch.exp(torch.logsumexp(neg.reshape(-1), dim=0) - (ln_n + 1.0)) - torch.mean(pos)


def select_estimator(name: str):
    """main_utils.py:141-144: 'dv' -> dv_bound_loss, 'infonce' -> infonce_bound_loss.  The reference
    leaves ``mi_critic`` unbound for any other value (UnboundLocalError at :224); here the two new
    estimators are selectable and anything else raises immediately."""
    table = {"dv": dv_bound_loss, "infonce": infonce_bound_loss,
             "infonce_row": infonce_row_loss, "infonce_sym": infonce_sym_loss,
             "js": js_bound_loss, "nwj": nwj_bound_loss}
    if name not in table:
        raise ValueError(f"unknown mi_estimator {name!r} (reference: main_utils.py:141-144)")
    return table[name]
