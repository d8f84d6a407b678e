// The batch-sharded step (SURVEY 8e) as ONE host call: rank r owns rows [r Bl, (r+1) Bl) of the image and text embeddings;
// the text embeddings and study ids are all-gathered, every rank runs the single pass over its row block against ALL
// columns, the [B, D] dY contributions are reduce-scattered and dW is all-reduced.  Included into mi_b200.cu (uses its
// helpers: Bump, run_gemm, ref_sample_impl, single_pass_impl, the finalisation kernels).  Not a standalone header.
//
// NCCL is called directly (ncclAllGather / ncclAllReduce / ncclReduceScatter on the communicator the caller hands in —
// torch.distributed's own, so no second communicator and no extra NVLink buffers), resolved at run time from the
// libnccl.so.2 already loaded in the process.  All collectives of a context go to ONE communication stream in program
// order; the compute stream and the communication stream meet only through events:
//
//   compute stream                                   communication stream
//   --------------                                   --------------------
//   own text rows -> their slot of Y_all   --ev-->   all-gather study ids, all-gather Y (in place)
//   T = X W; references from the OWN column block
//   (strided sample); lambda_r             --ev-->   all-reduce(max) lambda
//   mask pre-pass (after the ids)
//   score tiles of the own column block              (text embeddings of the other ranks still arriving)
//   <--ev-- wait Y; the other column blocks
//   <--ev-- wait lambda; row sums, guard, scalars --ev--> all-gather the 8 loss scalars; merge -> loss, LSE, guard -> host
//   dY contraction  (ok_raw complete)      --ev-->   reduce-scatter ok_raw -> dY          (under the dT contraction)
//   dT contraction; finalise dT; dW = X^T dT --ev-->   all-reduce dW                       (under the dX GEMM)
//   dX = dT W^T;  <--ev-- finalise dY;  <--ev-- dW
//
// The host reads ONE number per step, the merged guard count, as soon as the score tiles are done (it waits for an event on
// the communication stream, not for the step); a non-zero count makes the call return MI_GUARD_TRIPPED on EVERY rank (the
// count is the same everywhere) and the caller repeats the step on the exact path.
//
// Symmetric InfoNCE (exact references: no guard, no host read) replaces the references and the single pass by:
//
//   row+col statistics, OWN column tiles first       (aux stream: the mask, after the ids; other ranks' Y still arriving)
//   <--ev-- wait Y; the remaining column tiles
//   fold own diag into own column partials  --ev-->  ONE all-gather of the records {8 fp64 scalars | B fp32 column partials}
//   <--ev-- c (fp64 log-sum-exp over ranks), loss   merge (fixed order: the same bits on every rank)
//   gradient pass (refq = row lse, refk = c)  --ev-->  reduce-scatter of the final dY contributions     (under the dT contraction)
//   dW = X^T dT                                --ev-->  all-reduce dW                                  (under the dX GEMM)
//
// The gradient pass needs every column's log-sum-exp, so the merge is a hard barrier between the two score computations.
#include <dlfcn.h>

namespace {

typedef void* ncclComm_p;
struct NcclApi {
  int (*all_gather)(const void*, void*, size_t, int, ncclComm_p, cudaStream_t) = nullptr;
  int (*all_reduce)(const void*, void*, size_t, int, int, ncclComm_p, cudaStream_t) = nullptr;
  int (*reduce_scatter)(const void*, void*, size_t, int, int, ncclComm_p, cudaStream_t) = nullptr;
  int (*comm_count)(ncclComm_p, int*) = nullptr;
  int (*comm_rank)(ncclComm_p, int*) = nullptr;
  const char* (*error_string)(int) = nullptr;
  bool ok = false;
};
// nccl.h: ncclDataType_t / ncclRedOp_t values (stable across NCCL 2.x)
constexpr int kNcclUint8 = 1, kNcclInt32 = 2, kNcclFloat32 = 7, kNcclFloat64 = 8, kNcclBf16 = 9, kNcclSum = 0, kNcclMax = 2;

const NcclApi& nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);      // torch has loaded it already
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW);
    if (!h) h = RTLD_DEFAULT;
    api.all_gather = reinterpret_cast<decltype(api.all_gather)>(dlsym(h, "ncclAllGather"));
    api.all_reduce = reinterpret_cast<decltype(api.all_reduce)>(dlsym(h, "ncclAllReduce"));
    api.reduce_scatter = reinterpret_cast<decltype(api.reduce_scatter)>(dlsym(h, "ncclReduceScatter"));
    api.comm_count = reinterpret_cast<decltype(api.comm_count)>(dlsym(h, "ncclCommCount"));
    api.comm_rank = reinterpret_cast<decltype(api.comm_rank)>(dlsym(h, "ncclCommUserRank"));
    api.error_string = reinterpret_cast<decltype(api.error_string)>(dlsym(h, "ncclGetErrorString"));
    api.ok = api.all_gather && api.all_reduce && api.reduce_scatter && api.comm_count && api.comm_rank;
  });
  return api;
}
int nccl_fail(int r, const char* where) {
  const NcclApi& n = nccl_api();
  std::snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: NCCL error %d (%s)", where, r, n.error_string ? n.error_string(r) : "?");
  return MI_ERR_CUDA;
}
#define MI_NCCL(call) do { int r__ = (call); if (r__ != 0) return nccl_fail(r__, #call); } while (0)

}  // namespace

struct mi_dist_ctx {
  ncclComm_p comm; int rank, world, device;
  cudaStream_t comm_stream;
  cudaStream_t aux_stream;     // the negatives-mask pre-pass of the whole column set runs here, beside the projection / references
  cudaEvent_t ev_in, ev_lamloc, ev_sid, ev_y, ev_lam, ev_s, ev_k, ev_m, ev_rs, ev_dwg, ev_dw, ev_drain, ev_mask, ev_start;
  double* guard_host;      // pinned: the merged guard count of the step in flight
};

namespace {

// everything the step keeps in the caller's workspace besides the stage scratch
struct ShardBufs {
  __nv_bfloat16 *T, *Y_all, *dT16;
  int *sid_all, *flag;
  float *ref, *diag, *lam_loc, *lam, *wrow, *rows, *lse32, *oq_raw, *ok_raw, *c;
  double *scal, *scal_all, *scratch8;
  uint8_t* rec_all;        // symmetric estimator: the ranks' packed records {8 fp64 scalars | B fp32 column partials | pad}
};

int sharded_impl(mi_dist_ctx* ctx, int world, int rank, const void* X_, const void* Y_, const void* W_, const int* sid_local,
                 long long Bl, long long D, int critic, int estimator, int precision, float inv_tau,
                 double* loss_out, float* dX, float* dY, float* dW, Bump& ws, int check_guard, cudaStream_t S) {
  typedef __nv_bfloat16 bf;
  if (Bl <= 0 || D <= 0 || (D % 8) != 0) return MI_ERR_BAD_ARG;
  if (precision & MI_PREC_FP32X3) return MI_ERR_BAD_ARG;     // three-piece operands: the MLP critic only
  if (estimator < MI_EST_DV || estimator > MI_EST_INFONCE_SYM) return MI_ERR_BAD_ARG;
  const bool bilinear = critic == MI_CRITIC_BILINEAR;
  const bool sym = estimator == MI_EST_INFONCE_SYM;
  const bool dv_like = estimator == MI_EST_DV || estimator == MI_EST_INFONCE_REF;
  const bool strict = (precision & 1) == MI_PREC_BF16_STRICT;
  if (world < 1 || rank < 0 || rank >= world) return MI_ERR_BAD_ARG;
  const long long Bg = Bl * world, off = static_cast<long long>(rank) * Bl;
  const int tsplit = (bilinear && strict) ? 2 : 1;
  const long long Dp = round_up(D, kSplitAlign);
  const long long ldT = tsplit == 2 ? 2 * Dp : D;
  // symmetric record of one rank: 64 B of scalars, then the column partials, padded to 16 B
  const size_t rec_bytes = 64 + static_cast<size_t>(round_up(Bg * 4, 16));
  ShardBufs b{};
  b.T = bilinear ? ws.take<bf>(static_cast<size_t>(Bl) * ldT) : nullptr;
  b.Y_all = ws.take<bf>(static_cast<size_t>(Bg) * D);
  b.dT16 = bilinear ? ws.take<bf>(static_cast<size_t>(Bl) * ldT) : nullptr;
  b.sid_all = ws.take<int>(Bg);
  b.ref = ws.take<float>(Bl); b.rows = ws.take<float>(static_cast<size_t>(Bl) * 4);
  if (sym) {
    b.rec_all = ws.take<uint8_t>(static_cast<size_t>(world) * rec_bytes);
    b.c = ws.take<float>(Bg);
    b.scratch8 = ws.take<double>(merge_sym_scratch_doubles(Bg));
  } else {
    b.flag = ws.take<int>(1);
    b.diag = ws.take<float>(Bl); b.lam_loc = ws.take<float>(1); b.lam = ws.take<float>(1);
    b.wrow = ws.take<float>(Bl); b.lse32 = ws.take<float>(1);
    b.oq_raw = (bilinear || !dX) ? ws.take<float>(static_cast<size_t>(Bl) * D) : nullptr;      // dot: dX doubles as the raw buffer
    b.scal = ws.take<double>(8); b.scal_all = ws.take<double>(static_cast<size_t>(world) * 8); b.scratch8 = ws.take<double>(8);
  }
  b.ok_raw = ws.take<float>(static_cast<size_t>(Bg) * D);
  const long long k_pad_all = cdiv(Bg, mi::TILE_N) * mi::TILE_N;
  const MaskBuf all_mask = take_mask(ws, Bl, k_pad_all, Bg);      // rows: this rank's; columns: everyone's
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  const size_t mk = ws.mark();
  const int incl = dv_like ? 0 : 1;
  const float gam = 1.f / static_cast<float>(Bg);
  const long long stride = ref_stride_auto(Bl, Bl, D);
  // the own column block is a SUBSET of the row's columns whenever there is more than one rank: margin even at stride 1
  const float margin = (world > 1 || stride > 1) ? kRefMargin : 0.f;
  const Opnd Yloc{static_cast<const bf*>(Y_), D, 1};
  if (ws.dry) {          // planning: the stage scratch of every stage, one after the other
    const Opnd To{nullptr, ldT, tsplit}, Ya{nullptr, D, 1};
    if (sym) {
      MI_TRY(stats_rc_impl(To, Ya, nullptr, nullptr, off, Bl, Bg, D, 1.f, nullptr, nullptr, nullptr, nullptr, nullptr, ws, nullptr,
                           nullptr, false, &all_mask, true));
      ws.release(mk);
      // (planned as mi_score_grad_workspace_bytes plans the stage op, for its largest operand variant: a hi/lo K)
      GradOut oq, okk;
      MI_TRY(grad_impl(To, Opnd{nullptr, D, 2}, nullptr, nullptr, off, Bl, Bg, D, 1.f, nullptr, 1.f, nullptr, 1.f, 1, precision & 1,
                       1.f, gam, oq, &okk, ws, nullptr, nullptr, &all_mask));
    } else {
      MI_TRY(ref_sample_impl(To, Yloc, nullptr, nullptr, 0, Bl, Bl, D, 1.f, incl, 0, Bl, stride, margin, nullptr, nullptr, nullptr, ws, nullptr));
      ws.release(mk);
      MI_TRY(single_pass_impl(To, Ya, nullptr, nullptr, off, Bl, Bg, D, 1.f, incl, precision, gam, nullptr, nullptr, nullptr,
                              nullptr, nullptr, nullptr, nullptr, nullptr, ws, nullptr));
    }
    ws.release(mk);
    if (bilinear) {        // dW split-K partials
      GemmArgs g; g.M = D; g.N = D; g.k_blocks = static_cast<int>(round_up(Bl, kSplitAlign) / bk()) * tsplit;
      g.ksplit = choose_ksplit(cdiv(D, rows_per_mblk()) * cdiv(D, mi::TILE_N), g.k_blocks, strict ? cdiv(g.k_blocks, 16) : 1);
      MI_TRY(run_gemm(g, ws, nullptr));
      ws.release(mk);
    }
    return MI_OK;
  }
  const NcclApi& nc = nccl_api();
  if (!nc.ok) { std::snprintf(g_cuda_err, sizeof(g_cuda_err), "libnccl.so.2 not found in the process"); return MI_ERR_CUDA; }
  const bf* X = static_cast<const bf*>(X_); const bf* Y = static_cast<const bf*>(Y_); const bf* W = static_cast<const bf*>(W_);
  if (!X || !Y || !sid_local || !loss_out || (bilinear && !W) || !dY || (!dX && !bilinear)) return MI_ERR_BAD_ARG;
  cudaStream_t Cs = ctx->comm_stream, As = ctx->aux_stream;
  Bump none(nullptr, 0, false);
  MI_CUDA(cudaEventRecord(ctx->ev_start, S));              // the auxiliary stream joins the step here (workspace reuse is ordered)
  MI_CUDA(cudaStreamWaitEvent(As, ctx->ev_start, 0));

  // ---- exchange: ids, text embeddings (in place: the own rows are in their slot before the collective starts)
  MI_CUDA(cudaMemcpyAsync(b.Y_all + off * D, Y, static_cast<size_t>(Bl) * D * sizeof(bf), cudaMemcpyDeviceToDevice, S));
  MI_CUDA(cudaEventRecord(ctx->ev_in, S));
  MI_CUDA(cudaStreamWaitEvent(Cs, ctx->ev_in, 0));
  if (world > 1) {
    MI_NCCL(nc.all_gather(sid_local, b.sid_all, static_cast<size_t>(Bl), kNcclInt32, ctx->comm, Cs));
    MI_CUDA(cudaEventRecord(ctx->ev_sid, Cs));
    MI_NCCL(nc.all_gather(b.Y_all + off * D, b.Y_all, static_cast<size_t>(Bl) * D, kNcclBf16, ctx->comm, Cs));
  } else {
    MI_CUDA(cudaMemcpyAsync(b.sid_all, sid_local, static_cast<size_t>(Bl) * 4, cudaMemcpyDeviceToDevice, Cs));
    MI_CUDA(cudaEventRecord(ctx->ev_sid, Cs));
  }
  MI_CUDA(cudaEventRecord(ctx->ev_y, Cs));
  // ---- the negatives mask of (own rows) x (all columns): needs the gathered ids only — built on the auxiliary stream while
  //      the compute stream projects and samples
  MI_CUDA(cudaStreamWaitEvent(As, ctx->ev_sid, 0));
  MI_TRY(build_mask(all_mask, b.sid_all + off, b.sid_all, Bl, Bg, k_pad_all, As));
  MI_CUDA(cudaEventRecord(ctx->ev_mask, As));
  // ---- local: projection, references from the own column block, lambda
  if (bilinear) {
    if (tsplit == 2) {
      MI_CUDA(cudaMemsetAsync(b.T, 0, static_cast<size_t>(Bl) * ldT * sizeof(bf), S));
      MI_CUDA(cudaMemsetAsync(b.dT16, 0, static_cast<size_t>(Bl) * ldT * sizeof(bf), S));
    }
    GemmArgs g;
    g.a = MapSpec{X, Bl, D, D};
    g.b_mn = true; g.b = MapSpec{W, D, D, D};
    g.M = Bl; g.N = D; g.k_blocks = static_cast<int>(cdiv(D, bk()));
    g.out_bf16 = b.T; g.ld_out16 = ldT; g.out_bf16_lo = tsplit == 2 ? b.T + Dp : nullptr;
    MI_TRY(run_gemm(g, none, S));
  }
  const Opnd To = bilinear ? Opnd{b.T, ldT, tsplit} : Opnd{X, D, 1};
  const Opnd Ya{b.Y_all, D, 1};
  float* oq_raw = b.oq_raw ? b.oq_raw : dX;      // (single pass)
  if (sym) {
    // ---- row + column statistics of this rank's rows against ALL columns (exact references: no guard), the own column
    //      block first; the own positive pairs are folded into the own slots of the column partials, which go straight
    //      into this rank's record of the packed exchange
    uint8_t* rec = b.rec_all + static_cast<size_t>(rank) * rec_bytes;
    MI_CUDA(cudaStreamWaitEvent(S, ctx->ev_mask, 0));
    MI_TRY(stats_rc_impl(To, Ya, b.sid_all + off, b.sid_all, off, Bl, Bg, D, inv_tau, b.rows, reinterpret_cast<double*>(rec),
                         nullptr, nullptr, reinterpret_cast<float*>(rec + 64), ws, S, ctx->ev_y, /*k_local_valid=*/true, &all_mask,
                         /*include_pos=*/true));
    ws.release(mk);
    make_ref_kernel<<<blocks_for(Bl, 256), 256, 0, S>>>(b.ref, reinterpret_cast<const float4*>(b.rows), 3, nullptr, Bl);
    MI_LAUNCH_CHECK("make_ref_kernel");
    MI_CUDA(cudaEventRecord(ctx->ev_s, S));
    // ---- ONE all-gather of the records; every rank merges them the same way (fixed order: the same bits everywhere)
    MI_CUDA(cudaStreamWaitEvent(Cs, ctx->ev_s, 0));
    if (world > 1) MI_NCCL(nc.all_gather(rec, b.rec_all, rec_bytes, kNcclUint8, ctx->comm, Cs));
    MI_TRY(merge_sym_impl(reinterpret_cast<const double*>(b.rec_all), static_cast<long long>(rec_bytes / 8),
                          reinterpret_cast<const float*>(b.rec_all + 64), static_cast<long long>(rec_bytes / 4), world, Bg,
                          loss_out, b.c, b.scratch8, Cs));
    MI_CUDA(cudaEventRecord(ctx->ev_m, Cs));
    // ---- the gradient pass needs every column reference c_j: G = (1/2B)(e^{S - r_i} + e^{S - c_j}), positives included.
    //      dT (or dX) and this rank's dY contributions come out final; ev_k marks the contributions complete.
    MI_CUDA(cudaStreamWaitEvent(S, ctx->ev_m, 0));
    GradOut oq, okk;
    if (bilinear) { oq.bf16 = b.dT16; oq.ld16 = ldT; oq.split = tsplit; }
    else { oq.f32 = dX; oq.ld = D; }
    okk.f32 = b.ok_raw; okk.ld = D;
    const float w = 0.5f / static_cast<float>(Bg);
    MI_TRY(grad_impl(To, Ya, b.sid_all + off, b.sid_all, off, Bl, Bg, D, inv_tau, b.ref, w, b.c, w, 1, precision & 1, inv_tau, gam,
                     oq, &okk, ws, S, ctx->ev_k, &all_mask));
    ws.release(mk);
  } else {
    MI_TRY(ref_sample_impl(To, Yloc, sid_local, sid_local, 0, Bl, Bl, D, inv_tau, incl, 0, Bl, stride, margin, b.ref, b.diag, b.lam_loc, ws, S));
    ws.release(mk);
    MI_CUDA(cudaEventRecord(ctx->ev_lamloc, S));
    MI_CUDA(cudaStreamWaitEvent(Cs, ctx->ev_lamloc, 0));
    if (world > 1) MI_NCCL(nc.all_reduce(b.lam_loc, b.lam, 1, kNcclFloat32, kNcclMax, ctx->comm, Cs));
    else MI_CUDA(cudaMemcpyAsync(b.lam, b.lam_loc, 4, cudaMemcpyDeviceToDevice, Cs));
    MI_CUDA(cudaEventRecord(ctx->ev_lam, Cs));
    // ---- the single pass over this rank's rows against ALL columns
    MI_CUDA(cudaStreamWaitEvent(S, ctx->ev_mask, 0));
    MI_CUDA(cudaMemsetAsync(b.flag, 0, sizeof(int), S));
    MI_TRY(single_pass_impl(To, Ya, b.sid_all + off, b.sid_all, off, Bl, Bg, D, inv_tau, incl, precision, gam, b.ref, b.lam, b.diag,
                            b.rows, oq_raw, b.ok_raw, b.wrow, b.flag, ws, S, ctx->ev_k, b.scal, ctx->ev_s, ctx->ev_y, nullptr, nullptr,
                            /*k_local_valid=*/true, &all_mask, ctx->ev_lam));
    ws.release(mk);
    // ---- scalars: exchange and merge on the communication stream, under the contractions; the guard goes to the host.
    //      (The rows are reduced inside the pass, on the compute stream, BEFORE the dY contraction is launched: the engine's
    //      persistent grid takes every SM, so a collective that is not already running when it starts waits for it to end —
    //      measured: deferring the reduction to this stream delayed the scalar all-gather by the whole contraction.)
    MI_CUDA(cudaStreamWaitEvent(Cs, ctx->ev_s, 0));
    if (world > 1) MI_NCCL(nc.all_gather(b.scal, b.scal_all, 8, kNcclFloat64, ctx->comm, Cs));
    else MI_CUDA(cudaMemcpyAsync(b.scal_all, b.scal, 64, cudaMemcpyDeviceToDevice, Cs));
    merge_scal_kernel<<<1, 32, 0, Cs>>>(b.scal_all, world, b.scratch8);
    MI_LAUNCH_CHECK("merge_scal_kernel");
    loss_finalize_kernel<<<1, 32, 0, Cs>>>(b.scratch8, nullptr, Bg, estimator, loss_out, b.lse32, dv_like ? b.lam : nullptr, nullptr);
    MI_LAUNCH_CHECK("loss_finalize_kernel");
    if (check_guard) MI_CUDA(cudaMemcpyAsync(ctx->guard_host, loss_out + 7, sizeof(double), cudaMemcpyDeviceToHost, Cs));
    MI_CUDA(cudaEventRecord(ctx->ev_m, Cs));
    if (check_guard) {
      MI_CUDA(cudaEventSynchronize(ctx->ev_m));            // the score tiles are done; the contractions are still running
      if (ctx->guard_host[0] != 0.0) {                     // same verdict on every rank: abandon the step (no collective is pending)
        MI_CUDA(cudaStreamWaitEvent(S, ctx->ev_m, 0));
        return MI_GUARD_TRIPPED;
      }
    }
  }
  // ---- reduce-scatter of the dY contributions (as soon as they are complete: under the dT contraction)
  MI_CUDA(cudaStreamWaitEvent(Cs, ctx->ev_k, 0));
  if (world > 1) MI_NCCL(nc.reduce_scatter(b.ok_raw, dY, static_cast<size_t>(Bl) * D, kNcclFloat32, kNcclSum, ctx->comm, Cs));
  else MI_CUDA(cudaMemcpyAsync(dY, b.ok_raw, static_cast<size_t>(Bl) * D * 4, cudaMemcpyDeviceToDevice, Cs));
  MI_CUDA(cudaEventRecord(ctx->ev_rs, Cs));
  // ---- finalise: dT, dW (all-reduced), dX, dY
  MI_CUDA(cudaStreamWaitEvent(S, ctx->ev_m, 0));
  if (!sym) {
    finalize_q_kernel<<<blocks_capped(Bl * D / 8, 256), 256, 0, S>>>(oq_raw, D, Bl, b.ref, b.wrow, b.lse32, dv_like ? 1 : 0, inv_tau, gam,
                                                                     b.Y_all + off * D, D, 1, Dp, bilinear ? nullptr : dX,
                                                                     bilinear ? b.dT16 : nullptr, (bilinear && tsplit == 2) ? b.dT16 + Dp : nullptr,
                                                                     ldT, nullptr);
    MI_LAUNCH_CHECK("finalize_q_kernel");
  }
  if (bilinear) {
    if (dW) {
      GemmArgs g;
      const int kb = static_cast<int>(round_up(Bl, kSplitAlign) / bk());
      g.a_mn = true; g.a = MapSpec{X, Bl, D, D};
      g.b_mn = true; g.b = MapSpec{b.dT16, Bl, tsplit == 2 ? Dp + D : D, ldT};
      g.M = D; g.N = D; g.seg_len = kb; g.k_blocks = kb;
      if (tsplit == 2) { g.k_blocks = 2 * kb; g.b_noff[1] = static_cast<int>(Dp); }
      g.ksplit = choose_ksplit(cdiv(D, rows_per_mblk()) * cdiv(D, mi::TILE_N), g.k_blocks, strict ? cdiv(g.k_blocks, 16) : 1);
      g.out_f32 = dW; g.ld_out = D;
      MI_TRY(run_gemm(g, ws, S));
      ws.release(mk);
      MI_CUDA(cudaEventRecord(ctx->ev_dwg, S));
      MI_CUDA(cudaStreamWaitEvent(Cs, ctx->ev_dwg, 0));
      if (world > 1) MI_NCCL(nc.all_reduce(dW, dW, static_cast<size_t>(D) * D, kNcclFloat32, kNcclSum, ctx->comm, Cs));
      MI_CUDA(cudaEventRecord(ctx->ev_dw, Cs));
    }
    if (dX) {
      const Opnd dTo{b.dT16, ldT, tsplit};
      MI_TRY(gemm_impl(dTo, Opnd{W, D, 1}, Bl, D, D, 1.f, 0.f, nullptr, 0, dX, D, nullptr, 0, 1, 1, ws, S));
      ws.release(mk);
    }
  }
  MI_CUDA(cudaStreamWaitEvent(S, ctx->ev_rs, 0));
  if (!sym) {       // (the symmetric gradient pass wrote its dY contributions final)
    finalize_k_kernel<<<blocks_capped(Bl * D / 8, 256), 256, 0, S>>>(dY, D, Bl, b.lam, b.lse32, dv_like ? 1 : 0, inv_tau, gam,
                                                                     To.p, To.ld, To.split, Dp, 0, Bl);
    MI_LAUNCH_CHECK("finalize_k_kernel");
  }
  if (bilinear && dW) MI_CUDA(cudaStreamWaitEvent(S, ctx->ev_dw, 0));
  return MI_OK;
}

}  // namespace
