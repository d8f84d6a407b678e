// Part of libmi_b200.so: included by mi_b200.cu INSIDE its anonymous namespace, after the tile-engine launchers
// (Bump, GemmArgs, run_gemm, launch_engine, the statistics kernels).  Not a standalone header.
#pragma once

// ============================================================================================
// Generalised Discrimination Value (validate.py:16-49, SURVEY 8f-3): per-class z-scoring, then the sums of all
// pairwise Euclidean distances inside each class and between the classes — the same tile machinery with a
// sqrt(|a|^2 + |b|^2 - 2 a.b) epilogue; no N x N matrix is stored.
// ============================================================================================
__global__ void col_moments_kernel(const float* __restrict__ X, long long N, long long D, long long rows_per_block,
                                   double* __restrict__ sum, double* __restrict__ sumsq) {
  const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (c >= D) return;
  const long long r0 = blockIdx.y * rows_per_block, r1 = (r0 + rows_per_block < N) ? r0 + rows_per_block : N;
  double s = 0.0, q = 0.0;
  for (long long r = r0; r < r1; ++r) { const double v = X[r * D + c]; s += v; q += v * v; }
  atomicAdd(sum + c, s); atomicAdd(sumsq + c, q);
}
// StandardScaler (validate.py:16-21): mean, population std; constant features keep scale 1 (sklearn's rule)
__global__ void col_scale_kernel(const double* __restrict__ sum, const double* __restrict__ sumsq, long long N, long long D,
                                 float* __restrict__ mean_f, float* __restrict__ scale_f) {
  const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (c >= D) return;
  const double n = static_cast<double>(N), mean = sum[c] / n;
  double var = sumsq[c] / n - mean * mean;
  if (var < 0.0) var = 0.0;
  const double eps = 2.220446049250313e-16;
  const double bound = n * eps * var + (n * mean * eps) * (n * mean * eps);
  mean_f[c] = static_cast<float>(mean);
  scale_f[c] = static_cast<float>((var <= bound) ? 1.0 : sqrt(var));
}
// one warp per row: z = (x - mean) / scale (fp32, as the in-place float32 transform), bf16 hi (+ lo) operand row, |z|^2
__global__ void zscore_split_kernel(const float* __restrict__ X, long long N, long long D, const float* __restrict__ mean,
                                    const float* __restrict__ scale, __nv_bfloat16* __restrict__ Z, long long pitch, long long Dp,
                                    int split, float* __restrict__ norm2) {
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= N) return;
  float acc = 0.f;
  for (long long c = lane; c < D; c += 32) {
    const float z = (X[row * D + c] - mean[c]) / scale[c];
    const __nv_bfloat16 h = __float2bfloat16(z);
    float used = __bfloat162float(h);
    Z[row * pitch + c] = h;
    if (split == 2) {
      const __nv_bfloat16 l = __float2bfloat16(z - used);
      Z[row * pitch + Dp + c] = l;
      used += __bfloat162float(l);
    }
    acc = fmaf(used, used, acc);
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) norm2[row] = acc;
}
// out[slot] = sum of a partial array (fp64 accumulation); one block
__global__ void sum_f32_to_f64_kernel(const float* __restrict__ in, long long n, double* __restrict__ out) {
  __shared__ double sh[32];
  double a = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) a += in[i];
  for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) { double t = 0.0; for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i]; out[0] = t; }
}
// validate.py:23-49 — note the reference's normalisers count ELEMENTS (N * D), not samples
__global__ void gdv_finalize_kernel(const double* __restrict__ sums, long long Np, long long Nn, long long D, double* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double tp = static_cast<double>(Np) * D, tn = static_cast<double>(Nn) * D;
  const double intra_p = sums[0] * 2.0 / (tp * (tp - 1.0));
  const double intra_n = sums[1] * 2.0 / (tn * (tn - 1.0));
  const double inter = sums[2] / (tp * tn);
  out[0] = ((intra_p + intra_n) / 2.0 - inter) / sqrt(static_cast<double>(Np + Nn));
  out[1] = intra_p; out[2] = intra_n; out[3] = inter;
}

int gdv_impl(const float* pos, const float* neg, long long Np, long long Nn, long long D, int precision, double* out,
             Bump& ws, cudaStream_t stream) {
  if (Np <= 1 || Nn <= 1 || D <= 0 || (D % 8) != 0) return MI_ERR_BAD_ARG;
  if (precision & MI_PREC_FP32X3) return MI_ERR_BAD_ARG;     // three-piece operands: the MLP critic only
  typedef __nv_bfloat16 bf;
  const int sp = (precision & 1) == MI_PREC_BF16_STRICT ? 2 : 1;
  const long long Dp = round_up(D, kSplitAlign), pitch = sp == 2 ? 2 * Dp : D, ext = sp == 2 ? Dp + D : D;
  const long long N[2] = {Np, Nn};
  const float* X[2] = {pos, neg};
  bf* Z[2]; float* nrm[2];
  const long long nmax = Np > Nn ? Np : Nn;
  const long long npad = cdiv(nmax, mi::TILE_N) * mi::TILE_N + mi::TILE_N;
  for (int c = 0; c < 2; ++c) { Z[c] = ws.take<bf>(N[c] * pitch); nrm[c] = ws.take<float>(npad); }
  double* mom = ws.take<double>(2 * D);
  float* mean = ws.take<float>(D); float* scale = ws.take<float>(D);
  double* sums = ws.take<double>(4);
  const int mb_max = static_cast<int>(cdiv(nmax, rows_per_mblk()));
  const int nt_max = static_cast<int>(cdiv(nmax, mi::TILE_N));
  const long long rows_padded_max = static_cast<long long>(mb_max) * rows_per_mblk();
  const int split_max = nt_max < 64 ? nt_max : 64;
  float* part = ws.take<float>(static_cast<size_t>(split_max) * mi::kColQuarters * rows_padded_max);
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (ws.dry) return MI_OK;
  if (!pos || !neg || !out) return MI_ERR_BAD_ARG;
  for (int c = 0; c < 2; ++c) {
    MI_CUDA(cudaMemsetAsync(mom, 0, 2 * D * sizeof(double), stream));
    MI_CUDA(cudaMemsetAsync(nrm[c], 0, npad * sizeof(float), stream));
    if (sp == 2) MI_CUDA(cudaMemsetAsync(Z[c], 0, static_cast<size_t>(N[c]) * pitch * sizeof(bf), stream));
    const long long rpb = 256;
    dim3 grid(static_cast<unsigned>(cdiv(D, 128)), static_cast<unsigned>(cdiv(N[c], rpb)));
    col_moments_kernel<<<grid, 128, 0, stream>>>(X[c], N[c], D, rpb, mom, mom + D);
    MI_LAUNCH_CHECK("col_moments_kernel");
    col_scale_kernel<<<blocks_for(D, 128), 128, 0, stream>>>(mom, mom + D, N[c], D, mean, scale);
    MI_LAUNCH_CHECK("col_scale_kernel");
    zscore_split_kernel<<<blocks_for(N[c] * 32, 256), 256, 0, stream>>>(X[c], N[c], D, mean, scale, Z[c], pitch, Dp, sp, nrm[c]);
    MI_LAUNCH_CHECK("zscore_split_kernel");
  }
  const int pairs_ab[3][2] = {{0, 0}, {1, 1}, {0, 1}};
  for (int t = 0; t < 3; ++t) {
    const int a = pairs_ab[t][0], b = pairs_ab[t][1];
    Sched sc;
    sc.n_mblk = static_cast<int>(cdiv(N[a], rows_per_mblk()));
    sc.n_ntile = static_cast<int>(cdiv(N[b], mi::TILE_N));
    sc.n_split = choose_split(sc.n_mblk, sc.n_ntile, num_pairs());
    if (sc.n_split > split_max) sc.n_split = split_max;
    sc.n_ksplit = 1; sc.order = 0;
    single_segment(sc);
    const int kb = static_cast<int>(sp == 2 ? Dp / bk() : cdiv(D, bk()));
    sc.k_blocks = kb; sc.seg_len = kb;
    if (sp == 2) { sc.k_blocks = 3 * kb; sc.a_seg[1] = kb; sc.b_seg[2] = kb; }      // hi*hi + lo*hi + hi*lo
    mi::EpiDist::Params ep;
    ep.na = nrm[a]; ep.nb = nrm[b]; ep.rows = static_cast<int>(N[a]); ep.cols = static_cast<int>(N[b]);
    ep.same = a == b ? 1 : 0; ep.part = part; ep.rows_padded = sc.n_mblk * rows_per_mblk();
    const long long n_part = static_cast<long long>(sc.n_split) * mi::kColQuarters * ep.rows_padded;
    MI_CUDA(cudaMemsetAsync(part, 0, n_part * sizeof(float), stream));
    MI_TRY(launch_engine<mi::EpiDist>(MapSpec{Z[a], N[a], ext, pitch}, MapSpec{Z[b], N[b], ext, pitch}, sc, ep, stream));
    sum_f32_to_f64_kernel<<<1, 1024, 0, stream>>>(part, n_part, sums + t);
    MI_LAUNCH_CHECK("sum_f32_to_f64_kernel");
  }
  gdv_finalize_kernel<<<1, 32, 0, stream>>>(sums, Np, Nn, D, out);
  MI_LAUNCH_CHECK("gdv_finalize_kernel");
  return MI_OK;
}

