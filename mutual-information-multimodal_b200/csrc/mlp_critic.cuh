// Part of libmi_b200.so: included by mi_b200.cu INSIDE its anonymous namespace, after the tile-engine launchers
// (Bump, GemmArgs, run_gemm, launch_engine, the statistics kernels).  Not a standalone header.
#pragma once

// ============================================================================================
// Concat-MLP critic — the reference's own mi_discriminator = make_mlp(1536, [1024, 512])
// (main_utils.py:77, model.py:18-32) on every (image i, text j) pair, without the pair tensor.
//
//   layer 1 is separable:  W1 [x_i ; y_j] + b1 = (W1x x_i + b1) + W1y y_j = A_i + C_j     (two [B, H1] GEMMs)
//   per pair (i, j):       h1 = relu(A_i + C_j);  z2 = W2 h1 + b2;  S_ij = w3 . relu(z2) + b3
//
// Pairs are processed in row panels (rows i in [r0, r0 + R), all columns j; pair index p = (i - r0) B + j):
//   forward   H[p,:] = bf16 h1  ->  tile engine  Z2 = H W2^T  with the EpiMlpFwd epilogue  ->  S (fp32 [B, B])
//   loss      row statistics of S over the negatives mask (symmetric InfoNCE: and column statistics) -> DV / InfoNCE
//             exactly as for the separable critics; G = dL/dS
//   backward  recompute Z2 with the EpiMlpDz epilogue -> dZ2 panel (bf16), dw3, db2;
//             dW2 += dZ2^T H          (both operands read MN-major, contraction over the pairs, split-K)
//             dZ1  = (dZ2 W2) . [H > 0]  (W2 read MN-major; ReLU mask in the epilogue), reduced over j -> dA_i, over i -> dC_j
//             dX = dA W1x, dY = dC W1y, dW1 = [dA^T X | dC^T Y], db1 = sum_i dA_i
// Strict ("fp32-accumulate") mode keeps every bf16 operand as a hi/lo pair and adds the cross terms as K segments;
// fp32 mode keeps three pieces (24 significant bits, six K segments) and bounds every accumulation chain (kFp32ChainK).
//
// dv / infonce (global log-sum-exp) run as a SINGLE PASS (mlp_single_pass below): the softmax weights are formed against
// a reference logit fixed before the pass (maximum over a sample of pairs + margin), so the Z2 accumulator that gives
// the logit also gives dZ2 — Z2 is not recomputed (6 instead of 8 B^2 H1 H2 flops), [B, B] logits / gradients are not
// stored, and the dZ1 reductions happen in the epilogue of their GEMM (EpiMlpDa).  The positive pairs (weight -1/B, not
// a softmax weight) are a separate B-pair panel.  A guard that finds the reference outside the safe window repeats the
// step with the two-pass sequence above behind a device-side predicate.
// ============================================================================================
// fp32 [R, C] (pitch ld_in) -> bf16 [R, pitch]: `split` pieces, p0 = RN(x) in columns [0, C), p1 = RN(x - p0) in
// [Cp, Cp + C) (split >= 2), p2 = RN(x - p0 - p1) in [2 Cp, 2 Cp + C) (split == 3: the kThird instantiation, so that
// the fast / strict one carries none of its code), zeros elsewhere
template <bool kThird>
__global__ void split_f32_kernel(const float* __restrict__ in, long long ld_in, __nv_bfloat16* __restrict__ out, long long pitch,
                                 int split, long long Cp, long long R, long long C, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= R * pitch) return;
  const long long r = idx / pitch, c = idx - r * pitch;
  float v = 0.f;
  if (c < C) v = __bfloat162float(__float2bfloat16(in[r * ld_in + c]));
  else if (split >= 2 && c >= Cp && c < Cp + C) {
    const float x = in[r * ld_in + (c - Cp)];
    v = x - __bfloat162float(__float2bfloat16(x));
  } else if (kThird && c >= 2 * Cp && c < 2 * Cp + C) {
    const float x = in[r * ld_in + (c - 2 * Cp)];
    const float d = x - __bfloat162float(__float2bfloat16(x));                 // exact
    v = d - __bfloat162float(__float2bfloat16(d));
  }
  out[idx] = __float2bfloat16(v);
}
__global__ void pad_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, long long n, long long n_pad) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n_pad) dst[i] = (i < n) ? src[i] : 0.f;
}
// predicated memset (the two-pass repeat must not clear anything unless it runs)
__global__ void zero_u4_kernel(uint4* __restrict__ p, long long n16, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n16; i += (long long)gridDim.x * blockDim.x)
    p[i] = make_uint4(0u, 0u, 0u, 0u);
}
__global__ void fill_f32_kernel(float* __restrict__ p, long long n, float v) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
// the third pieces of 8 values v whose first two are packed in hi / lo: RN((v - p0) - p1), both differences exact
__device__ __forceinline__ uint4 third_pieces8(const float (&v)[8], const uint32_t (&hi)[4], const uint32_t (&lo)[4]) {
  uint32_t r[4];
#pragma unroll
  for (int t = 0; t < 4; ++t)
    r[t] = ptx::pack_bf16((v[2 * t] - __uint_as_float(hi[t] << 16)) - __uint_as_float(lo[t] << 16),
                          (v[2 * t + 1] - __uint_as_float(hi[t] & 0xffff0000u)) - __uint_as_float(lo[t] & 0xffff0000u));
  return make_uint4(r[0], r[1], r[2], r[3]);
}
// H[p, k] = relu(A[i, k] + C[j, k]) as bf16 pieces (p0, + p1 at column Hp, + p2 at 2 Hp), 8 columns per thread;
// pairs p = (i - r0) Bk + j of a row panel, or the positive pairs i = p, j = q_off + p (diag)
__global__ void mlp_gen_kernel(const float* __restrict__ A, const float* __restrict__ Cm, long long H1, long long Bk, long long r0,
                               long long P, __nv_bfloat16* __restrict__ H, long long pitch, long long Hp, int split, int diag,
                               long long q_off, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const long long h8 = H1 >> 3;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < P * h8; idx += (long long)gridDim.x * blockDim.x) {
    const long long p = idx / h8, k = (idx - p * h8) << 3;
    const long long i = diag ? p : r0 + p / Bk, j = diag ? q_off + p : p % Bk;
    const float4* a4 = reinterpret_cast<const float4*>(A + i * H1 + k);
    const float4* c4 = reinterpret_cast<const float4*>(Cm + j * H1 + k);
    const float4 a0 = __ldg(a4), a1 = __ldg(a4 + 1), c0 = __ldg(c4), c1 = __ldg(c4 + 1);
    const float v[8] = {fmaxf(a0.x + c0.x, 0.f), fmaxf(a0.y + c0.y, 0.f), fmaxf(a0.z + c0.z, 0.f), fmaxf(a0.w + c0.w, 0.f),
                        fmaxf(a1.x + c1.x, 0.f), fmaxf(a1.y + c1.y, 0.f), fmaxf(a1.z + c1.z, 0.f), fmaxf(a1.w + c1.w, 0.f)};
    uint32_t hi[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) hi[t] = ptx::pack_bf16(v[2 * t], v[2 * t + 1]);
    *reinterpret_cast<uint4*>(H + p * pitch + k) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if (split >= 2) {
      uint32_t lo[4];
#pragma unroll
      for (int t = 0; t < 4; ++t)
        lo[t] = ptx::pack_bf16(v[2 * t] - __uint_as_float(hi[t] << 16), v[2 * t + 1] - __uint_as_float(hi[t] & 0xffff0000u));
      *reinterpret_cast<uint4*>(H + p * pitch + Hp + k) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      if (split == 3) *reinterpret_cast<uint4*>(H + p * pitch + 2 * Hp + k) = third_pieces8(v, hi, lo);
    }
  }
}
// The single pass' panel: pairs in the padded order p = il * Bp + j (j >= B: zero rows), plus the ReLU mask as bits
// (mask[p][w] bit b <=> A[i, 32 w + b] + C[j, 32 w + b] > 0, from the fp32 sum).
// A thread owns 8 columns of kGenJ text rows j (its C values stay in registers) and walks the image rows of its
// blockIdx.y slice: the A row of an image is fetched once per kGenJ pairs, C never again; 4 * wpr threads per text row
// (the 4 threads of a mask word are consecutive lanes), every 2 KB row segment of H is written by consecutive threads.
constexpr int kGenJ = 4;
// kThird: fp32 mode (the third pieces at 2 Hp); the fast / strict instantiation carries none of that code
template <bool kThird>
__global__ void __launch_bounds__(256, 3) mlp_gen2_kernel(const float* __restrict__ A, const float* __restrict__ Cm, long long H1, long long B,
                                                       long long Bp, long long r0, long long rr, __nv_bfloat16* __restrict__ H,
                                                       long long pitch, long long Hp, int split, uint32_t* __restrict__ mask, int wpr) {
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long tpr = 4LL * wpr;
  const long long jg = t / tpr;
  const int k = static_cast<int>(t - jg * tpr) << 3;
  const int lane = threadIdx.x & 31;
  const bool kin = k < H1;
  float c[kGenJ][8];
  bool jin[kGenJ], real[kGenJ];
#pragma unroll
  for (int q = 0; q < kGenJ; ++q) {
    const long long j = jg * kGenJ + q;
    jin[q] = j < Bp; real[q] = kin && j < B;
#pragma unroll
    for (int e = 0; e < 8; ++e) c[q][e] = 0.f;
    if (real[q]) {
      const float4* c4 = reinterpret_cast<const float4*>(Cm + j * H1 + k);
      const float4 c0 = __ldg(c4), c1 = __ldg(c4 + 1);
      c[q][0] = c0.x; c[q][1] = c0.y; c[q][2] = c0.z; c[q][3] = c0.w; c[q][4] = c1.x; c[q][5] = c1.y; c[q][6] = c1.z; c[q][7] = c1.w;
    }
  }
  const long long per = (rr + gridDim.y - 1) / gridDim.y;
  const long long il0 = blockIdx.y * per, il1 = il0 + per < rr ? il0 + per : rr;
  for (long long il = il0; il < il1; ++il) {
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (kin) {
      const float4* a4 = reinterpret_cast<const float4*>(A + (r0 + il) * H1 + k);
      const float4 a0 = __ldg(a4), a1 = __ldg(a4 + 1);
      a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
    }
#pragma unroll
    for (int q = 0; q < kGenJ; ++q) {
      const long long p = il * Bp + jg * kGenJ + q;
      float v[8];
      uint32_t bits = 0;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        v[e] = real[q] ? fmaxf(a[e] + c[q][e], 0.f) : 0.f;
        bits |= (v[e] > 0.f ? 1u : 0u) << e;
      }
      uint32_t w = bits << (8 * (lane & 3));
      w |= __shfl_xor_sync(0xffffffffu, w, 1);
      w |= __shfl_xor_sync(0xffffffffu, w, 2);
      if (jin[q] && (lane & 3) == 0) mask[p * wpr + (k >> 5)] = w;
      if (jin[q] && kin) {
        uint32_t hi[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) hi[e] = ptx::pack_bf16(v[2 * e], v[2 * e + 1]);
        *reinterpret_cast<uint4*>(H + p * pitch + k) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        if (split >= 2) {
          uint32_t lo[4];
#pragma unroll
          for (int e = 0; e < 4; ++e)
            lo[e] = ptx::pack_bf16(v[2 * e] - __uint_as_float(hi[e] << 16), v[2 * e + 1] - __uint_as_float(hi[e] & 0xffff0000u));
          *reinterpret_cast<uint4*>(H + p * pitch + Hp + k) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          if (kThird) *reinterpret_cast<uint4*>(H + p * pitch + 2 * Hp + k) = third_pieces8(v, hi, lo);
        }
      }
    }
  }
}
// dst[s, :] = src[s * stride, :]  (the sampled rows of the reference-logit estimate)
__global__ void gather_rows_kernel(const float* __restrict__ src, long long stride, long long C, float* __restrict__ dst, long long n) {
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= n * C) return;
  const long long s = idx / C, c = idx - s * C;
  dst[idx] = src[s * stride * C + c];
}
// S[r0 * Bk + p] = b3 + sum of the column-quarter partials
__global__ void mlp_logit_merge_kernel(const float* __restrict__ part, int rows_padded, long long P, const float* __restrict__ b3,
                                       float* __restrict__ S, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (p >= P) return;
  float a = b3[0];
#pragma unroll
  for (int q = 0; q < mi::kColQuarters; ++q) a += part[(size_t)q * rows_padded + p];
  S[p] = a;
}
// one warp per row of S [Bq, Bk] (image rows at q_off): {lse over the negatives, #negatives, S[i, q_off + i],
// lse over negatives and the positive}
__global__ void mlp_row_stats_kernel(const float* __restrict__ S, const int* __restrict__ sid_q, const int* __restrict__ sid_k,
                                     long long Bq, long long Bk, long long q_off, float4* __restrict__ row_out,
                                     const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= Bq) return;
  const int my = sid_q[row];
  float m = mi::neg_inf(), s = 0.f, cnt = 0.f;
  for (long long j = lane; j < Bk; j += 32) {
    if (sid_k[j] != my) {                                 // main_utils.py:105 (the diagonal has equal ids)
      const float v = S[row * Bk + j];
      const float mn = fmaxf(m, v);
      s = s * expf(m - mn) + expf(v - mn); m = mn; cnt += 1.f;
    }
  }
  for (int o = 16; o; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    const float mn = fmaxf(m, m2);
    if (mn > mi::neg_inf()) s = s * expf(m - mn) + s2 * expf(m2 - mn);
    m = mn;
  }
  if (lane == 0) {
    const float diag = S[row * Bk + q_off + row];
    const float lse_neg = (cnt > 0.f && s > 0.f) ? m + logf(s) : mi::neg_inf();
    const float hi = fmaxf(lse_neg, diag), lo = fminf(lse_neg, diag);
    row_out[row] = make_float4(lse_neg, cnt, diag, hi + log1pf(expf(lo - hi)));
  }
}
// Columns of S [Bq, Bk] (symmetric InfoNCE), in two launches.  Part 1: thread = column j (consecutive threads read
// consecutive j of a row), blockIdx.y = a slice of the rows; the same online (max, sum exp) as mlp_row_stats_kernel over
// the slice's negatives of column j, and their count.  part = {m, s, cnt}, each [gridDim.y][Bk].
constexpr int kMlpColSplits = 32;                         // most row slices (the part buffer is planned for this many)
__global__ void mlp_col_part_kernel(const float* __restrict__ S, const int* __restrict__ sid_q, const int* __restrict__ sid_k,
                                    long long Bq, long long Bk, float* __restrict__ part, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (j >= Bk) return;
  const long long per = (Bq + gridDim.y - 1) / gridDim.y;
  const long long i0 = blockIdx.y * per, i1 = i0 + per < Bq ? i0 + per : Bq;
  const int my = sid_k[j];
  float m = mi::neg_inf(), s = 0.f, cnt = 0.f;
  for (long long i = i0; i < i1; ++i) {
    if (sid_q[i] != my) {
      const float v = S[i * Bk + j];
      const float mn = fmaxf(m, v);
      s = s * expf(m - mn) + expf(v - mn); m = mn; cnt += 1.f;
    }
  }
  const long long o = blockIdx.y * Bk + j, n = static_cast<long long>(gridDim.y) * Bk;
  part[o] = m; part[n + o] = s; part[2 * n + o] = cnt;
}
// Part 2, per column j: merge of the n_split slices, then the positive pair S[j - q_off, j] if it lies in the block.
// col_lse[j] = log-sum-exp over {i in the block : (i, j) in negatives u positives} (-inf: none).  col_out (square block
// only): the float4 of mlp_row_stats_kernel's layout for the column, {lse over the negatives, #negatives, S[j, j], col_lse[j]}.
__global__ void mlp_col_merge_kernel(const float* __restrict__ part, int n_split, const float* __restrict__ S, long long Bq,
                                     long long Bk, long long q_off, float* __restrict__ col_lse, float4* __restrict__ col_out,
                                     const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (j >= Bk) return;
  const long long n = static_cast<long long>(n_split) * Bk;
  float m = mi::neg_inf(), s = 0.f, cnt = 0.f;
  for (int y = 0; y < n_split; ++y) {
    const float m2 = part[y * Bk + j], s2 = part[n + y * Bk + j];
    cnt += part[2 * n + y * Bk + j];
    const float mn = fmaxf(m, m2);
    if (mn > mi::neg_inf()) s = s * expf(m - mn) + s2 * expf(m2 - mn);
    m = mn;
  }
  const float lse_neg = (cnt > 0.f && s > 0.f) ? m + logf(s) : mi::neg_inf();
  const long long i = j - q_off;
  float diag = mi::neg_inf(), lse = lse_neg;
  if (i >= 0 && i < Bq) {
    diag = S[i * Bk + j];
    const float hi = fmaxf(lse_neg, diag), lo = fminf(lse_neg, diag);
    lse = hi + log1pf(expf(lo - hi));
  }
  col_lse[j] = lse;
  if (col_out) col_out[j] = make_float4(lse_neg, cnt, diag, lse);
}
// the same float4 per row from the single pass' sums: lse over the negatives = ref + log(sum_j g~)
__global__ void mlp_rows_from_sums_kernel(const float* __restrict__ rowsum, const float* __restrict__ rowcnt,
                                          const float* __restrict__ diag, const float* __restrict__ ref, long long B,
                                          float4* __restrict__ row_out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B) return;
  float s = rowsum[i];
  if (!(s >= 0.f)) s = INFINITY;                            // NaN must trip the guard, not vanish in a max
  const float cnt = rowcnt[i], d = diag[i];
  const float lse_neg = cnt > 0.f ? static_cast<float>(static_cast<double>(ref[0]) + mi::kMlpSpMargin + log(static_cast<double>(s)))
                                  : mi::neg_inf();
  const float hi = fmaxf(lse_neg, d), lo = fminf(lse_neg, d);
  row_out[i] = make_float4(lse_neg, cnt, d, hi + log1pf(expf(lo - hi)));
}
// G = dL/dS over a block [Bq, Bk] (image rows at q_off) of a batch of Bg.  dv / infonce (mi_critics.py:3-23): softmax
// over ALL negatives (lse = the global log-sum-exp), -1/Bg on the diagonal; row InfoNCE: (1/Bg) softmax over {positive} u
// negatives of the row, minus 1/Bg on the diagonal; symmetric InfoNCE (col_lse != NULL: the log-sum-exp of every column
// over ALL rows of the batch): the mean of the row and the column softmax, minus 1/Bg on the diagonal.
__global__ void mlp_g_kernel(const float* __restrict__ S, const int* __restrict__ sid_q, const int* __restrict__ sid_k, long long Bq,
                             long long Bk, long long q_off, long long Bg, int dv_like, const float* __restrict__ lse,
                             const float4* __restrict__ rows, const float* __restrict__ col_lse, float* __restrict__ G,
                             const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= Bq * Bk) return;
  const long long i = idx / Bk, j = idx - i * Bk;
  const float inv_b = 1.f / static_cast<float>(Bg);
  const bool neg = sid_q[i] != sid_k[j];
  const bool pos = j == q_off + i;
  float g = 0.f;
  if (dv_like) g = neg ? expf(S[idx] - lse[0]) : (pos ? -inv_b : 0.f);
  else if (neg || pos) {
    const float v = S[idx];
    const float e = col_lse ? 0.5f * (expf(v - rows[i].w) + expf(v - col_lse[j])) : expf(v - rows[i].w);
    g = inv_b * e - (pos ? inv_b : 0.f);
  }
  G[idx] = g;
}
// One read of the dZ1 panel gives both reductions.  A block owns a slab [32 rows il] x [all j] x [64 columns]:
// thread = (column pair, j group); for every j it loads the 32 il values (32 independent loads in flight), adds them into
// its 32 register accumulators (-> dA[il]) and sends their sum to dC[j] with one atomicAdd per column.
template <typename T>
__global__ void __launch_bounds__(256) mlp_reduce_both_kernel(const T* __restrict__ dz1, long long ld, long long H1, long long Bk,
                                                              long long R, long long r0, float* __restrict__ dA, float* __restrict__ dC,
                                                              const int* __restrict__ run_if) {
  MI_PRED(run_if);
  constexpr int IL = 32, JG = 8;
  __shared__ float sh[IL][64];
  const int kk = threadIdx.x & 31, jg = threadIdx.x >> 5;
  const long long k = blockIdx.x * 64LL + 2 * kk;
  const long long il0 = blockIdx.y * (long long)IL;
  const bool kin = k < H1;
  float ax[IL], ay[IL];
#pragma unroll
  for (int i = 0; i < IL; ++i) { ax[i] = 0.f; ay[i] = 0.f; }
  if (kin) {
    // blockIdx.z splits the j range so that large batches (few il rows per panel) still fill the machine
    const long long jchunk = (Bk + gridDim.z - 1) / gridDim.z;
    const long long j0 = blockIdx.z * jchunk, j1 = (j0 + jchunk < Bk) ? j0 + jchunk : Bk;
    for (long long j = j0 + jg; j < j1; j += JG) {
      float sx = 0.f, sy = 0.f;
#pragma unroll
      for (int i = 0; i < IL; ++i) {
        if (il0 + i < R) {
          const T* src = dz1 + ((il0 + i) * Bk + j) * ld + k;
          float vx, vy;
          if constexpr (sizeof(T) == 2) {
            const float2 v = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(src));
            vx = v.x; vy = v.y;
          } else {
            const float2 v = *reinterpret_cast<const float2*>(src);
            vx = v.x; vy = v.y;
          }
          ax[i] += vx; ay[i] += vy; sx += vx; sy += vy;
        }
      }
      atomicAdd(dC + j * H1 + k, sx);
      atomicAdd(dC + j * H1 + k + 1, sy);
    }
  }
  for (int t = threadIdx.x; t < IL * 64; t += 256) sh[t >> 6][t & 63] = 0.f;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < IL; ++i) { atomicAdd(&sh[i][2 * kk], ax[i]); atomicAdd(&sh[i][2 * kk + 1], ay[i]); }   // 8 j groups per cell
  __syncthreads();
  for (int t = threadIdx.x; t < IL * 64; t += 256) {
    const int i = t >> 6, c = t & 63;
    if (il0 + i < R && blockIdx.x * 64LL + c < H1) atomicAdd(dA + (r0 + il0 + i) * H1 + blockIdx.x * 64LL + c, sh[i][c]);   // dA zeroed by the caller
  }
}
// out[c] = sum_r in[r, c]: a block owns 32 columns, its 8 warps stride over the rows (coalesced 128 B reads)
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ in, long long R, long long C, float* __restrict__ out) {
  __shared__ float sh[8][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long c = blockIdx.x * 32LL + lane;
  float a = 0.f;
  if (c < C) for (long long r = w; r < R; r += 8) a += in[r * C + c];
  sh[w][lane] = a;
  __syncthreads();
  if (w == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += sh[i][lane];
    out[c] = t;
  }
}
// one block: out[0] = sum in[0..n)
__global__ void sum_reduce_kernel(const float* __restrict__ in, long long n, float* __restrict__ out, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  __shared__ double sh[32];
  double a = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) a += in[i];
  for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) { double t = 0.0; for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i]; out[0] = static_cast<float>(t); }
}
// one block, after loss_finalize_kernel: t = sum of g~ over the rows' negatives (fp64); total = t, or the sum over every
// row block of the batch (`total_in`, sharded step).  The softmax weights are g~ / total, so cfac = 1 / total takes the
// sums from reference units to weights without going through e^{ref - LSE}.
// Guard (guard_out = 1, cfac = 0): total outside [1e-30, 1e30] (overflow of some e^{S - ref}, or every negative
// flushed to zero) while negatives exist (n_neg[0] > 0).  db3 = the block's share of sum of dL/dlogit over all pairs:
// t cfac - frac, frac = Bq / Bg (the positive pairs of the block); summed over the blocks: 1 - 1 (analytically 0).
__global__ void mlp_weights_kernel(const float* __restrict__ rowsum, long long n, const double* __restrict__ total_in, double frac,
                                   const double* __restrict__ n_neg, float* __restrict__ cfac, float* __restrict__ db3,
                                   double* __restrict__ guard_out) {
  __shared__ double sh[32];
  double a = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) a += rowsum[i];
  for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i];
    const double total = total_in ? total_in[0] : t;
    const bool any_neg = n_neg[0] > 0.0;
    const bool ok = total >= 1e-30 && total <= 1e30;
    const float c = (any_neg && ok) ? static_cast<float>(1.0 / total) : 0.f;
    cfac[0] = c;
    db3[0] = any_neg ? static_cast<float>(t * static_cast<double>(c) - frac) : static_cast<float>(-frac);
    if (any_neg && !ok && guard_out) guard_out[0] = 1.0;
  }
}
// one block: out[0] = sum in[0..n) in fp64 (the block's sum of g~ travels in slot 7 of its scalar row)
__global__ void sum_f64_kernel(const float* __restrict__ in, long long n, double* __restrict__ out) {
  __shared__ double sh[32];
  double a = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) a += in[i];
  for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) { double t = 0.0; for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i]; out[0] = t; }
}
// sharded step, after the merge of the blocks' scalar rows: the single pass' guard on the global sum of g~ (merged[7]),
// the same window as mlp_weights_kernel
__global__ void mlp_block_guard_kernel(const double* __restrict__ merged, double* __restrict__ loss_out) {
  const double t = merged[7];
  if (loss_out[3] > 0.0 && !(t >= 1e-30 && t <= 1e30)) loss_out[7] += 1.0;
}
// the global log-sum-exp as the float the estimator's G uses (loss_finalize_kernel's lse_f)
__global__ void lse_from_loss_kernel(const double* __restrict__ loss_out, float* __restrict__ lse_f) { lse_f[0] = (float)loss_out[2]; }
__global__ void copy_f32_kernel(const float* __restrict__ in, float* __restrict__ out, long long n) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i];
}
// x *= cfac: the single pass' sums leave reference units
__global__ void mlp_rescale_kernel(float* __restrict__ x, long long n, const float* __restrict__ cfac) {
  const float c = cfac[0];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) x[i] *= c;
}
// a += z; c += z  (the positive pairs (i, i) feed row i of dA and of dC)
__global__ void mlp_add_diag_kernel(const float* __restrict__ z, long long n, float* __restrict__ a, float* __restrict__ c) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = z[i];
    a[i] += v; c[i] += v;
  }
}

struct MlpDims { long long B, D, H1, H2; };
// Bq image rows (global rows q_off ..) against Bk text rows of a batch of Bg (single GPU: Bq = Bk = Bg, q_off = 0)
struct MlpBlock { long long Bq, Bk, q_off, Bg; const int *sid_q, *sid_k; };
struct MlpParams { const float *W1, *b1, *W2, *b2, *W3, *b3; };
struct MlpGrads { float *dX, *dY, *dW1, *db1, *dW2, *db2, *dW3, *db3; };

long long g_mlp_max_pairs = 1LL << 20;                    // bounds the panel buffers (H, dZ2, dZ1): 5 GB fast, 10 GB strict
std::atomic<int> g_mlp_mode{3};                           // bit 0: single pass for dv-like estimators, bit 1: fused dZ1 reductions
// fp32 mode (sp = 3) takes 2/3 of the pairs per panel: 13 KB per pair (H 6, dZ2 3, dZ1 4) instead of strict's 10 KB
inline long long mlp_panel_rows(long long B, long long cols, int sp) {
  long long R = (sp == 3 ? 2 * g_mlp_max_pairs / 3 : g_mlp_max_pairs) / cols;
  if (R < 1) R = 1;
  if (R > B) R = B;
  return R;
}

// The K segments of a product over K of two operands kept as sp bf16 pieces [p0 | p1 (| p2)] per row (piece t at t times
// the padded width): the terms of order < sp — p0 p0 (sp = 1); p0 p0, p1 p0, p0 p1 (strict); in fp32 mode the six terms
// smallest first, p0 p2, p1 p1, p2 p0, p0 p1, p1 p0, p0 p0: the tensor cores truncate every accumulation to the
// accumulator's precision, so the five correction segments are added while the accumulator is still ~2^-8 of its final
// size and only the p0 p0 segment's MMAs lose bits at full size.  The pieces of a K-major operand lie kb K blocks apart
// (a_seg / b_seg); those of an MN-major operand a_off / b_off rows apart (a_moff / b_noff: the padded M / N width).
// T = GemmArgs or Sched (arrays zeroed by the caller).
template <class T>
void piece_segments(T& g, int sp, long long K, bool a_mn, long long a_off, bool b_mn, long long b_off) {
  static constexpr int ta2[3] = {0, 1, 0}, tb2[3] = {0, 0, 1};
  static constexpr int ta3[6] = {0, 1, 2, 0, 1, 0}, tb3[6] = {2, 1, 0, 1, 0, 0};
  const int* ta = sp == 3 ? ta3 : ta2;
  const int* tb = sp == 3 ? tb3 : tb2;
  const bool k_pad = sp > 1 && !(a_mn && b_mn);             // K-major pieces start at round_up(K, kSplitAlign)
  const int kb = static_cast<int>(k_pad ? round_up(K, kSplitAlign) / bk() : cdiv(K, bk()));
  const int n = sp == 3 ? 6 : sp == 2 ? 3 : 1;
  g.k_blocks = n * kb; g.seg_len = kb;
  for (int s = 0; s < n; ++s) {
    if (a_mn) g.a_moff[s] = static_cast<int>(ta[s] * a_off); else g.a_seg[s] = ta[s] * kb;
    if (b_mn) g.b_noff[s] = static_cast<int>(tb[s] * b_off); else g.b_seg[s] = tb[s] * kb;
  }
}
void kk_segments(GemmArgs& g, int sp, long long K) { piece_segments(g, sp, K, false, 0, false, 0); }

// fp32 mode: the longest accumulation chain into one TMEM accumulator, in K elements (64 K blocks with CTA pairs, 128
// single-CTA).  The tensor cores truncate each accumulation (DESIGN 3.4: a chain of n MMAs loses ~n 2^-25 relative), so
// the contractions over pairs (dW2) and rows (dW1) are cut into split-K partial tiles of at most this length, summed by
// reduce_partials_kernel in fp32 with round-to-nearest.  The contractions that feed an epilogue (Z2 over H1, dZ1 over H2,
// layer 1 over D) cannot be split: mlp_dims_ok keeps them within one chain (6 round_up(K, 128) <= kFp32ChainK).
constexpr long long kFp32ChainK = 8192;
long long mlp_chain_min_ks(int sp, int k_blocks) { return sp == 3 ? cdiv(static_cast<long long>(k_blocks) * bk(), kFp32ChainK) : 1; }

// memset that respects the launch predicate of this thread
int zero_async(void* p, size_t bytes, cudaStream_t stream) {
  if (bytes == 0) return MI_OK;
  if (t_run_if == nullptr) { MI_CUDA(cudaMemsetAsync(p, 0, bytes, stream)); return MI_OK; }
  const long long n16 = static_cast<long long>((bytes + 15) / 16);       // workspace blocks are 256 B aligned and padded
  zero_u4_kernel<<<blocks_capped(n16, 256), 256, 0, stream>>>(static_cast<uint4*>(p), n16, t_run_if);
  MI_LAUNCH_CHECK("zero_u4_kernel");
  return MI_OK;
}

// everything the two sequences share: dimensions, operands, scratch
struct MlpCtx {
  long long Bq, Bk, q_off, Bg, D, H1, H2, Dp, Hp, H2p, pX, pH, pZ, eX, eH, eZ, h2_pad;
  int sp, nt2, estimator;
  const int *sid_q, *sid_k;
  MlpParams prm;
  __nv_bfloat16 *X16, *Y16, *W1x, *W1y, *W2h, *Hpan, *DZ2, *DZ1h, *dA16, *dC16;
  float *A32, *C32, *b2p, *w3p, *S, *rows_r, *lse_f, *part, *G, *DZ1, *dA32, *dC32, *acc_w3, *acc_b2, *dW2, *db3v;
  float *col_part, *col_lse, *cols_r;     // symmetric InfoNCE: column partials, column log-sum-exp, column float4s
  double *scal, *scal_col;
  double* loss_out;
  cudaStream_t stream;
  size_t mk;
};

// the dZ2 epilogues: their three-piece form in fp32 mode
template <class Epi, class Epi3>
int mlp_launch_dz(const MlpCtx& c, const MapSpec& a, const MapSpec& b, const Sched& sc, const typename Epi::Params& ep) {
  return c.sp == 3 ? launch_engine<Epi3>(a, b, sc, ep, c.stream) : launch_engine<Epi>(a, b, sc, ep, c.stream);
}
// Z2 = H W2^T over one panel of P pairs, handed to an epilogue policy
void mlp_z2_sched(const MlpCtx& c, long long P, Sched& sc) {
  sc.n_mblk = static_cast<int>(cdiv(P, rows_per_mblk()));
  sc.n_ntile = c.nt2; sc.n_split = 1; sc.n_ksplit = 1; sc.order = 0;
  single_segment(sc);
  piece_segments(sc, c.sp, c.H1, false, 0, false, 0);
}
// dW2 (+)= dZ2^T H : contraction over the panel's pairs, both operands MN-major
int mlp_dw2_gemm(const MlpCtx& c, long long P, bool accumulate, Bump& ws) {
  GemmArgs g;
  g.a_mn = true; g.a = MapSpec{c.DZ2, P, c.eZ, c.pZ};
  g.b_mn = true; g.b = MapSpec{c.Hpan, P, c.eH, c.pH};
  g.M = c.H2; g.N = c.H1;
  piece_segments(g, c.sp, P, true, c.H2p, true, c.Hp);
  const long long tiles = cdiv(c.H2, rows_per_mblk()) * cdiv(c.H1, mi::TILE_N);
  g.ksplit = choose_ksplit(tiles, g.k_blocks, mlp_chain_min_ks(c.sp, g.k_blocks));
  g.order = 0;      // the 8 tiles of a K split stream the same rows of dZ2 / H: neighbours share them in L2
  g.out_f32 = c.dW2; g.ld_out = c.H1; g.accumulate = accumulate;
  if (ws.dry) g.out_f32 = reinterpret_cast<float*>(16);
  MI_TRY(run_gemm(g, ws, c.stream));
  ws.release(c.mk);
  return MI_OK;
}
// dZ1 = (dZ2 W2) . [H > 0] as a stored panel: W2 [H2, H1] read in place as the MN-major B operand
int mlp_dz1_gemm(const MlpCtx& c, long long P, float* out_f32, __nv_bfloat16* out_bf16, Bump& ws) {
  GemmArgs g;
  g.a = MapSpec{c.DZ2, P, c.eZ, c.pZ};
  g.b_mn = true; g.b = MapSpec{c.W2h, c.H2, c.eH, c.pH};
  g.M = P; g.N = c.H1;
  piece_segments(g, c.sp, c.H2, false, 0, true, c.Hp);
  g.out_f32 = out_f32; g.ld_out = c.H1; g.out_bf16 = out_bf16; g.ld_out16 = c.H1; g.relu_mask = c.Hpan; g.ld_mask = c.pH;
  if (ws.dry) g.out_f32 = reinterpret_cast<float*>(16);
  MI_TRY(run_gemm(g, ws, c.stream));
  ws.release(c.mk);
  return MI_OK;
}
int mlp_reduce_panel(const MlpCtx& c, long long cols, long long rr, long long r0) {
  dim3 rg(static_cast<unsigned>(cdiv(c.H1, 64)), static_cast<unsigned>(cdiv(rr, 32)), 1);
  const long long blocks = static_cast<long long>(rg.x) * rg.y;
  long long jz = blocks >= num_sms() ? 1 : cdiv(4LL * num_sms(), blocks);
  if (jz > cols / 64) jz = cols / 64;
  rg.z = static_cast<unsigned>(jz < 1 ? 1 : jz);
  if (c.sp == 1) mlp_reduce_both_kernel<__nv_bfloat16><<<rg, 256, 0, c.stream>>>(c.DZ1h, c.H1, c.H1, cols, rr, r0, c.dA32, c.dC32, t_run_if);
  else mlp_reduce_both_kernel<float><<<rg, 256, 0, c.stream>>>(c.DZ1, c.H1, c.H1, cols, rr, r0, c.dA32, c.dC32, t_run_if);
  MI_LAUNCH_CHECK("mlp_reduce_both_kernel");
  return MI_OK;
}
int mlp_zero_accumulators(const MlpCtx& c, long long dc_rows) {
  MI_TRY(zero_async(c.dC32, static_cast<size_t>(dc_rows) * c.H1 * sizeof(float), c.stream));
  MI_TRY(zero_async(c.dA32, static_cast<size_t>(c.Bq) * c.H1 * sizeof(float), c.stream));
  MI_TRY(zero_async(c.acc_w3, static_cast<size_t>(c.h2_pad) * sizeof(float), c.stream));
  MI_TRY(zero_async(c.acc_b2, static_cast<size_t>(c.h2_pad) * sizeof(float), c.stream));
  return MI_OK;
}

// ---- the two-pass sequence: logits of every pair -> estimator -> recompute Z2 for the backward.  Exact for every input
//      (running-max statistics); every estimator.  All launches carry this thread's launch predicate.
int mlp_tp_gen_panel(const MlpCtx& c, long long r0, long long P) {
  mlp_gen_kernel<<<blocks_capped(P * (c.H1 >> 3), 256), 256, 0, c.stream>>>(c.A32, c.C32, c.H1, c.Bk, r0, P, c.Hpan, c.pH, c.Hp, c.sp, 0, 0,
                                                                           t_run_if);
  MI_LAUNCH_CHECK("mlp_gen_kernel");
  return MI_OK;
}
// forward: the logits S [Bq, Bk] of the block, its row statistics (c.rows_r) and its scalar row (c.scal)
int mlp_tp_fwd(const MlpCtx& c, bool dry) {
  if (dry) return MI_OK;
  const long long Bq = c.Bq, Bk = c.Bk, H2 = c.H2;
  cudaStream_t stream = c.stream;
  const long long R = mlp_panel_rows(Bq, Bk, c.sp);
  for (long long r0 = 0; r0 < Bq; r0 += R) {
    const long long rr = (Bq - r0 < R) ? (Bq - r0) : R, P = rr * Bk;
    MI_TRY(mlp_tp_gen_panel(c, r0, P));
    Sched sc; mlp_z2_sched(c, P, sc);
    mi::EpiMlpFwd::Params ep;
    ep.b2 = c.b2p; ep.w3 = c.w3p; ep.part = c.part; ep.rows_padded = sc.n_mblk * rows_per_mblk();
    MI_TRY(launch_engine<mi::EpiMlpFwd>(MapSpec{c.Hpan, P, c.eH, c.pH}, MapSpec{c.W2h, H2, c.eH, c.pH}, sc, ep, stream));
    mlp_logit_merge_kernel<<<blocks_for(P, 256), 256, 0, stream>>>(c.part, ep.rows_padded, P, c.prm.b3, c.S + r0 * Bk, t_run_if);
    MI_LAUNCH_CHECK("mlp_logit_merge_kernel");
  }
  // ---- estimator on S (same reductions and fp64 finalisation as the separable critics)
  mlp_row_stats_kernel<<<blocks_for(Bq * 32, 256), 256, 0, stream>>>(c.S, c.sid_q, c.sid_k, Bq, Bk, c.q_off,
                                                                     reinterpret_cast<float4*>(c.rows_r), t_run_if);
  MI_LAUNCH_CHECK("mlp_row_stats_kernel");
  stats_reduce_kernel<<<1, 1024, 0, stream>>>(reinterpret_cast<const float4*>(c.rows_r), static_cast<int>(Bq), c.scal, t_run_if);
  MI_LAUNCH_CHECK("stats_reduce_kernel");
  return MI_OK;
}
// column statistics of the block's stored logits (symmetric InfoNCE): col_lse [Bk] as mlp_col_merge_kernel; `square`
// (the block is the batch): also the columns' float4s (c.cols_r) reduced to the scalar row c.scal_col.  The row slices
// fill the machine: Bk / 256 column blocks alone are 16 - 32 blocks at Bk = 4096 - 8192.
int mlp_col_stats(const MlpCtx& c, float* col_lse, bool square) {
  const unsigned gx = blocks_for(c.Bk, 256);
  long long ny = cdiv(4LL * num_sms(), gx);
  if (ny > kMlpColSplits) ny = kMlpColSplits;
  if (ny > c.Bq) ny = c.Bq;
  mlp_col_part_kernel<<<dim3(gx, static_cast<unsigned>(ny)), 256, 0, c.stream>>>(c.S, c.sid_q, c.sid_k, c.Bq, c.Bk, c.col_part, t_run_if);
  MI_LAUNCH_CHECK("mlp_col_part_kernel");
  float4* cols = square ? reinterpret_cast<float4*>(c.cols_r) : nullptr;
  mlp_col_merge_kernel<<<gx, 256, 0, c.stream>>>(c.col_part, static_cast<int>(ny), c.S, c.Bq, c.Bk, c.q_off, col_lse, cols, t_run_if);
  MI_LAUNCH_CHECK("mlp_col_merge_kernel");
  if (square) {
    stats_reduce_kernel<<<1, 1024, 0, c.stream>>>(cols, static_cast<int>(c.Bk), c.scal_col, t_run_if);
    MI_LAUNCH_CHECK("stats_reduce_kernel");
  }
  return MI_OK;
}
// backward, once the loss is known (c.lse_f: the global log-sum-exp; c.rows_r: the block's row statistics; c.col_lse:
// symmetric InfoNCE, the log-sum-exp of every column over the batch): G, then Z2
// recomputed panel by panel.  `resident`: the forward's only panel is still in c.Hpan.
int mlp_tp_bwd(const MlpCtx& c, bool resident, Bump& ws) {
  const long long Bq = c.Bq, Bk = c.Bk, H2 = c.H2;
  const bool dry = ws.dry;
  cudaStream_t stream = c.stream;
  const long long R = mlp_panel_rows(Bq, Bk, c.sp);
  if (!dry) {
    const int dv_like = (c.estimator == MI_EST_DV || c.estimator == MI_EST_INFONCE_REF) ? 1 : 0;
    const float* col_lse = c.estimator == MI_EST_INFONCE_SYM ? c.col_lse : nullptr;
    mlp_g_kernel<<<blocks_for(Bq * Bk, 256), 256, 0, stream>>>(c.S, c.sid_q, c.sid_k, Bq, Bk, c.q_off, c.Bg, dv_like, c.lse_f,
                                                               reinterpret_cast<const float4*>(c.rows_r), col_lse, c.G, t_run_if);
    MI_LAUNCH_CHECK("mlp_g_kernel");
    MI_TRY(mlp_zero_accumulators(c, Bk));
  }
  for (long long r0 = 0; r0 < Bq; r0 += R) {
    const long long rr = (Bq - r0 < R) ? (Bq - r0) : R, P = rr * Bk;
    if (!dry) {
      if (!resident) MI_TRY(mlp_tp_gen_panel(c, r0, P));
      Sched sc; mlp_z2_sched(c, P, sc);
      mi::EpiMlpDz::Params ep;
      ep.b2 = c.b2p; ep.w3 = c.w3p; ep.g = c.G + r0 * Bk; ep.rows = static_cast<int>(P); ep.cols = static_cast<int>(H2);
      ep.dz = c.DZ2; ep.dz_lo = c.sp >= 2 ? c.DZ2 + c.H2p : nullptr; ep.dz_lo2 = c.sp == 3 ? c.DZ2 + 2 * c.H2p : nullptr; ep.pitch = c.pZ; ep.dw3 = c.acc_w3; ep.db2 = c.acc_b2;
      MI_TRY((mlp_launch_dz<mi::EpiMlpDz, mi::EpiMlpDz3>(c, MapSpec{c.Hpan, P, c.eH, c.pH}, MapSpec{c.W2h, H2, c.eH, c.pH}, sc, ep)));
    }
    MI_TRY(mlp_dw2_gemm(c, P, r0 > 0, ws));
    MI_TRY(mlp_dz1_gemm(c, P, c.sp >= 2 ? c.DZ1 : nullptr, c.sp == 1 ? c.DZ1h : nullptr, ws));
    if (!dry) MI_TRY(mlp_reduce_panel(c, Bk, rr, r0));
  }
  if (!dry) {
    sum_reduce_kernel<<<1, 1024, 0, stream>>>(c.G, Bq * Bk, c.db3v, t_run_if);
    MI_LAUNCH_CHECK("sum_reduce_kernel");
  }
  return MI_OK;
}
// the whole two-pass step of one GPU (the block is the batch)
int mlp_two_pass(const MlpCtx& c, bool plan, Bump& ws) {
  MI_TRY(mlp_tp_fwd(c, ws.dry));
  if (!ws.dry) {
    const bool sym = c.estimator == MI_EST_INFONCE_SYM;
    if (sym) MI_TRY(mlp_col_stats(c, c.col_lse, true));
    loss_finalize_kernel<<<1, 32, 0, c.stream>>>(c.scal, sym ? c.scal_col : nullptr, c.Bg, c.estimator, c.loss_out, c.lse_f, nullptr,
                                                 t_run_if);
    MI_LAUNCH_CHECK("loss_finalize_kernel");
  }
  if (!plan) return MI_OK;
  return mlp_tp_bwd(c, mlp_panel_rows(c.Bq, c.Bk, c.sp) >= c.Bq, ws);
}

// reference of the single pass: the maximum logit over an n x n strided sample of the block's OWN pairs (image rows
// x the text rows at the same global indices; the margin is added in the epilogue)
constexpr long long kMlpRefSample = 256;
int mlp_reference_logit(const MlpCtx& c, float* As, float* Cs, float* Ssmp, float* ref) {
  const long long ns = c.Bq < kMlpRefSample ? c.Bq : kMlpRefSample, stride = c.Bq / ns, P = ns * ns;
  cudaStream_t stream = c.stream;
  gather_rows_kernel<<<blocks_for(ns * c.H1, 256), 256, 0, stream>>>(c.A32, stride, c.H1, As, ns);
  MI_LAUNCH_CHECK("gather_rows_kernel");
  gather_rows_kernel<<<blocks_for(ns * c.H1, 256), 256, 0, stream>>>(c.C32 + c.q_off * c.H1, stride, c.H1, Cs, ns);
  MI_LAUNCH_CHECK("gather_rows_kernel");
  mlp_gen_kernel<<<blocks_capped(P * (c.H1 >> 3), 256), 256, 0, stream>>>(As, Cs, c.H1, ns, 0, P, c.Hpan, c.pH, c.Hp, c.sp, 0, 0, nullptr);
  MI_LAUNCH_CHECK("mlp_gen_kernel");
  Sched sc; mlp_z2_sched(c, P, sc);
  mi::EpiMlpFwd::Params ep;
  ep.b2 = c.b2p; ep.w3 = c.w3p; ep.part = c.part; ep.rows_padded = sc.n_mblk * rows_per_mblk();
  MI_TRY(launch_engine<mi::EpiMlpFwd>(MapSpec{c.Hpan, P, c.eH, c.pH}, MapSpec{c.W2h, c.H2, c.eH, c.pH}, sc, ep, stream));
  mlp_logit_merge_kernel<<<blocks_for(P, 256), 256, 0, stream>>>(c.part, ep.rows_padded, P, c.prm.b3, Ssmp, nullptr);
  MI_LAUNCH_CHECK("mlp_logit_merge_kernel");
  max_reduce_kernel<<<1, 1024, 0, stream>>>(Ssmp, P, ref, 0.f, nullptr);
  MI_LAUNCH_CHECK("max_reduce_kernel");
  return MI_OK;
}

// image rows walked per unit of the fused dZ1 kernel: the unit count should fill whole rounds of the CTA pairs
void mlp_da_chunks(long long rr, long long per_chunk_units, int& chunk_len, int& n_chunks) {
  const long long U = num_pairs();
  const long long min_len = rr < 32 ? rr : 32;          // the flush of a unit's running sums is amortised over >= 32 tiles
  double best = -1.0;
  chunk_len = static_cast<int>(rr); n_chunks = 1;
  const long long nc_max = rr / min_len < 1 ? 1 : rr / min_len;         // full-length chunks stay >= min_len
  for (long long nc = 1; nc <= nc_max; ++nc) {
    const long long len = cdiv(rr, nc), real_nc = cdiv(rr, len), units = per_chunk_units * real_nc;
    const double eff = static_cast<double>(units) / static_cast<double>(cdiv(units, U) * U);
    if (eff > best + 1e-9) { best = eff; chunk_len = static_cast<int>(len); n_chunks = static_cast<int>(real_nc); }
  }
}

// ---- the single pass (dv / infonce): see the header of this file
struct MlpSpBuf { float *As, *Cs, *Ssmp, *ref, *cfac, *rowsum, *rowcnt, *diag, *gd, *DZ1d; uint32_t* mask; int* flag; double* guard_a; };
// the panels against the reference sb.ref: raw accumulators in reference units (dW2, dA, dC, dw3, db2), the rows' sums of
// g~ (sb.rowsum) and the block's scalar row (c.scal)
int mlp_sp_panels(const MlpCtx& c, const MlpSpBuf& sb, float* S_out, Bump& ws) {
  const long long Bq = c.Bq, Bk = c.Bk, H1 = c.H1, H2 = c.H2;
  const bool dry = ws.dry;
  cudaStream_t stream = c.stream;
  const long long Bp = round_up(Bk, rows_per_mblk());
  const long long R = mlp_panel_rows(Bq, Bp, c.sp);
  const int wpr = static_cast<int>(round_up(cdiv(H1, 32), 2));          // even: the epilogue reads word pairs
  const bool fused_da = (g_mlp_mode.load(std::memory_order_relaxed) & 2) != 0;
  if (!dry) {
    MI_TRY(mlp_zero_accumulators(c, Bp));
    MI_CUDA(cudaMemsetAsync(sb.rowsum, 0, static_cast<size_t>(2 * Bq) * sizeof(float), stream));      // rowsum | rowcnt
  }
  for (long long r0 = 0; r0 < Bq; r0 += R) {
    const long long rr = (Bq - r0 < R) ? (Bq - r0) : R, P = rr * Bp;
    if (!dry) {
      {
        dim3 gg(blocks_for(cdiv(Bp, kGenJ) * 4 * wpr, 256), 1, 1);
        long long ny = cdiv(16LL * num_sms(), gg.x);              // enough blocks in flight to saturate the HBM writes
        if (ny > rr) ny = rr;
        gg.y = static_cast<unsigned>(ny < 1 ? 1 : ny);
        if (c.sp == 3) mlp_gen2_kernel<true><<<gg, 256, 0, stream>>>(c.A32, c.C32, H1, Bk, Bp, r0, rr, c.Hpan, c.pH, c.Hp, c.sp, sb.mask, wpr);
        else mlp_gen2_kernel<false><<<gg, 256, 0, stream>>>(c.A32, c.C32, H1, Bk, Bp, r0, rr, c.Hpan, c.pH, c.Hp, c.sp, sb.mask, wpr);
        MI_LAUNCH_CHECK("mlp_gen2_kernel");
      }
      Sched sc; mlp_z2_sched(c, P, sc);
      mi::EpiMlpSp::Params ep;
      ep.b2 = c.b2p; ep.w3 = c.w3p; ep.b3 = c.prm.b3; ep.ref = sb.ref; ep.sid_q = c.sid_q; ep.sid_k = c.sid_k;
      ep.B = static_cast<int>(Bk); ep.Bp = static_cast<int>(Bp); ep.r0 = static_cast<int>(r0); ep.rr = static_cast<int>(rr);
      ep.q_off = static_cast<int>(c.q_off);
      ep.cols = static_cast<int>(H2);
      ep.dz = c.DZ2; ep.dz_lo = c.sp >= 2 ? c.DZ2 + c.H2p : nullptr; ep.dz_lo2 = c.sp == 3 ? c.DZ2 + 2 * c.H2p : nullptr; ep.pitch = c.pZ; ep.dw3 = c.acc_w3; ep.db2 = c.acc_b2;
      ep.rowsum = sb.rowsum; ep.rowcnt = sb.rowcnt; ep.diag_out = sb.diag; ep.S_out = S_out;
      MI_TRY((mlp_launch_dz<mi::EpiMlpSp, mi::EpiMlpSp3>(c, MapSpec{c.Hpan, P, c.eH, c.pH}, MapSpec{c.W2h, H2, c.eH, c.pH}, sc, ep)));
    }
    MI_TRY(mlp_dw2_gemm(c, P, r0 > 0, ws));
    if (fused_da) {
      if (!dry) {
        Sched sc;
        single_segment(sc);
        sc.order = 2;
        sc.n_ntile = static_cast<int>(cdiv(H1, mi::TILE_N));
        sc.grp = static_cast<int>(Bp / rows_per_mblk()); sc.n_il = static_cast<int>(rr);
        mlp_da_chunks(rr, static_cast<long long>(sc.n_ntile) * sc.grp, sc.chunk_len, sc.n_chunks);
        sc.n_mblk = sc.grp * sc.n_il; sc.n_split = 1; sc.n_ksplit = 1;
        piece_segments(sc, c.sp, H2, false, 0, true, c.Hp);
        mi::EpiMlpDa::Params ep;
        ep.mask = sb.mask; ep.wpr = wpr; ep.B = static_cast<int>(Bk); ep.Bp = static_cast<int>(Bp);
        ep.r0 = static_cast<int>(r0); ep.rr = static_cast<int>(rr); ep.cols = static_cast<int>(H1);
        ep.dA = c.dA32; ep.dC = c.dC32;
        MI_TRY((launch_engine<mi::EpiMlpDa, false, true>(MapSpec{c.DZ2, P, c.eZ, c.pZ}, MapSpec{c.W2h, H2, c.eH, c.pH}, sc, ep, stream)));
      }
    } else {
      MI_TRY(mlp_dz1_gemm(c, P, c.sp >= 2 ? c.DZ1 : nullptr, c.sp == 1 ? c.DZ1h : nullptr, ws));
      if (!dry) MI_TRY(mlp_reduce_panel(c, Bp, rr, r0));
    }
  }
  if (!dry) {
    // ---- estimator: row statistics from the sums, reduced like the separable critics' rows
    mlp_rows_from_sums_kernel<<<blocks_for(Bq, 256), 256, 0, stream>>>(sb.rowsum, sb.rowcnt, sb.diag, sb.ref, Bq, reinterpret_cast<float4*>(c.rows_r));
    MI_LAUNCH_CHECK("mlp_rows_from_sums_kernel");
    stats_reduce_kernel<<<1, 1024, 0, stream>>>(reinterpret_cast<const float4*>(c.rows_r), static_cast<int>(Bq), c.scal, nullptr);
    MI_LAUNCH_CHECK("stats_reduce_kernel");
  }
  return MI_OK;
}
// the rest of the single pass once the loss is known (c.loss_out: n_neg of the batch; `total`: the sum of g~ over every
// row block, NULL = this block is the batch; `guard_out`: where a trip of the weights' guard is reported, or NULL):
// softmax weights, reference units -> weights, and the block's positive pairs (i, q_off + i): dL/dlogit = -1/Bg
// (mi_critics.py:6,18), one panel of Bq pairs
int mlp_sp_finish(const MlpCtx& c, const MlpSpBuf& sb, const double* total, double* guard_out, Bump& ws) {
  const long long Bq = c.Bq, Bk = c.Bk, H1 = c.H1, H2 = c.H2;
  const bool dry = ws.dry;
  cudaStream_t stream = c.stream;
  if (!dry) {
    mlp_weights_kernel<<<1, 1024, 0, stream>>>(sb.rowsum, Bq, total, static_cast<double>(Bq) / static_cast<double>(c.Bg), c.loss_out + 3,
                                               sb.cfac, c.db3v, guard_out);
    MI_LAUNCH_CHECK("mlp_weights_kernel");
    float* bufs[5] = {c.dW2, c.dA32, c.dC32, c.acc_w3, c.acc_b2};
    const long long lens[5] = {H2 * H1, Bq * H1, Bk * H1, c.h2_pad, c.h2_pad};
    for (int t = 0; t < 5; ++t) {
      mlp_rescale_kernel<<<blocks_capped(lens[t], 256), 256, 0, stream>>>(bufs[t], lens[t], sb.cfac);
      MI_LAUNCH_CHECK("mlp_rescale_kernel");
    }
    mlp_gen_kernel<<<blocks_capped(Bq * (H1 >> 3), 256), 256, 0, stream>>>(c.A32, c.C32, H1, Bk, 0, Bq, c.Hpan, c.pH, c.Hp, c.sp, 1, c.q_off,
                                                                          nullptr);
    MI_LAUNCH_CHECK("mlp_gen_kernel");
    fill_f32_kernel<<<blocks_for(Bq, 256), 256, 0, stream>>>(sb.gd, Bq, -1.f / static_cast<float>(c.Bg));
    MI_LAUNCH_CHECK("fill_f32_kernel");
    Sched sc; mlp_z2_sched(c, Bq, sc);
    mi::EpiMlpDz::Params ep;
    ep.b2 = c.b2p; ep.w3 = c.w3p; ep.g = sb.gd; ep.rows = static_cast<int>(Bq); ep.cols = static_cast<int>(H2);
    ep.dz = c.DZ2; ep.dz_lo = c.sp >= 2 ? c.DZ2 + c.H2p : nullptr; ep.dz_lo2 = c.sp == 3 ? c.DZ2 + 2 * c.H2p : nullptr; ep.pitch = c.pZ; ep.dw3 = c.acc_w3; ep.db2 = c.acc_b2;
    MI_TRY((mlp_launch_dz<mi::EpiMlpDz, mi::EpiMlpDz3>(c, MapSpec{c.Hpan, Bq, c.eH, c.pH}, MapSpec{c.W2h, H2, c.eH, c.pH}, sc, ep)));
  }
  MI_TRY(mlp_dw2_gemm(c, Bq, true, ws));
  MI_TRY(mlp_dz1_gemm(c, Bq, sb.DZ1d, nullptr, ws));
  if (!dry) {
    mlp_add_diag_kernel<<<blocks_capped(Bq * H1, 256), 256, 0, stream>>>(sb.DZ1d, Bq * H1, c.dA32, c.dC32 + c.q_off * H1);
    MI_LAUNCH_CHECK("mlp_add_diag_kernel");
  }
  return MI_OK;
}

void mlp_ctx_dims(MlpCtx& c, long long D, long long H1, long long H2, int precision) {
  c.D = D; c.H1 = H1; c.H2 = H2;
  c.sp = precision == MI_PREC_FP32X3 ? 3 : (precision & 1) == MI_PREC_BF16_STRICT ? 2 : 1;
  const int sp = c.sp;
  c.Dp = round_up(D, kSplitAlign); c.Hp = round_up(H1, kSplitAlign); c.H2p = round_up(H2, kSplitAlign);
  c.pX = sp > 1 ? sp * c.Dp : D; c.pH = sp > 1 ? sp * c.Hp : H1; c.pZ = sp > 1 ? sp * c.H2p : H2;
  c.eX = (sp - 1) * c.Dp + D; c.eH = (sp - 1) * c.Hp + H1; c.eZ = (sp - 1) * c.H2p + H2;   // TMA extents
  c.nt2 = static_cast<int>(cdiv(H2, mi::TILE_N));
  c.h2_pad = static_cast<long long>(c.nt2) * mi::TILE_N;
}
// precision: MI_PREC_BF16_FAST, MI_PREC_BF16_STRICT or MI_PREC_FP32X3; fp32 mode also needs the unsplittable contractions
// over D and H1 (layer 1, Z2) to stay within one bounded chain (kFp32ChainK): D, H1 <= 1280
bool mlp_precision_ok(int precision, long long D, long long H1) {
  if (precision == MI_PREC_BF16_FAST || precision == MI_PREC_BF16_STRICT) return true;
  return precision == MI_PREC_FP32X3 && 6 * round_up(D, kSplitAlign) <= kFp32ChainK && 6 * round_up(H1, kSplitAlign) <= kFp32ChainK;
}
bool mlp_dims_ok(const MlpDims& d, int estimator, int precision) {
  if (d.B <= 0 || d.D <= 0 || d.H1 <= 0 || d.H2 <= 0 || (d.D % 8) != 0 || (d.H1 % 8) != 0 || (d.H2 % 8) != 0) return false;
  if (d.H2 > mi::EpiMlpDz::kMaxTiles * mi::TILE_N) return false;
  if (!mlp_precision_ok(precision, d.D, d.H1)) return false;
  return estimator == MI_EST_DV || estimator == MI_EST_INFONCE_REF || estimator == MI_EST_INFONCE_ROW || estimator == MI_EST_INFONCE_SYM;
}
// fp32 [R, C] (pitch ld_in) -> the bf16 operand (c.sp pieces, see split_f32_kernel) of pitch `pitch`, piece t at column t Cp
int mlp_split(const MlpCtx& c, const float* in, long long ld_in, __nv_bfloat16* out, long long pitch, long long Cp, long long R, long long C) {
  if (c.sp == 3) split_f32_kernel<true><<<blocks_for(R * pitch, 256), 256, 0, c.stream>>>(in, ld_in, out, pitch, c.sp, Cp, R, C, nullptr);
  else split_f32_kernel<false><<<blocks_for(R * pitch, 256), 256, 0, c.stream>>>(in, ld_in, out, pitch, c.sp, Cp, R, C, nullptr);
  MI_LAUNCH_CHECK("split_f32_kernel");
  return MI_OK;
}

// Carves the buffers of the MLP path over a block and runs its prologue: bf16 operands, layer 1 (A = X W1x^T + b1 for the
// Bq image rows, C = Y W1y^T for the Bk text rows; fp32 out).  What the sharded step keeps between its forward and its
// backward call (logits, row statistics, raw accumulators) comes from `keep`, the caller-owned state; on a single GPU
// `keep` is the workspace itself.  `args_ok`: the caller's own pointer checks (reported after the workspace check).
int mlp_setup(MlpCtx& c, MlpSpBuf& sb, const float* X, const float* Y, const MlpParams& prm, const MlpBlock& blk, const MlpDims& d,
              int estimator, int precision, bool plan, float* S_out, float* dW2_out, double* loss_out, bool args_ok,
              Bump& ws, Bump& keep, cudaStream_t stream) {
  if (blk.Bq <= 0 || blk.Bk <= 0 || blk.q_off < 0 || blk.q_off + blk.Bq > blk.Bk || blk.Bk > blk.Bg) return MI_ERR_BAD_ARG;
  typedef __nv_bfloat16 bf;
  const long long Bq = blk.Bq, Bk = blk.Bk, D = d.D, H1 = d.H1, H2 = d.H2;
  c.Bq = Bq; c.Bk = Bk; c.q_off = blk.q_off; c.Bg = blk.Bg; c.sid_q = blk.sid_q; c.sid_k = blk.sid_k;
  c.estimator = estimator; c.prm = prm; c.stream = stream; c.loss_out = loss_out;
  mlp_ctx_dims(c, D, H1, H2, precision);
  const int sp = c.sp;
  const long long Bp = round_up(Bk, rows_per_mblk());
  const long long Pmax1 = mlp_panel_rows(Bq, Bk, sp) * Bk, Pmax2 = mlp_panel_rows(Bq, Bp, sp) * Bp;
  const long long ns_ref = Bq < kMlpRefSample ? Bq : kMlpRefSample;      // the reference-logit sample is a panel too
  long long Pmax = Pmax1 > Pmax2 ? Pmax1 : Pmax2;
  if (Pmax < ns_ref * ns_ref) Pmax = ns_ref * ns_ref;
  const long long rows_padded_max = cdiv(Pmax, rows_per_mblk()) * rows_per_mblk();
  const long long pX = c.pX, pH = c.pH, pZ = c.pZ;

  c.X16 = ws.take<bf>(Bq * pX); c.Y16 = ws.take<bf>(Bk * pX);
  c.W1x = ws.take<bf>(H1 * pX); c.W1y = ws.take<bf>(H1 * pX);
  c.W2h = ws.take<bf>(H2 * pH);
  c.A32 = ws.take<float>(Bq * H1); c.C32 = ws.take<float>(Bk * H1);
  c.b2p = ws.take<float>(c.h2_pad); c.w3p = ws.take<float>(c.h2_pad);
  c.S = S_out ? S_out : keep.take<float>(Bq * Bk);
  c.rows_r = keep.take<float>(Bq * 4);
  c.scal = ws.take<double>(8);
  // symmetric InfoNCE: planned by every size query (it does not know the estimator), carved only for this estimator
  const bool cols = ws.dry || estimator == MI_EST_INFONCE_SYM;
  c.col_part = cols ? ws.take<float>(3LL * kMlpColSplits * Bk) : nullptr;
  c.col_lse = cols ? ws.take<float>(Bk) : nullptr;
  c.cols_r = cols ? ws.take<float>(Bk * 4) : nullptr;
  c.scal_col = cols ? ws.take<double>(8) : nullptr;
  c.lse_f = ws.take<float>(1);
  c.db3v = ws.take<float>(1);
  c.Hpan = ws.take<bf>(Pmax * pH);
  c.part = ws.take<float>(mi::kColQuarters * rows_padded_max);
  c.G = plan ? ws.take<float>(Bq * Bk) : nullptr;
  c.DZ2 = plan ? ws.take<bf>(Pmax * pZ) : nullptr;
  // dZ1 panel: bf16 in fast mode (half the bytes of the HBM-write-bound masked contraction), fp32 in strict / fp32 mode
  c.DZ1 = (plan && sp >= 2) ? ws.take<float>(Pmax * H1) : nullptr;
  c.DZ1h = (plan && sp == 1) ? ws.take<bf>(Pmax * H1) : nullptr;
  c.dA32 = plan ? keep.take<float>(Bq * H1) : nullptr; c.dC32 = plan ? keep.take<float>(Bp * H1) : nullptr;
  c.dA16 = plan ? ws.take<bf>(Bq * pH) : nullptr; c.dC16 = plan ? ws.take<bf>(Bk * pH) : nullptr;
  c.acc_w3 = plan ? keep.take<float>(c.h2_pad) : nullptr; c.acc_b2 = plan ? keep.take<float>(c.h2_pad) : nullptr;
  float* dW2_tmp = (plan && !dW2_out) ? keep.take<float>(H2 * H1) : nullptr;
  if (plan) {
    const long long ns = ns_ref;
    sb.As = ws.take<float>(ns * H1); sb.Cs = ws.take<float>(ns * H1); sb.Ssmp = ws.take<float>(ns * ns);
    sb.ref = ws.take<float>(1); sb.cfac = ws.take<float>(1);
    sb.rowsum = keep.take<float>(2 * Bq); sb.rowcnt = sb.rowsum ? sb.rowsum + Bq : nullptr;
    sb.diag = keep.take<float>(Bq); sb.gd = ws.take<float>(Bq);
    sb.DZ1d = ws.take<float>(Bq * H1);
    sb.mask = ws.take<uint32_t>(Pmax2 * round_up(cdiv(H1, 32), 2));
    sb.flag = ws.take<int>(1); sb.guard_a = ws.take<double>(1);
  }
  if (!ws.ok() || !keep.ok()) return MI_ERR_WORKSPACE;
  c.mk = ws.mark();
  c.dW2 = dW2_out ? dW2_out : dW2_tmp;
  const size_t mk = c.mk;
  const bool dry = ws.dry;
  if (!dry && (!args_ok || !X || !Y || !prm.W1 || !prm.b1 || !prm.W2 || !prm.b2 || !prm.W3 || !prm.b3)) return MI_ERR_BAD_ARG;

  if (!dry) {
    MI_TRY(mlp_split(c, X, D, c.X16, pX, c.Dp, Bq, D));
    MI_TRY(mlp_split(c, Y, D, c.Y16, pX, c.Dp, Bk, D));
    MI_TRY(mlp_split(c, prm.W1, 2 * D, c.W1x, pX, c.Dp, H1, D));            // W1 = [W1x | W1y]  (nn.Linear weight [H1, 2D])
    MI_TRY(mlp_split(c, prm.W1 + D, 2 * D, c.W1y, pX, c.Dp, H1, D));
    MI_TRY(mlp_split(c, prm.W2, H1, c.W2h, pH, c.Hp, H2, H1));
    pad_f32_kernel<<<blocks_for(c.h2_pad, 256), 256, 0, stream>>>(prm.b2, c.b2p, H2, c.h2_pad);
    MI_LAUNCH_CHECK("pad_f32_kernel");
    pad_f32_kernel<<<blocks_for(c.h2_pad, 256), 256, 0, stream>>>(prm.W3, c.w3p, H2, c.h2_pad);
    MI_LAUNCH_CHECK("pad_f32_kernel");
    // the gaps between the pieces / beyond a ragged K are never written by the generators
    if (sp >= 2 || (H1 % bk()) != 0) MI_CUDA(cudaMemsetAsync(c.Hpan, 0, static_cast<size_t>(Pmax) * pH * sizeof(bf), stream));
    if (c.DZ2 && (sp >= 2 || (H2 % bk()) != 0)) MI_CUDA(cudaMemsetAsync(c.DZ2, 0, static_cast<size_t>(Pmax) * pZ * sizeof(bf), stream));
  }
  // ---- layer 1: A = X W1x^T + b1, C = Y W1y^T  (fp32 out)
  for (int side = 0; side < 2; ++side) {
    GemmArgs g;
    const long long rows = side == 0 ? Bq : Bk;
    g.a = MapSpec{side == 0 ? c.X16 : c.Y16, rows, c.eX, pX};
    g.b = MapSpec{side == 0 ? c.W1x : c.W1y, H1, c.eX, pX};
    g.M = rows; g.N = H1; kk_segments(g, sp, D);
    g.out_f32 = side == 0 ? c.A32 : c.C32; g.ld_out = H1;
    g.bias = side == 0 ? prm.b1 : nullptr;
    MI_TRY(run_gemm(g, ws, stream));
    ws.release(mk);
  }
  return MI_OK;
}

// ---- layer 1 backward of ONE side over R rows (image side: dZ = dA, In = X, W1x; text side: dZ = dC, In = Y, W1y):
//      dIn = dZ W1side, dW1[:, side] = dZ^T In (dW1_side points at the side's first column of the [H1, 2D] gradient),
//      db1 = column sums of dZ (optional).  dZ comes as fp32 and as its bf16 operand; In16 / W16 are the bf16 operands.
int mlp_layer1_bwd(const MlpCtx& c, long long R, const float* dZ32, __nv_bfloat16* dZ16, __nv_bfloat16* In16, __nv_bfloat16* W16,
                   float* dIn, float* dW1_side, float* db1, Bump& ws) {
  const long long D = c.D, H1 = c.H1, pX = c.pX, pH = c.pH;
  const int sp = c.sp;
  const bool dry = ws.dry;
  const size_t mk = ws.mark();
  if (db1 && !dry) { colsum_kernel<<<blocks_for(H1, 32), 256, 0, c.stream>>>(dZ32, R, H1, db1); MI_LAUNCH_CHECK("colsum_kernel"); }
  if (dIn || dry) {   // dIn = dZ W1side : W1side [H1, D] read in place as the MN-major B operand
    GemmArgs g;
    g.a = MapSpec{dZ16, R, c.eH, pH};
    g.b_mn = true; g.b = MapSpec{W16, H1, c.eX, pX};
    g.M = R; g.N = D;
    piece_segments(g, sp, H1, false, 0, true, c.Dp);
    g.out_f32 = dIn; g.ld_out = D;
    if (dry) { g.out_f32 = reinterpret_cast<float*>(16); }
    MI_TRY(run_gemm(g, ws, c.stream));
    ws.release(mk);
  }
  if (dW1_side || dry) {   // dW1[:, side] = dZ^T In : contraction over the rows, both operands MN-major
    GemmArgs g;
    g.a_mn = true; g.a = MapSpec{dZ16, R, c.eH, pH};
    g.b_mn = true; g.b = MapSpec{In16, R, c.eX, pX};
    g.M = H1; g.N = D;
    piece_segments(g, sp, R, true, c.Hp, true, c.Dp);
    const long long tiles = cdiv(H1, rows_per_mblk()) * cdiv(D, mi::TILE_N);
    g.ksplit = choose_ksplit(tiles, g.k_blocks, mlp_chain_min_ks(sp, g.k_blocks));
    g.out_f32 = dW1_side; g.ld_out = 2 * D;
    if (dry) { g.out_f32 = reinterpret_cast<float*>(16); }
    MI_TRY(run_gemm(g, ws, c.stream));
    ws.release(mk);
  }
  return MI_OK;
}

// ---- the single-GPU step: the block form with Bq = Bk = Bg = B, q_off = 0, one id vector
int mlp_impl(const float* X, const float* Y, const MlpParams& prm, const int* sid, const MlpDims& d, int estimator, int precision,
             double* loss_out, float* S_out, const MlpGrads& gr, Bump& ws, cudaStream_t stream) {
  if (!mlp_dims_ok(d, estimator, precision)) return MI_ERR_BAD_ARG;
  const long long B = d.B, D = d.D, H1 = d.H1, H2 = d.H2;
  const bool grads = gr.dX || gr.dY || gr.dW1 || gr.db1 || gr.dW2 || gr.db2 || gr.dW3 || gr.db3;
  const bool plan = grads || ws.dry;
  const bool dv_like = estimator == MI_EST_DV || estimator == MI_EST_INFONCE_REF;
  // the workspace is planned for both sequences (the size query does not know the estimator's path)
  const bool single = dv_like && plan && (g_mlp_mode.load(std::memory_order_relaxed) & 1) != 0;
  MlpCtx c;
  MlpSpBuf sb{};
  MI_TRY(mlp_setup(c, sb, X, Y, prm, MlpBlock{B, B, 0, B, sid, sid}, d, estimator, precision, plan, S_out, gr.dW2, loss_out,
                   sid && loss_out, ws, ws, stream));
  const bool dry = ws.dry;
  if (single || dry) {
    if (!dry) MI_TRY(mlp_reference_logit(c, sb.As, sb.Cs, sb.Ssmp, sb.ref));
    MI_TRY(mlp_sp_panels(c, sb, S_out, ws));
    if (!dry) {
      // the shared fp64 finalisation (its guard checks |ref - LSE|)
      loss_finalize_kernel<<<1, 32, 0, stream>>>(c.scal, nullptr, B, estimator, loss_out, c.lse_f, nullptr, nullptr);
      MI_LAUNCH_CHECK("loss_finalize_kernel");
    }
    MI_TRY(mlp_sp_finish(c, sb, nullptr, dry ? nullptr : loss_out + 7, ws));
    if (!dry) {
      guard_to_flag_kernel<<<1, 1, 0, stream>>>(loss_out, sb.flag, sb.guard_a);
      MI_LAUNCH_CHECK("guard_to_flag_kernel");
    }
    {   // the two-pass sequence repeats the step if (and only if) the guard tripped
      PredGuard pg(dry ? nullptr : sb.flag);
      MI_TRY(mlp_two_pass(c, plan, ws));
    }
    if (!dry) {
      guard_report_kernel<<<1, 1, 0, stream>>>(sb.flag, sb.guard_a, loss_out);
      MI_LAUNCH_CHECK("guard_report_kernel");
    }
  } else {
    MI_TRY(mlp_two_pass(c, plan, ws));
  }
  if (!plan) return MI_OK;
  if (!dry) {
    if (gr.dW3) { copy_f32_kernel<<<blocks_for(H2, 256), 256, 0, stream>>>(c.acc_w3, gr.dW3, H2); MI_LAUNCH_CHECK("copy_f32_kernel"); }
    if (gr.db2) { copy_f32_kernel<<<blocks_for(H2, 256), 256, 0, stream>>>(c.acc_b2, gr.db2, H2); MI_LAUNCH_CHECK("copy_f32_kernel"); }
    if (gr.db3) { copy_f32_kernel<<<1, 32, 0, stream>>>(c.db3v, gr.db3, 1); MI_LAUNCH_CHECK("copy_f32_kernel"); }
    MI_TRY(mlp_split(c, c.dA32, H1, c.dA16, c.pH, c.Hp, B, H1));
    MI_TRY(mlp_split(c, c.dC32, H1, c.dC16, c.pH, c.Hp, B, H1));
  }
  MI_TRY(mlp_layer1_bwd(c, B, c.dA32, c.dA16, c.X16, c.W1x, gr.dX, gr.dW1, gr.db1, ws));
  MI_TRY(mlp_layer1_bwd(c, B, c.dC32, c.dC16, c.Y16, c.W1y, gr.dY, gr.dW1 ? gr.dW1 + D : nullptr, nullptr, ws));
  return MI_OK;
}

// ---- the stages of the batch-sharded step (DESIGN 8.4): one row block of Bq image rows against all Bk = Bg text rows.
//      The caller's collectives go between the stages; everything that must survive from the forward to the backward
//      lives in the caller-owned `state` (the scratch workspace is reused by whatever runs in between).
enum MlpStage { kMlpStageRef = 0, kMlpStageFwd = 1, kMlpStageBwd = 2 };
struct MlpBlockIO {
  float* ref_out;           // stage ref: [1] maximum logit of the sample of the block's own pairs
  const float* ref;         // stage fwd (single pass): [1] the reference of every block (maximum over the blocks)
  int two_pass;
  double* scal_out;         // stage fwd: [8] the block's scalar row (mi_score_stats layout, slot 7 = its sum of g~)
  float* col_lse_out;       // stage fwd, symmetric InfoNCE: [Bk] log-sum-exp of every column over the block's rows
  const double* loss;       // stage bwd: [8] loss_out of the batch (mi_mlp_block_merge)
  const double* merged;     // stage bwd: [8] merged scalar row (slot 7 = the batch's sum of g~)
  const float* col_lse;     // stage bwd, symmetric InfoNCE: [Bk] log-sum-exp of every column over the batch
  float* dC_part;           // stage bwd: [Bk, H1] the block's contribution to dL/dC
  MlpGrads gr;              // stage bwd: dX (the block's rows), dW1 (image half), db1, dW2, db2, dW3, db3 of the block
};
int mlp_block_impl(int stage, const float* X, const float* Y, const MlpParams& prm, const MlpBlock& blk, const MlpDims& d,
                   int estimator, int precision, const MlpBlockIO& io, Bump& ws, Bump& keep, cudaStream_t stream) {
  if (!mlp_dims_ok(d, estimator, precision)) return MI_ERR_BAD_ARG;
  const long long H1 = d.H1, H2 = d.H2;
  const bool sym = estimator == MI_EST_INFONCE_SYM;       // the two-pass sequence only: columns need every row first
  bool args_ok = true;
  if (stage == kMlpStageRef) args_ok = io.ref_out != nullptr;
  else if (stage == kMlpStageFwd)
    args_ok = blk.sid_q && blk.sid_k && io.scal_out && (io.two_pass || io.ref) && (!sym || (io.two_pass && io.col_lse_out));
  else if (stage == kMlpStageBwd)
    args_ok = blk.sid_q && blk.sid_k && io.loss && io.dC_part && (io.two_pass || io.merged) && (!sym || (io.two_pass && io.col_lse));
  else return MI_ERR_BAD_ARG;
  MlpCtx c;
  MlpSpBuf sb{};
  MI_TRY(mlp_setup(c, sb, X, Y, prm, blk, d, estimator, precision, true, nullptr, nullptr, const_cast<double*>(io.loss), args_ok,
                   ws, keep, stream));
  const bool dry = ws.dry;
  if (stage == kMlpStageRef) {
    if (!dry) MI_TRY(mlp_reference_logit(c, sb.As, sb.Cs, sb.Ssmp, io.ref_out));
    return MI_OK;
  }
  if (stage == kMlpStageFwd) {
    if (!dry) c.scal = io.scal_out;
    if (io.two_pass) {
      MI_TRY(mlp_tp_fwd(c, dry));
      if (!dry && sym) MI_TRY(mlp_col_stats(c, io.col_lse_out, false));
      return MI_OK;
    }
    sb.ref = const_cast<float*>(io.ref);
    MI_TRY(mlp_sp_panels(c, sb, nullptr, ws));
    if (!dry) {
      sum_f64_kernel<<<1, 1024, 0, stream>>>(sb.rowsum, c.Bq, c.scal + 7);
      MI_LAUNCH_CHECK("sum_f64_kernel");
    }
    return MI_OK;
  }
  if (io.two_pass) {
    if (!dry) {
      c.col_lse = const_cast<float*>(io.col_lse);
      lse_from_loss_kernel<<<1, 1, 0, stream>>>(io.loss, c.lse_f);
      MI_LAUNCH_CHECK("lse_from_loss_kernel");
    }
    MI_TRY(mlp_tp_bwd(c, false, ws));
  } else {
    MI_TRY(mlp_sp_finish(c, sb, io.merged ? io.merged + 7 : nullptr, nullptr, ws));
  }
  const MlpGrads& gr = io.gr;
  if (!dry) {
    if (gr.dW3) { copy_f32_kernel<<<blocks_for(H2, 256), 256, 0, stream>>>(c.acc_w3, gr.dW3, H2); MI_LAUNCH_CHECK("copy_f32_kernel"); }
    if (gr.db2) { copy_f32_kernel<<<blocks_for(H2, 256), 256, 0, stream>>>(c.acc_b2, gr.db2, H2); MI_LAUNCH_CHECK("copy_f32_kernel"); }
    if (gr.db3) { copy_f32_kernel<<<1, 32, 0, stream>>>(c.db3v, gr.db3, 1); MI_LAUNCH_CHECK("copy_f32_kernel"); }
    if (gr.dW2) { copy_f32_kernel<<<blocks_for(H2 * H1, 256), 256, 0, stream>>>(c.dW2, gr.dW2, H2 * H1); MI_LAUNCH_CHECK("copy_f32_kernel"); }
    MI_CUDA(cudaMemcpyAsync(io.dC_part, c.dC32, static_cast<size_t>(c.Bk) * H1 * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    MI_TRY(mlp_split(c, c.dA32, H1, c.dA16, c.pH, c.Hp, c.Bq, H1));
  }
  return mlp_layer1_bwd(c, c.Bq, c.dA32, c.dA16, c.X16, c.W1x, gr.dX, gr.dW1, gr.db1, ws);
}
// layer-1 backward of one side from fp32 inputs (the text side of the sharded step, after the exchange of dC)
int mlp_input_grad_impl(const float* dZ, const float* In, const float* W1, int side, long long R, long long D, long long H1, int precision,
                        float* dIn, float* dW1, float* db1, Bump& ws, cudaStream_t stream) {
  if (R <= 0 || D <= 0 || H1 <= 0 || (D % 8) != 0 || (H1 % 8) != 0 || (side != 0 && side != 1)) return MI_ERR_BAD_ARG;
  if (!mlp_precision_ok(precision, D, H1)) return MI_ERR_BAD_ARG;
  typedef __nv_bfloat16 bf;
  MlpCtx c;
  c.stream = stream;
  mlp_ctx_dims(c, D, H1, 8, precision);
  bf* dZ16 = ws.take<bf>(R * c.pH);
  bf* In16 = ws.take<bf>(R * c.pX);
  bf* W16 = ws.take<bf>(H1 * c.pX);
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (!ws.dry) {
    if (!dZ || !In || !W1) return MI_ERR_BAD_ARG;
    MI_TRY(mlp_split(c, dZ, H1, dZ16, c.pH, c.Hp, R, H1));
    MI_TRY(mlp_split(c, In, D, In16, c.pX, c.Dp, R, D));
    MI_TRY(mlp_split(c, W1 + side * D, 2 * D, W16, c.pX, c.Dp, H1, D));
  }
  return mlp_layer1_bwd(c, R, dZ, dZ16, In16, W16, dIn, dW1 ? dW1 + side * D : nullptr, db1, ws);
}
