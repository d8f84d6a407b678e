// libmi_b200.so — host launchers, auxiliary kernels and the extern "C" ABI declared in
// include/mi_b200.h.  The tensor-core work is in engine.cuh (tcgen05 / TMEM / TMA, sm_100a only).
// There is no CPU path: every entry point fails with MI_ERR_NO_DEVICE / MI_ERR_CUDA when no
// Blackwell device is available.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <functional>
#include <mutex>
#include <vector>
#include <cstdlib>
#include <cstring>
#include <cuda_bf16.h>

#include "../../include/mi_b200.h"
#include "engine.cuh"

namespace {

using mi::Sched;

// ------------------------------------------------------------------------------------ errors
thread_local char g_cuda_err[512] = "";
std::atomic<long long> g_launches{0};
// Process-wide knobs (bring-up / A-B experiments; set before the first call, not per call):
std::atomic<int> g_cta_group{-1};          // resolved lazily: env MI_CTA_GROUP or 2
std::atomic<int> g_overlap_reserve_sms{0}; // SMs left free for a concurrent collective by the engine launches after event_after_outk
std::atomic<long long> g_ref_sample_cols{2048};   // columns sampled per row for the single pass's softmax references
// Per-call state lives in thread-locals, so two host threads driving different streams never share it:
thread_local int t_reserve_sms = 0;        // applied to the next engine launches of this thread
thread_local const int* t_run_if = nullptr;   // device predicate of the launches of this thread (see Sched::run_if)
struct PredGuard {
  const int* prev;
  explicit PredGuard(const int* p) : prev(t_run_if) { t_run_if = p; }
  ~PredGuard() { t_run_if = prev; }
};
#define MI_PRED(p) do { if ((p) != nullptr && *(p) == 0) return; } while (0)

// optional per-launch CUDA-event timing of the tile-engine kernels (bench.py's roofline breakdown)
struct ProfRec { int kind; cudaEvent_t e0, e1; };
bool g_profiling = false;
std::vector<ProfRec> g_prof;
std::mutex g_prof_mu;
template <class Epi> struct EpiKind;

int cta_group() {
  int g = g_cta_group.load(std::memory_order_relaxed);
  if (g < 0) {
    const char* e = std::getenv("MI_CTA_GROUP");
    g = (e && e[0] == '1') ? 1 : 2;
    g_cta_group.store(g, std::memory_order_relaxed);
  }
  return g;
}

int set_cuda_err(cudaError_t e, const char* where) {
  std::snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", where, cudaGetErrorString(e));
  return MI_ERR_CUDA;
}
#define MI_CUDA(call)                                                   \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) return set_cuda_err(e__, #call);            \
  } while (0)
#define MI_TRY(call)                                                    \
  do {                                                                  \
    int s__ = (call);                                                   \
    if (s__ != MI_OK) return s__;                                       \
  } while (0)
#define MI_LAUNCH_CHECK(name)                                           \
  do {                                                                  \
    g_launches.fetch_add(1, std::memory_order_relaxed);                 \
    cudaError_t e__ = cudaGetLastError();                               \
    if (e__ != cudaSuccess) return set_cuda_err(e__, name);             \
  } while (0)

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) n = v;
    else { n = 148; (void)cudaGetLastError(); return 148; }   // planning on a box without a GPU
  }
  return n;
}

// ------------------------------------------------------------------------------------ workspace
struct Bump {
  uint8_t* base; size_t cap; size_t off; size_t peak; bool dry;
  Bump(void* b, size_t c, bool d) : base(static_cast<uint8_t*>(b)), cap(c), off(0), peak(0), dry(d) {}
  template <class T> T* take(size_t n) {
    off = (off + 255) & ~static_cast<size_t>(255);
    T* p = dry ? nullptr : reinterpret_cast<T*>(base + off);
    off += n * sizeof(T);
    if (off > peak) peak = off;
    return p;
  }
  // stream-ordered reuse: everything taken after mark() is dead once the stage's kernels are enqueued
  size_t mark() const { return off; }
  void release(size_t m) { off = m; }
  bool ok() const { return dry || (peak <= cap && (base != nullptr || peak == 0)); }
};

inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }
inline int gcd_i(int a, int b) { while (b) { int t = a % b; a = b; b = t; } return a; }

// ------------------------------------------------------------------------------------ TMA maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 matrix [rows, k_extent] with row pitch ld (elements); box = [box_rows x 64], 128 B swizzle,
// out-of-bounds elements read as zero (ragged rows and K tails need no special casing).
int make_tmap(CUtensorMap* m, const void* ptr, long long rows, long long k_extent, long long ld, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { std::snprintf(g_cuda_err, sizeof(g_cuda_err), "cuTensorMapEncodeTiled unavailable"); return MI_ERR_CUDA; }
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld % 8) != 0 || rows <= 0 || k_extent <= 0) return MI_ERR_BAD_ARG;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(k_extent), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(mi::ATOM_K), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    std::snprintf(g_cuda_err, sizeof(g_cuda_err), "cuTensorMapEncodeTiled failed with %d", static_cast<int>(r));
    return MI_ERR_CUDA;
  }
  return MI_OK;
}

// bf16 matrix [rows, cols] with row pitch ld (elements) as a STORE target: box 32 x 32, 64 B swizzle (the staging layout
// of EpiPStore); rows / columns beyond the matrix are clipped by the TMA engine.
int make_tmap_store32(CUtensorMap* m, const void* ptr, long long rows, long long cols, long long ld) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { std::snprintf(g_cuda_err, sizeof(g_cuda_err), "cuTensorMapEncodeTiled unavailable"); return MI_ERR_CUDA; }
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld % 8) != 0 || rows <= 0 || cols <= 0) return MI_ERR_BAD_ARG;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    std::snprintf(g_cuda_err, sizeof(g_cuda_err), "cuTensorMapEncodeTiled (store) failed with %d", static_cast<int>(r));
    return MI_ERR_CUDA;
  }
  return MI_OK;
}

// ------------------------------------------------------------------------------------ engine launch
struct MapSpec {          // a 2-D bf16 tensor map: `rows` x `k_extent` elements, row pitch ld
  const void* ptr; long long rows, k_extent, ld;
};

template <int kCG, class Epi, bool kAMN, bool kBMN>
int launch_engine_cg(const MapSpec& a, const MapSpec& b, const Sched& sc, const typename Epi::Params& ep, cudaStream_t stream) {
  using C = mi::Cfg<kCG>;
  CUtensorMap ta, tb;
  // MN-major A: the map's contiguous dimension is M, its rows are K; fetched as 64 x 64 boxes
  if (kAMN) MI_TRY(make_tmap(&ta, a.ptr, a.rows, a.k_extent, a.ld, 64));
  else MI_TRY(make_tmap(&ta, a.ptr, a.rows, a.k_extent, a.ld, mi::BLOCK_M));
  if (kBMN) MI_TRY(make_tmap(&tb, b.ptr, b.rows, b.k_extent, b.ld, 64));
  else MI_TRY(make_tmap(&tb, b.ptr, b.rows, b.k_extent, b.ld, C::kBRows));
  auto kern = mi::tile_engine_kernel<kCG, Epi, kAMN, kBMN>;
  constexpr int smem = C::template smem_bytes<Epi>();
  static std::atomic<unsigned long long> attr_devs{0};      // bit d: attribute set on device d (it is per device)
  int dev = 0;
  MI_CUDA(cudaGetDevice(&dev));
  const unsigned long long bit = 1ull << (dev & 63);
  if ((attr_devs.load(std::memory_order_acquire) & bit) == 0) {
    MI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_devs.fetch_or(bit, std::memory_order_release);
  }
  const int units = mi::num_units(sc);
  int pairs = (num_sms() - t_reserve_sms) / kCG;
  if (pairs > units) pairs = units;
  if (pairs < 1) pairs = 1;
  cudaLaunchConfig_t cfg;
  std::memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(static_cast<unsigned>(pairs * kCG), 1, 1);
  cfg.blockDim = dim3(mi::kNumThreads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  Sched scp = sc;
  scp.run_if = t_run_if;
  ProfRec rec; rec.kind = EpiKind<Epi>::value; rec.e0 = nullptr; rec.e1 = nullptr;
  if (g_profiling) {
    MI_CUDA(cudaEventCreate(&rec.e0)); MI_CUDA(cudaEventCreate(&rec.e1));
    MI_CUDA(cudaEventRecord(rec.e0, stream));
  }
  MI_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, scp, ep));
  MI_LAUNCH_CHECK("tile_engine_kernel");
  if (g_profiling) {
    MI_CUDA(cudaEventRecord(rec.e1, stream));
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.push_back(rec);
  }
  return MI_OK;
}

template <> struct EpiKind<mi::EpiStats> { static constexpr int value = 0; };
template <> struct EpiKind<mi::EpiStatsRC> { static constexpr int value = 0; };
template <> struct EpiKind<mi::EpiPStore> { static constexpr int value = 1; };
template <> struct EpiKind<mi::EpiJS<true>> { static constexpr int value = 1; };    // Jensen-Shannon dS panel
template <> struct EpiKind<mi::EpiJS<false>> { static constexpr int value = 0; };   // its statistics-only form
template <> struct EpiKind<mi::EpiStore> { static constexpr int value = 2; };
template <> struct EpiKind<mi::EpiMlpFwd> { static constexpr int value = 5; };   // MLP critic: two-pass epilogues
template <> struct EpiKind<mi::EpiMlpDz> { static constexpr int value = 5; };
template <> struct EpiKind<mi::EpiMlpSp> { static constexpr int value = 3; };    // single pass (forward + dZ2)
template <> struct EpiKind<mi::EpiMlpDa> { static constexpr int value = 4; };    // dZ1 with fused reductions
constexpr int kProfKinds = 6;
template <> struct EpiKind<mi::EpiDist> { static constexpr int value = 0; };

template <class Epi, bool kAMN = false, bool kBMN = false>
int launch_engine(const MapSpec& a, const MapSpec& b, const Sched& sc, const typename Epi::Params& ep, cudaStream_t stream) {
  if (cta_group() == 1) return launch_engine_cg<1, Epi, kAMN, kBMN>(a, b, sc, ep, stream);
  return launch_engine_cg<2, Epi, kAMN, kBMN>(a, b, sc, ep, stream);
}

inline int rows_per_mblk() { return mi::BLOCK_M * cta_group(); }
inline int num_pairs() { return num_sms() / cta_group(); }
inline long long round_up(long long a, long long b) { return cdiv(a, b) * b; }
inline int bk() { return mi::block_k(cta_group()); }      // K block per pipeline stage
constexpr long long kSplitAlign = 128;                    // lo half of a hi/lo pair starts at round_up(width, 128)

// N-range splits per M block for the streaming (stats / dS-panel) passes: make the unit count a
// multiple of the number of CTA pairs, then refine while units stay long enough to amortise.
int choose_split(int n_mblk, int n_ntile, int U) {
  int ns = U / gcd_i(n_mblk, U);
  if (ns > n_ntile) {
    ns = static_cast<int>(cdiv(4LL * U, n_mblk));
    if (ns > n_ntile) ns = n_ntile;
    if (ns < 1) ns = 1;
    return ns;
  }
  while (ns * 2 <= n_ntile / 8 && n_mblk * ns < 8 * U) ns *= 2;
  return ns;
}

// K splits of a GEMM with few output tiles: the split that minimises (rounds of the CTA pairs) x (K blocks per unit),
// with a small charge per split for the partial-sum pass; at least min_ks (strict mode bounds the accumulation chains).
int choose_ksplit(long long tiles, int k_blocks, long long min_ks = 1) {
  const long long U = num_pairs();
  long long hi = k_blocks / 4;
  if (hi < 1) hi = 1;
  long long lo = min_ks < 1 ? 1 : min_ks;
  if (lo > hi) lo = hi;
  long long best = lo;
  double best_cost = 1e300;
  for (long long ks = lo; ks <= hi && ks <= 4 * U; ++ks) {
    const double cost = static_cast<double>(cdiv(tiles * ks, U)) * static_cast<double>(cdiv(k_blocks, ks)) + 0.25 * static_cast<double>(ks);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = ks; }
  }
  return static_cast<int>(best);
}

void single_segment(Sched& sc) {
  sc.nt_base = 0;
  sc.seg_len = sc.k_blocks;
  sc.grp = 1; sc.chunk_len = 1; sc.n_chunks = 1; sc.n_il = 1;
  for (int i = 0; i < 4; ++i) { sc.a_seg[i] = 0; sc.b_seg[i] = 0; sc.a_moff[i] = 0; sc.b_noff[i] = 0; }
}

// ------------------------------------------------------------------------------------ aux kernels
// Every kernel of the single-pass / statistics paths takes a trailing `run_if` launch predicate (see Sched::run_if).
__global__ void pad_int_kernel(const int* __restrict__ src, int* __restrict__ dst, long long n, long long n_pad, int fill,
                               const int* __restrict__ run_if) {
  MI_PRED(run_if);
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n_pad) dst[i] = (i < n) ? src[i] : fill;
}
// dst[s] = src[s * stride], s < n: the study ids of a strided column sample
__global__ void gather_int_kernel(const int* __restrict__ src, long long stride, int* __restrict__ dst, long long n,
                                  const int* __restrict__ run_if) {
  MI_PRED(run_if);
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i * stride];
}

// ---- exclusion lists: for every row, the columns that share its study id (hash grouping, O(B)).
// A slot holds (1 << 32) | (uint32) id; 0 = empty, so EVERY int32 id (INT_MIN included) is a legal key.
__device__ __forceinline__ uint32_t hash_sid(int key, uint32_t mask) {
  return (static_cast<uint32_t>(key) * 2654435761u >> 7) & mask;
}
__device__ __forceinline__ unsigned long long slot_key(int key) { return (1ull << 32) | static_cast<uint32_t>(key); }
__global__ void excl_init_kernel(unsigned long long* __restrict__ keys, int* __restrict__ counts, int* __restrict__ members,
                                 long long slots, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < slots) {
    keys[i] = 0ull; counts[i] = 0;
    reinterpret_cast<int4*>(members)[i] = make_int4(-1, -1, -1, -1);
  }
}
__global__ void excl_insert_kernel(const int* __restrict__ sid_k, long long Bk, unsigned long long* keys, int* counts, int* members,
                                   uint32_t mask, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= Bk) return;
  const int key = sid_k[k];
  const unsigned long long sk = slot_key(key);
  uint32_t h = hash_sid(key, mask);
  while (true) {
    const unsigned long long prev = atomicCAS(&keys[h], 0ull, sk);
    if (prev == 0ull || prev == sk) break;
    h = (h + 1) & mask;
  }
  const int t = atomicAdd(&counts[h], 1);
  if (t < mi::kMaxExcl) members[h * mi::kMaxExcl + t] = static_cast<int>(k);
}
__global__ void excl_lookup_kernel(const int* __restrict__ sid_q, long long Bq, const unsigned long long* __restrict__ keys,
                                   const int* __restrict__ counts, const int* __restrict__ members, uint32_t mask,
                                   int4* __restrict__ excl, int* __restrict__ n_same, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (q >= Bq) return;
  const int key = sid_q[q];
  const unsigned long long sk = slot_key(key);
  uint32_t h = hash_sid(key, mask);
  int4 e = make_int4(-1, -1, -1, -1);
  int n = 0;
  while (true) {
    const unsigned long long kk = keys[h];
    if (kk == sk) { n = counts[h]; if (n <= mi::kMaxExcl) e = reinterpret_cast<const int4*>(members)[h]; break; }
    if (kk == 0ull) break;
    h = (h + 1) & mask;
  }
  excl[q] = e; n_same[q] = n;
}

// refk2[c] = (refk[c] - ln wk) * log2(e), zero padded
__global__ void make_refk2_kernel(const float* __restrict__ refk, float ln_wk, float* __restrict__ dst, long long n, long long n_pad) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n_pad) dst[i] = (i < n) ? (refk[i] - ln_wk) * mi::kLog2e : 0.f;
}

// 4 elements / thread.  The float4 load and uint2 store need 16- / 8-byte aligned pointers; a contiguous view at an element
// offset (x[1:], a slice of a flat parameter buffer) is not, and takes the scalar path for all of its elements.
__global__ void cast_f32_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, long long n) {
  long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 4;
  const bool vec = ((reinterpret_cast<unsigned long long>(in) & 15ull) | (reinterpret_cast<unsigned long long>(out) & 7ull)) == 0;
  if (vec && i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(in + i);
    uint2 o; o.x = ptx::pack_bf16(v.x, v.y); o.y = ptx::pack_bf16(v.z, v.w);
    *reinterpret_cast<uint2*>(out + i) = o;
  } else {
    const long long end = i + 4 < n ? i + 4 : n;
    for (; i < end; ++i) out[i] = __float2bfloat16(in[i]);
  }
}

// out[c, r] = in[r, c]; 64x64 tiles through shared memory, coalesced on both sides
__global__ void transpose_bf16_kernel(const __nv_bfloat16* __restrict__ in, long long ld_in,
                                      __nv_bfloat16* __restrict__ out, long long ld_out, long long R, long long C) {
  __shared__ __nv_bfloat16 tile[64][66];
  const long long r0 = blockIdx.y * 64LL, c0 = blockIdx.x * 64LL;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;   // 256 threads: 64 x 4
  for (int i = ty; i < 64; i += 4) {
    const long long r = r0 + i, c = c0 + tx;
    tile[i][tx] = (r < R && c < C) ? in[r * ld_in + c] : __float2bfloat16(0.f);
  }
  __syncthreads();
  for (int i = ty; i < 64; i += 4) {
    const long long c = c0 + i, r = r0 + tx;
    if (c < C && r < R) out[c * ld_out + r] = tile[tx][i];
  }
}

// diag[q] = scale * <Q[q,:], K[q_offset+q,:]> (the positive pair), one warp per row; hi/lo pairs summed
__global__ void diag_kernel(const __nv_bfloat16* __restrict__ Q, long long ldq, int q_split,
                            const __nv_bfloat16* __restrict__ K, long long ldk, int k_split,
                            long long q_offset, long long Bq, long long D, long long Dp, float scale, float* __restrict__ diag,
                            const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= Bq) return;
  const __nv_bfloat16* q = Q + row * ldq;
  const __nv_bfloat16* k = K + (q_offset + row) * ldk;
  float acc = 0.f;
  for (long long d = lane * 2; d < D; d += 64) {
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(q + d));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(k + d));
    float ax = a.x, ay = a.y, bx = b.x, by = b.y;
    if (q_split == 2) { const float2 l = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(q + Dp + d)); ax += l.x; ay += l.y; }
    if (k_split == 2) { const float2 l = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(k + Dp + d)); bx += l.x; by += l.y; }
    acc = fmaf(ax, bx, acc); acc = fmaf(ay, by, acc);
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) diag[row] = acc * scale;
}

// ---- single-pass path -------------------------------------------------------------------------------
// row L2 norms of a bf16 matrix (hi/lo pairs summed), one warp per row (mi_row_norm_max: a stage op kept for callers)
__global__ void row_norm_kernel(const __nv_bfloat16* __restrict__ A, long long ld, int split, long long Dp,
                                long long rows, long long D, float* __restrict__ norm) {
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const __nv_bfloat16* a = A + row * ld;
  float acc = 0.f;
  for (long long d = lane * 2; d < D; d += 64) {
    float2 v = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(a + d));
    if (split == 2) { const float2 l = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(a + Dp + d)); v.x += l.x; v.y += l.y; }
    acc = fmaf(v.x, v.x, acc); acc = fmaf(v.y, v.y, acc);
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) norm[row] = sqrtf(acc);
}
// one block: out[0] = max_i in[i] - offset (NaN entries are ignored by fmaxf; all-NaN / empty gives -inf)
__global__ void max_reduce_kernel(const float* __restrict__ in, long long n, float* __restrict__ out, float offset,
                                  const int* __restrict__ run_if) {
  MI_PRED(run_if);
  __shared__ float sh[32];
  float m = mi::neg_inf();
  for (long long i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, in[i]);
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) { float g = mi::neg_inf(); for (int i = 0; i < (int)(blockDim.x >> 5); ++i) g = fmaxf(g, sh[i]); out[0] = g - offset; }
}

// The single pass writes P~ = incl e^{S - ref_q} BEFORE the exact row statistics are known, so it needs a per-row reference
// close enough to the row's log-sum-exp that neither P~ nor its row sum leaves the fp32 / bf16 range (about +-87 in the
// exponent).  ref_q is the log-sum-exp over a strided SAMPLE of the row's columns (computed by the statistics epilogue on
// K[c0 + s * stride]); with stride 1 the sample is every column and ref_q is exact.  Merge of the sample's (max, sum) partials:
//   include_diag = 0:  ref = LSE over the sampled negatives            (the positive pair if the sample has no negative)
//   include_diag = 1:  ref = logaddexp(that, positive-pair score)
// `margin` (sampled references only) lifts the reference above the sample's log-sum-exp: the row's true maximum may sit
// above everything the sample saw, and the window is one-sided — P~ may fall to 1e-38 but must stay below ~1e30.
__global__ void ref_merge_kernel(const float4* __restrict__ part, int n_part, int rows_padded, int q_rows,
                                 const float* __restrict__ diag_in, int include_diag, float margin, float* __restrict__ ref_out,
                                 const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= q_rows) return;
  float m = mi::neg_inf();
  for (int p = 0; p < n_part; ++p) m = fmaxf(m, part[(size_t)p * rows_padded + row].x);
  float s = 0.f;
  for (int p = 0; p < n_part; ++p) {
    const float4 v = part[(size_t)p * rows_padded + row];
    if (v.y > 0.f) s += v.y * exp2f(v.x - m);
  }
  const float diag = diag_in[row];
  const float lse = (s > 0.f) ? (m + log2f(s)) * mi::kLn2 : mi::neg_inf();
  float ref;
  if (include_diag) {
    const float hi = fmaxf(lse, diag), lo = fminf(lse, diag);
    ref = (lo > mi::neg_inf()) ? hi + log1pf(expf(lo - hi)) : hi;
  } else {
    ref = (lse > mi::neg_inf()) ? lse : diag;
  }
  ref_out[row] = ref + margin;
}

// rows of one panel: l = sum of the partial row sums of P~ = e^{S - ref};  row_out = {lse_neg, n_neg, diag, lse_all},
// wrow = weight of the row inside the G^T Q contraction.  flag counts the rows whose reference left the safe window
// (l not in [1e-30, 1e30], NaN included, or the row's weight e^{ref - lambda} would overflow): the caller must then
// repeat the step with exact references (stride 1), for which l = 1 by construction.
__global__ void sum_merge_kernel(const float* __restrict__ part, int n_part, int rows_padded, int rows,
                                 const float* __restrict__ ref, const float* __restrict__ lambda, const int* __restrict__ n_same,
                                 int k_cols, const float* __restrict__ diag_in, int include_diag, float inv_bg,
                                 float4* __restrict__ row_out, float* __restrict__ wrow,
                                 int* __restrict__ flag, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= rows) return;
  float l = 0.f;
  for (int p = 0; p < n_part; ++p) l += part[(size_t)p * rows_padded + row];
  const float cnt = static_cast<float>(k_cols - n_same[row]);
  const float diag = diag_in[row], r = ref[row];
  const float n_incl = cnt + (include_diag ? 1.f : 0.f);
  bool bad = n_incl > 0.f && !(l >= 1e-30f && l <= 1e30f);
  float lse_neg, lse_all;
  if (include_diag) {
    lse_all = r + logf(l);
    lse_neg = cnt > 0.f ? lse_all + log1pf(-fminf(expf(diag - lse_all), 1.f)) : mi::neg_inf();
    wrow[row] = inv_bg / l;                                          // (1/B) e^{ref - r_i}
  } else {
    lse_neg = (cnt > 0.f && l > 0.f) ? r + logf(l) : mi::neg_inf();
    const float hi = fmaxf(lse_neg, diag), lo = fminf(lse_neg, diag);
    lse_all = hi + log1pf(expf(lo - hi));
    const float d = r - lambda[0];
    wrow[row] = expf(d);                                             // e^{ref - lambda}; e^{lambda - LSE} is applied at the end
    bad = bad || !(d <= 80.f);                                       // lambda far below this row's reference (or NaN)
  }
  if (bad) atomicAdd(flag, 1);
  row_out[row] = make_float4(lse_neg, cnt, diag, lse_all);
}
// out[r, c] = bf16(w[r] * in[r, c]) (+ residual half at out_lo), row-major: the MN-major B operand of P~^T (w Q).  8 elements / thread
__global__ void scale_rows_kernel(const __nv_bfloat16* __restrict__ in, long long ld_in, int in_split, long long Dp,
                                  const float* __restrict__ w, __nv_bfloat16* __restrict__ out, __nv_bfloat16* __restrict__ out_lo,
                                  long long ld_out, long long R, long long C, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  for (long long idx = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 8; idx < R * C;
       idx += (long long)gridDim.x * blockDim.x * 8) {
  const long long r = idx / C, c = idx - r * C;         // C % 8 == 0: the 8 elements share a row
  const uint4 hv = *reinterpret_cast<const uint4*>(in + r * ld_in + c);
  const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
  float v[8];
#pragma unroll
  for (int j = 0; j < 4; ++j) { v[2 * j] = __uint_as_float(hw[j] << 16); v[2 * j + 1] = __uint_as_float(hw[j] & 0xffff0000u); }
  if (in_split == 2) {
    const uint4 lv = *reinterpret_cast<const uint4*>(in + r * ld_in + Dp + c);
    const uint32_t lw[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) { v[2 * j] += __uint_as_float(lw[j] << 16); v[2 * j + 1] += __uint_as_float(lw[j] & 0xffff0000u); }
  }
  const float wr = w[r];
  uint32_t h[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { v[2 * j] *= wr; v[2 * j + 1] *= wr; h[j] = ptx::pack_bf16(v[2 * j], v[2 * j + 1]); }
  *reinterpret_cast<uint4*>(out + r * ld_out + c) = make_uint4(h[0], h[1], h[2], h[3]);
  if (out_lo) {
    uint32_t l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
      l[j] = ptx::pack_bf16(v[2 * j] - __uint_as_float(h[j] << 16), v[2 * j + 1] - __uint_as_float(h[j] & 0xffff0000u));
    *reinterpret_cast<uint4*>(out_lo + r * ld_out + c) = make_uint4(l[0], l[1], l[2], l[3]);
  }
  }
}
// Oq[i,:] = alpha (c_i Oraw[i,:] - gamma Kdiag[i,:]),  c_i = e^{ref_i - LSE} (DV) or wrow_i (row InfoNCE).  8 elements / thread
__global__ void finalize_q_kernel(const float* __restrict__ raw, long long D, long long rows, const float* __restrict__ ref,
                                  const float* __restrict__ wrow, const float* __restrict__ lse, int dv_like,
                                  float alpha, float gamma, const __nv_bfloat16* __restrict__ kdiag, long long ldk, int k_split, long long Dp,
                                  float* __restrict__ out_f32, __nv_bfloat16* __restrict__ out_bf16, __nv_bfloat16* __restrict__ out_lo, long long ld16,
                                  const int* __restrict__ run_if) {
  MI_PRED(run_if);
  for (long long idx = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 8; idx < rows * D;
       idx += (long long)gridDim.x * blockDim.x * 8) {
  const long long i = idx / D, d = idx - i * D;          // D % 8 == 0
  const float c = dv_like ? expf(ref[i] - lse[0]) : (wrow != nullptr ? wrow[i] : 1.f);
  const uint4 kv = *reinterpret_cast<const uint4*>(kdiag + i * ldk + d);
  const uint32_t kw[4] = {kv.x, kv.y, kv.z, kv.w};
  float kd[8];
#pragma unroll
  for (int j = 0; j < 4; ++j) { kd[2 * j] = __uint_as_float(kw[j] << 16); kd[2 * j + 1] = __uint_as_float(kw[j] & 0xffff0000u); }
  if (k_split == 2) {
    const uint4 lv = *reinterpret_cast<const uint4*>(kdiag + i * ldk + Dp + d);
    const uint32_t lw[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) { kd[2 * j] += __uint_as_float(lw[j] << 16); kd[2 * j + 1] += __uint_as_float(lw[j] & 0xffff0000u); }
  }
  const float4 r0 = *reinterpret_cast<const float4*>(raw + idx), r1 = *reinterpret_cast<const float4*>(raw + idx + 4);
  const float rv[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
  float o[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) o[j] = alpha * (c * rv[j] - gamma * kd[j]);
  if (out_f32) {
    *reinterpret_cast<float4*>(out_f32 + idx) = make_float4(o[0], o[1], o[2], o[3]);
    *reinterpret_cast<float4*>(out_f32 + idx + 4) = make_float4(o[4], o[5], o[6], o[7]);
  }
  if (out_bf16) {
    uint32_t h[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) h[j] = ptx::pack_bf16(o[2 * j], o[2 * j + 1]);
    *reinterpret_cast<uint4*>(out_bf16 + i * ld16 + d) = make_uint4(h[0], h[1], h[2], h[3]);
    if (out_lo) {
      uint32_t l[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        l[j] = ptx::pack_bf16(o[2 * j] - __uint_as_float(h[j] << 16), o[2 * j + 1] - __uint_as_float(h[j] & 0xffff0000u));
      *reinterpret_cast<uint4*>(out_lo + i * ld16 + d) = make_uint4(l[0], l[1], l[2], l[3]);
    }
  }
  }
}
// Ok[k,:] = alpha (kappa Ok[k,:] - gamma [0 <= k-q_offset < Bq] Q[k-q_offset,:]),  kappa = e^{lambda - LSE} (DV) or 1.  8 elements / thread
__global__ void finalize_k_kernel(float* __restrict__ ok, long long D, long long Bk, const float* __restrict__ lambda,
                                  const float* __restrict__ lse, int dv_like, float alpha, float gamma,
                                  const __nv_bfloat16* __restrict__ Q, long long ldq, int q_split, long long Dp,
                                  long long q_offset, long long Bq) {
  const float kappa = dv_like ? expf(lambda[0] - lse[0]) : 1.f;
  for (long long idx = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 8; idx < Bk * D;
       idx += (long long)gridDim.x * blockDim.x * 8) {
    const long long k = idx / D, d = idx - k * D;          // D % 8 == 0
    float qd[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const long long q = k - q_offset;
    if (q >= 0 && q < Bq) {
      const uint4 hv = *reinterpret_cast<const uint4*>(Q + q * ldq + d);
      const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) { qd[2 * j] = __uint_as_float(hw[j] << 16); qd[2 * j + 1] = __uint_as_float(hw[j] & 0xffff0000u); }
      if (q_split == 2) {
        const uint4 lv = *reinterpret_cast<const uint4*>(Q + q * ldq + Dp + d);
        const uint32_t lw[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) { qd[2 * j] += __uint_as_float(lw[j] << 16); qd[2 * j + 1] += __uint_as_float(lw[j] & 0xffff0000u); }
      }
    }
    float4 a = *reinterpret_cast<const float4*>(ok + idx), b = *reinterpret_cast<const float4*>(ok + idx + 4);
    a.x = alpha * (kappa * a.x - gamma * qd[0]); a.y = alpha * (kappa * a.y - gamma * qd[1]);
    a.z = alpha * (kappa * a.z - gamma * qd[2]); a.w = alpha * (kappa * a.w - gamma * qd[3]);
    b.x = alpha * (kappa * b.x - gamma * qd[4]); b.y = alpha * (kappa * b.y - gamma * qd[5]);
    b.z = alpha * (kappa * b.z - gamma * qd[6]); b.w = alpha * (kappa * b.w - gamma * qd[7]);
    *reinterpret_cast<float4*>(ok + idx) = a; *reinterpret_cast<float4*>(ok + idx + 4) = b;
  }
}

// merge the (split, half) partials of one row -> {lse_neg, n_neg, diag, lse_all}
__global__ void stats_merge_kernel(const float4* __restrict__ part, int n_part, int rows_padded, int q_rows,
                                   const int* __restrict__ n_same, int k_cols, const float* __restrict__ diag_in,
                                   float4* __restrict__ row_out) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= q_rows) return;
  float m = mi::neg_inf();
  for (int p = 0; p < n_part; ++p) m = fmaxf(m, part[(size_t)p * rows_padded + row].x);
  float s = 0.f;
  for (int p = 0; p < n_part; ++p) {
    const float4 v = part[(size_t)p * rows_padded + row];
    if (v.y > 0.f) s += v.y * exp2f(v.x - m);
  }
  const float diag = diag_in[row];
  const float cnt = static_cast<float>(k_cols - n_same[row]);     // negatives: columns of a different study
  const float lse_neg = (cnt > 0.f && s > 0.f) ? (m + log2f(s)) * mi::kLn2 : mi::neg_inf();
  const float hi = fmaxf(lse_neg, diag), lo = fminf(lse_neg, diag);
  const float lse_all = hi + log1pf(expf(lo - hi));
  row_out[row] = make_float4(lse_neg, cnt, diag, lse_all);
}

// columns of the square score matrix: merge the per-32-row-block partial log2-sum-exp2 values (EpiStatsRC) of column j
// -> col_out[j] = {lse_neg, n_neg, diag, lse_all} (the layout of row_out).  block = 32 columns x 8 row-block slices.
__global__ void col_merge_kernel(const float* __restrict__ colpart, int n_rb, long long pitch, int k_cols,
                                 const int* __restrict__ n_same, int q_rows, const float* __restrict__ diag_in,
                                 float4* __restrict__ col_out) {
  __shared__ float shm[8][33], shs[8][33];
  const int col = blockIdx.x * 32 + threadIdx.x;
  float m = mi::neg_inf(), s = 0.f;
  if (col < k_cols) {
    for (int rb = threadIdx.y; rb < n_rb; rb += 8) {
      const float x = colpart[(size_t)rb * pitch + col];
      if (x > mi::neg_inf()) {
        const float mn = fmaxf(m, x);
        s = s * exp2f(m - mn) + exp2f(x - mn);       // (m = -inf, s = 0 on the first hit: 0 * 0 + 1)
        m = mn;
      }
    }
  }
  shm[threadIdx.y][threadIdx.x] = m; shs[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y != 0 || col >= k_cols) return;
  float gm = mi::neg_inf();
  for (int y = 0; y < 8; ++y) gm = fmaxf(gm, shm[y][threadIdx.x]);
  float gs = 0.f;
  for (int y = 0; y < 8; ++y) if (shs[y][threadIdx.x] > 0.f) gs += shs[y][threadIdx.x] * exp2f(shm[y][threadIdx.x] - gm);
  const float diag = diag_in[col];
  const float cnt = static_cast<float>(q_rows - n_same[col]);
  const float lse_neg = (cnt > 0.f && gs > 0.f) ? (gm + log2f(gs)) * mi::kLn2 : mi::neg_inf();
  const float hi = fmaxf(lse_neg, diag), lo = fminf(lse_neg, diag);
  const float lse_all = hi + log1pf(expf(lo - hi));
  col_out[col] = make_float4(lse_neg, cnt, diag, lse_all);
}

// columns of a row BLOCK of the score matrix (a rank's rows in the batch-sharded step): the natural-log log-sum-exp of
// column j over the block's negatives (-inf if it has none); the ranks' values are merged by the caller.
__global__ void col_lse_kernel(const float* __restrict__ colpart, int n_rb, long long pitch, int k_cols, float* __restrict__ col_lse) {
  __shared__ float shm[8][33], shs[8][33];
  const int col = blockIdx.x * 32 + threadIdx.x;
  float m = mi::neg_inf(), s = 0.f;
  if (col < k_cols) {
    for (int rb = threadIdx.y; rb < n_rb; rb += 8) {
      const float x = colpart[(size_t)rb * pitch + col];
      if (x > mi::neg_inf()) {
        const float mn = fmaxf(m, x);
        s = s * exp2f(m - mn) + exp2f(x - mn);
        m = mn;
      }
    }
  }
  shm[threadIdx.y][threadIdx.x] = m; shs[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y != 0 || col >= k_cols) return;
  float gm = mi::neg_inf();
  for (int y = 0; y < 8; ++y) gm = fmaxf(gm, shm[y][threadIdx.x]);
  float gs = 0.f;
  for (int y = 0; y < 8; ++y) if (shs[y][threadIdx.x] > 0.f) gs += shs[y][threadIdx.x] * exp2f(shm[y][threadIdx.x] - gm);
  col_lse[col] = gs > 0.f ? (gm + log2f(gs)) * mi::kLn2 : mi::neg_inf();
}

// one block: scal = {max lse_neg, sum exp(lse_neg - max), sum n_neg, sum diag, sum (lse_all - diag), #rows w/o neg, 0, 0}
__global__ void stats_reduce_kernel(const float4* __restrict__ row_out, int q_rows, double* __restrict__ scal,
                                    const int* __restrict__ run_if) {
  MI_PRED(run_if);
  __shared__ double sh[6][32];
  __shared__ float shm[32];
  __shared__ float gmax;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
  float m = mi::neg_inf();
  for (int r = tid; r < q_rows; r += blockDim.x) m = fmaxf(m, row_out[r].x);
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) shm[w] = m;
  __syncthreads();
  if (tid == 0) { float g = mi::neg_inf(); for (int i = 0; i < nw; ++i) g = fmaxf(g, shm[i]); gmax = g; }
  __syncthreads();
  const float g = gmax;
  double acc[5] = {0, 0, 0, 0, 0};
  for (int r = tid; r < q_rows; r += blockDim.x) {
    const float4 v = row_out[r];
    if (v.x > mi::neg_inf()) acc[0] += exp((double)v.x - (double)g);
    acc[1] += v.y; acc[2] += v.z; acc[3] += (double)v.w - (double)v.z;
    if (!(v.y > 0.f)) acc[4] += 1.0;
  }
  for (int k = 0; k < 5; ++k) {
    double a = acc[k];
    for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) sh[k][w] = a;
  }
  __syncthreads();
  if (tid == 0) {
    double t[5] = {0, 0, 0, 0, 0};
    for (int k = 0; k < 5; ++k) for (int i = 0; i < nw; ++i) t[k] += sh[k][i];
    scal[0] = g; scal[1] = t[0]; scal[2] = t[1]; scal[3] = t[2]; scal[4] = t[3]; scal[5] = t[4]; scal[6] = 0; scal[7] = 0;
  }
}
// the same reduction over kRedBlocks blocks: each block reduces its slice relative to its own maximum, the last block to
// finish (atomic ticket) merges the slices and resets the ticket.  red = {double part[kRedBlocks][8]; unsigned ticket} (zeroed once).
constexpr int kRedBlocks = 64;
struct RedScratch { double* part; unsigned* ticket; };
__global__ void stats_reduce_mb_kernel(const float4* __restrict__ row_out, int q_rows, double* __restrict__ scal,
                                       double* __restrict__ part, unsigned* __restrict__ ticket, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  __shared__ double sh[5][8];
  __shared__ float shm[8];
  __shared__ float bmax;
  __shared__ bool last;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;     // 256 threads
  const int per = (q_rows + gridDim.x - 1) / gridDim.x;
  const int r0 = blockIdx.x * per, r1 = min(q_rows, r0 + per);
  float m = mi::neg_inf();
  for (int r = r0 + tid; r < r1; r += blockDim.x) m = fmaxf(m, row_out[r].x);
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) shm[w] = m;
  __syncthreads();
  if (tid == 0) { float g = mi::neg_inf(); for (int i = 0; i < nw; ++i) g = fmaxf(g, shm[i]); bmax = g; }
  __syncthreads();
  const float g = bmax;
  double acc[5] = {0, 0, 0, 0, 0};
  for (int r = r0 + tid; r < r1; r += blockDim.x) {
    const float4 v = row_out[r];
    if (v.x > mi::neg_inf()) acc[0] += exp((double)v.x - (double)g);
    acc[1] += v.y; acc[2] += v.z; acc[3] += (double)v.w - (double)v.z;
    if (!(v.y > 0.f)) acc[4] += 1.0;
  }
  for (int k = 0; k < 5; ++k) {
    double a = acc[k];
    for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) sh[k][w] = a;
  }
  __syncthreads();
  if (tid == 0) {
    double t[5] = {0, 0, 0, 0, 0};
    for (int k = 0; k < 5; ++k) for (int i = 0; i < nw; ++i) t[k] += sh[k][i];
    double* p = part + blockIdx.x * 8;
    p[0] = g; p[1] = t[0]; p[2] = t[1]; p[3] = t[2]; p[4] = t[3]; p[5] = t[4];
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last || tid != 0) return;
  __threadfence();
  double gm = -INFINITY;
  for (unsigned b = 0; b < gridDim.x; ++b) gm = fmax(gm, part[b * 8]);
  double s = 0, t[4] = {0, 0, 0, 0};
  for (unsigned b = 0; b < gridDim.x; ++b) {
    const double* v = part + b * 8;
    if (isfinite(v[0])) s += v[1] * exp(v[0] - gm);
    for (int k = 0; k < 4; ++k) t[k] += v[2 + k];
  }
  scal[0] = gm; scal[1] = s; scal[2] = t[0]; scal[3] = t[1]; scal[4] = t[2]; scal[5] = t[3]; scal[6] = 0; scal[7] = 0;
  *ticket = 0u;
}
// scal[6] = number of rows whose single-pass reference left the safe window (travels with the rank's scalars)
__global__ void flag_to_scal_kernel(const int* __restrict__ flag, double* __restrict__ scal, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  scal[6] = static_cast<double>(flag[0]);
}

// ranks' reduced scalars [world][8] -> one row of the same layout (global max / rescaled sum-exp, plain sums).
// Slot 7 is summed too: the MLP critic's sharded single pass carries each block's sum of g~ there (0 everywhere else).
// `pitch` (doubles) between the ranks' rows: 8, or the record size of the symmetric step's packed exchange.
__global__ void merge_scal_kernel(const double* __restrict__ scal_all, int world, double* __restrict__ out, long long pitch = 8) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double gm = -INFINITY;
  for (int r = 0; r < world; ++r) gm = fmax(gm, scal_all[r * pitch]);
  double s = 0, t[6] = {0, 0, 0, 0, 0, 0};
  for (int r = 0; r < world; ++r) {
    const double* v = scal_all + r * pitch;
    if (isfinite(v[0])) s += v[1] * exp(v[0] - gm);
    for (int k = 0; k < 6; ++k) t[k] += v[2 + k];
  }
  out[0] = gm; out[1] = s; out[2] = t[0]; out[3] = t[1]; out[4] = t[2]; out[5] = t[3]; out[6] = t[4]; out[7] = t[5];
}

// fused glue: loss from the reduced scalars (fp64), and the scalar references as floats
// loss_out = { loss, pos_mean, lse_neg, n_neg, loss_row, loss_col, rows w/o negatives, guard rows }
// `lambda` (dv-like single pass only): the guard also trips when e^{lambda - LSE} would leave the fp32 range.
__global__ void loss_finalize_kernel(const double* __restrict__ scal_row, const double* __restrict__ scal_col,
                                     long long B, int estimator, double* __restrict__ loss_out, float* __restrict__ lse_f,
                                     const float* __restrict__ lambda, const int* __restrict__ run_if) {
  MI_PRED(run_if);
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double lse = scal_row[0] + log(scal_row[1]);
  const double n_neg = scal_row[2];
  const double pos = scal_row[3] / (double)B;
  const double loss_row = scal_row[4] / (double)B;
  const double loss_col = scal_col ? scal_col[4] / (double)B : 0.0;
  if (estimator == MI_EST_JS) {   // scal_row in js_reduce_kernel's layout; lse_f = 1 / N_neg, the weight of every negative in G
    const double sp_neg = scal_row[0] / n_neg, sp_pos = scal_row[4] / (double)B;
    loss_out[0] = sp_neg + sp_pos; loss_out[1] = pos; loss_out[2] = sp_neg; loss_out[3] = n_neg;
    loss_out[4] = sp_pos; loss_out[5] = 0.0; loss_out[6] = scal_row[5]; loss_out[7] = 0.0;
    if (lse_f) *lse_f = (float)(1.0 / n_neg);
    return;
  }
  double loss;
  if (estimator == MI_EST_DV) loss = lse - log((double)(float)n_neg) - pos;   // fp32 N_neg as mi_critics.py:10
  else if (estimator == MI_EST_INFONCE_REF) loss = lse - pos;
  else if (estimator == MI_EST_INFONCE_ROW) loss = loss_row;
  else if (estimator == MI_EST_NWJ) loss = exp(lse - log(n_neg) - 1.0) - pos;   // fp64 ln N_neg (no reference to mirror)
  else loss = 0.5 * (loss_row + loss_col);
  const bool nwj = estimator == MI_EST_NWJ;
  double guard = scal_row[6];
  if (lambda != nullptr && (estimator == MI_EST_DV || estimator == MI_EST_INFONCE_REF || nwj) && n_neg > 0.0 &&
      !(fabs((double)lambda[0] - lse) <= 60.0)) guard += 1.0;
  loss_out[0] = loss; loss_out[1] = pos; loss_out[2] = lse; loss_out[3] = n_neg;
  loss_out[4] = nwj ? 0.0 : loss_row; loss_out[5] = loss_col; loss_out[6] = scal_row[5]; loss_out[7] = guard;
  // NWJ: G = kappa softmax_M(S) - I/B with kappa = e^{LSE - ln N_neg - 1}, i.e. DV's G with LSE replaced by 1 + ln N_neg: the
  // finalisations (c_q = e^{ref_q - lse_f}, e^{lambda - lse_f}) then need no change
  if (lse_f) *lse_f = nwj ? (float)(log(n_neg) + 1.0) : (float)lse;
}

// ---- Jensen-Shannon (no normaliser: the weights sigma(S) lie in (0, 1))
// rows of one panel: row_out = {sum_k M softplus(S) (the partial row sums added), n_neg, S_ii, softplus(-S_ii)}
__global__ void js_rows_kernel(const float* __restrict__ part, int n_part, int rows_padded, int rows,
                               const int* __restrict__ n_same, int k_cols, const float* __restrict__ diag_in,
                               float4* __restrict__ row_out) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= rows) return;
  float l = 0.f;
  for (int p = 0; p < n_part; ++p) l += part[(size_t)p * rows_padded + row];
  const float d = diag_in[row];
  row_out[row] = make_float4(l, static_cast<float>(k_cols - n_same[row]), d, fmaxf(-d, 0.f) + log1pf(expf(-fabsf(d))));
}
// one block of kJsRedThreads, fixed order: scal = {sum M softplus(S), 0, n_neg, sum S_ii, sum softplus(-S_ii), rows w/o negatives, 0, 0}
constexpr int kJsRedThreads = 256;
__global__ void js_reduce_kernel(const float4* __restrict__ row_out, long long rows, double* __restrict__ scal) {
  __shared__ double sh[5][kJsRedThreads];
  double a[5] = {0, 0, 0, 0, 0};
  for (long long r = threadIdx.x; r < rows; r += kJsRedThreads) {
    const float4 v = row_out[r];
    a[0] += v.x; a[1] += v.y; a[2] += v.z; a[3] += v.w;
    if (!(v.y > 0.f)) a[4] += 1.0;
  }
  for (int k = 0; k < 5; ++k) sh[k][threadIdx.x] = a[k];
  __syncthreads();
  for (int o = kJsRedThreads / 2; o; o >>= 1) {
    if ((int)threadIdx.x < o) for (int k = 0; k < 5; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    scal[0] = sh[0][0]; scal[1] = 0.0; scal[2] = sh[1][0]; scal[3] = sh[2][0]; scal[4] = sh[3][0]; scal[5] = sh[4][0];
    scal[6] = 0.0; scal[7] = 0.0;
  }
}
// the gradients from the raw contractions: out[i,:] = alpha (w[0] raw[i,:] - (sigma(-S_ii) / B) sub[i,:]), w[0] = 1 / N_neg.
// The positive pair's weight is per row.  raw may equal out_f32 (in place).  8 elements / thread.
__global__ void js_finalize_kernel(const float* raw, long long D, long long rows, const float* __restrict__ w,
                                   const float* __restrict__ diag, float inv_b, float alpha,
                                   const __nv_bfloat16* __restrict__ sub, long long ld_sub, int sub_split, long long Dp,
                                   float* out_f32, __nv_bfloat16* __restrict__ out_bf16, __nv_bfloat16* __restrict__ out_lo, long long ld16) {
  const float c = w[0];
  for (long long idx = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 8; idx < rows * D;
       idx += (long long)gridDim.x * blockDim.x * 8) {
    const long long i = idx / D, d = idx - i * D;          // D % 8 == 0
    const float gam = inv_b / (1.f + expf(diag[i]));       // sigma(-S_ii) / B
    const uint4 kv = *reinterpret_cast<const uint4*>(sub + i * ld_sub + d);
    const uint32_t kw[4] = {kv.x, kv.y, kv.z, kv.w};
    float kd[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) { kd[2 * j] = __uint_as_float(kw[j] << 16); kd[2 * j + 1] = __uint_as_float(kw[j] & 0xffff0000u); }
    if (sub_split == 2) {
      const uint4 lv = *reinterpret_cast<const uint4*>(sub + i * ld_sub + Dp + d);
      const uint32_t lw[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) { kd[2 * j] += __uint_as_float(lw[j] << 16); kd[2 * j + 1] += __uint_as_float(lw[j] & 0xffff0000u); }
    }
    const float4 r0 = *reinterpret_cast<const float4*>(raw + idx), r1 = *reinterpret_cast<const float4*>(raw + idx + 4);
    const float rv[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = alpha * (c * rv[j] - gam * kd[j]);
    if (out_f32) {
      *reinterpret_cast<float4*>(out_f32 + idx) = make_float4(o[0], o[1], o[2], o[3]);
      *reinterpret_cast<float4*>(out_f32 + idx + 4) = make_float4(o[4], o[5], o[6], o[7]);
    }
    if (out_bf16) {
      uint32_t h[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) h[j] = ptx::pack_bf16(o[2 * j], o[2 * j + 1]);
      *reinterpret_cast<uint4*>(out_bf16 + i * ld16 + d) = make_uint4(h[0], h[1], h[2], h[3]);
      if (out_lo) {
        uint32_t l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
          l[j] = ptx::pack_bf16(o[2 * j] - __uint_as_float(h[j] << 16), o[2 * j + 1] - __uint_as_float(h[j] & 0xffff0000u));
        *reinterpret_cast<uint4*>(out_lo + i * ld16 + d) = make_uint4(l[0], l[1], l[2], l[3]);
      }
    }
  }
}

// ---- symmetric InfoNCE over row blocks (the batch-sharded step): each rank's column partials carry its own positive
//      pairs (col_pos_fold_kernel), so column j of the batch is the plain log-sum-exp of the ranks' partials and
//      loss_col = (sum_j c_j - sum_i S_ii) / B, with sum_i S_ii = slot 3 of the merged scalar row.
// col_lse[i] = logaddexp(col_lse[i], diag[i]), i < n (the caller offsets col_lse to the block's own columns)
__global__ void col_pos_fold_kernel(float* __restrict__ col_lse, const float* __restrict__ diag, long long n) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = col_lse[i], d = diag[i];
  const float hi = fmaxf(x, d), lo = fminf(x, d);
  col_lse[i] = hi + log1pf(expf(lo - hi));
}
// c_out[j] = (fp32 of) the fp64 log-sum-exp of col_all[r * pitch + j] over the ranks; part[block] = sum of the block's fp64
// c_j.  256 threads; the fixed tree order makes the sums independent of timing (every rank computes the same bits).
constexpr int kSymColThreads = 256;
__global__ void sym_col_kernel(const float* __restrict__ col_all, long long pitch, int world, long long B,
                               float* __restrict__ c_out, double* __restrict__ part) {
  __shared__ double sh[kSymColThreads];
  const long long j = blockIdx.x * (long long)kSymColThreads + threadIdx.x;
  double c = 0.0;
  if (j < B) {
    double m = -INFINITY;
    for (int r = 0; r < world; ++r) m = fmax(m, (double)col_all[r * pitch + j]);
    double s = 0.0;
    for (int r = 0; r < world; ++r) {
      const double x = col_all[r * pitch + j];
      if (x > -INFINITY) s += exp(x - m);
    }
    c = m > -INFINITY ? m + log(s) : -INFINITY;
    c_out[j] = (float)c;
  }
  sh[threadIdx.x] = c;
  __syncthreads();
  for (int o = kSymColThreads / 2; o; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[blockIdx.x] = sh[0];
}
// the column scalar row in the layout of the rows (loss_finalize_kernel reads slot 4): {0, 0, 0, sum S_ii, sum_j c_j - sum S_ii, 0, 0, 0}
__global__ void sym_col_row_kernel(const double* __restrict__ part, int n_part, const double* __restrict__ row_merged,
                                   double* __restrict__ col_row) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double s = 0.0;
  for (int b = 0; b < n_part; ++b) s += part[b];
  for (int k = 0; k < 8; ++k) col_row[k] = 0.0;
  col_row[3] = row_merged[3];
  col_row[4] = s - row_merged[3];
}
inline long long merge_sym_scratch_doubles(long long B) { return 16 + cdiv(B, kSymColThreads); }
// The ranks' scalar rows (pitch in doubles) and column partials with their own positive pairs folded in (pitch in floats)
// -> c_out [B] (the column references of the gradient pass) and loss_out in the layout of the single-GPU symmetric call.
int merge_sym_impl(const double* scal_all, long long scal_pitch, const float* col_all, long long col_pitch, int world, long long B,
                   double* loss_out, float* c_out, double* scratch, cudaStream_t stream) {
  const int nb = static_cast<int>(cdiv(B, kSymColThreads));
  double* rows = scratch; double* cols = scratch + 8; double* part = scratch + 16;
  sym_col_kernel<<<nb, kSymColThreads, 0, stream>>>(col_all, col_pitch, world, B, c_out, part);
  MI_LAUNCH_CHECK("sym_col_kernel");
  merge_scal_kernel<<<1, 32, 0, stream>>>(scal_all, world, rows, scal_pitch);
  MI_LAUNCH_CHECK("merge_scal_kernel");
  sym_col_row_kernel<<<1, 32, 0, stream>>>(part, nb, rows, cols);
  MI_LAUNCH_CHECK("sym_col_row_kernel");
  loss_finalize_kernel<<<1, 32, 0, stream>>>(rows, cols, B, MI_EST_INFONCE_SYM, loss_out, nullptr, nullptr, nullptr);
  MI_LAUNCH_CHECK("loss_finalize_kernel");
  return MI_OK;
}
// flag[0] = (loss_out[7] != 0): the device predicate of the exact fallback
__global__ void guard_to_flag_kernel(const double* __restrict__ loss_out, int* __restrict__ flag, double* __restrict__ guard_a) {
  guard_a[0] = loss_out[7];
  flag[0] = (loss_out[7] != 0.0) ? 1 : 0;
}
// after the (predicated) exact repeat: loss_out[7] keeps the number of rows that tripped the sampled pass (informational:
// > 0 means the results come from the exact repeat); a trip of the exact repeat itself is impossible by construction
// (l = 1 for every row) and would poison the loss instead of passing silently.
__global__ void guard_report_kernel(const int* __restrict__ flag_a, const double* __restrict__ guard_a, double* __restrict__ loss_out) {
  if (flag_a[0] != 0) {
    if (loss_out[7] != 0.0) loss_out[0] = nan("");
    loss_out[7] = guard_a[0];
  }
}

// dst[i] = const (from device scalar) or column `col` of row_out
__global__ void make_ref_kernel(float* __restrict__ dst, const float4* __restrict__ rows, int col,
                                const float* __restrict__ scalar, long long n) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (scalar) { dst[i] = *scalar; return; }
  const float4 v = rows[i];
  dst[i] = col == 0 ? v.x : col == 1 ? v.y : col == 2 ? v.z : v.w;
}

// out[r, c] (pitch ld_out) (+)= sum_p part[p][r, c] (compact partials, pitch ldp): split-K reduction
__global__ void reduce_partials_kernel(const float* __restrict__ part, int n_part, long long stride, long long ldp,
                                       float* __restrict__ out, long long ld_out, long long rows, long long cols, int accumulate,
                                       const int* __restrict__ run_if) {
  MI_PRED(run_if);
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const long long r = i / cols, c = i - r * cols;
  float a = accumulate ? out[r * ld_out + c] : 0.f;
  for (int p = 0; p < n_part; ++p) a += part[(size_t)p * stride + r * ldp + c];
  out[r * ld_out + c] = a;
}

inline unsigned blocks_for(long long n, int t) { return static_cast<unsigned>(cdiv(n, t)); }
// grid of a grid-stride elementwise kernel: enough blocks to fill the machine, few enough that a predicated-off launch is cheap
inline unsigned blocks_capped(long long n, int t) {
  const long long want = cdiv(n, t), cap = 16LL * num_sms();
  return static_cast<unsigned>(want < cap ? (want < 1 ? 1 : want) : cap);
}

// ------------------------------------------------------------------------------------ stages
// A bf16 operand [rows, D]; split == 2 means a hi/lo pair stored as [hi | lo] in one row, lo starting
// at column round_up(D, 64), with zeros in the gap (fp32-accumulate "strict" mode).
struct Opnd { const __nv_bfloat16* p; long long ld; int split; };

inline long long opnd_k_extent(const Opnd& o, long long D) { return o.split == 2 ? round_up(D, kSplitAlign) + D : D; }

// K segments for S = Q K^T when one of the operands is a hi/lo pair: (Q_hi + Q_lo) K^T or Q (K_hi + K_lo)^T
int score_segments(Sched& sc, const Opnd& q, const Opnd& k, long long D) {
  const int kb = static_cast<int>(round_up(D, kSplitAlign) / bk());
  single_segment(sc);
  sc.seg_len = kb;
  if (q.split == 2 && k.split == 2) return MI_ERR_BAD_ARG;
  if (q.split == 2) { sc.k_blocks = 2 * kb; sc.a_seg[1] = kb; }
  else if (k.split == 2) { sc.k_blocks = 2 * kb; sc.b_seg[1] = kb; }
  else { sc.k_blocks = static_cast<int>(cdiv(D, bk())); sc.seg_len = sc.k_blocks; }
  return MI_OK;
}

struct GemmArgs {
  MapSpec a, b;
  bool a_mn = false;          // A stored M-contiguous (transposed view of a row-major [K, M] matrix)
  bool b_mn = false;          // B stored N-contiguous (a row-major [K, N] matrix used as it is)
  long long M = 0, N = 0;
  int k_blocks = 0;           // total K blocks (all segments)
  int seg_len = 0;            // 0: one segment
  int a_seg[4] = {0, 0, 0, 0}, b_seg[4] = {0, 0, 0, 0}, a_moff[4] = {0, 0, 0, 0}, b_noff[4] = {0, 0, 0, 0};
  int ksplit = 1;
  int order = 1;              // Sched::order of the units: 1 = the K splits of a tile on neighbouring CTA pairs, 0 = the tiles of a
                              // K split on neighbouring pairs (they read the same operand rows at the same time: L2 sharing)
  float alpha = 1.f, gamma = 0.f;
  const __nv_bfloat16* sub = nullptr; const __nv_bfloat16* sub_lo = nullptr; long long ld_sub = 0;
  long long sub_row0 = 0, sub_rows = -1;   // SUB row r applies to output row sub_row0 + r (default: all rows)
  float* out_f32 = nullptr; long long ld_out = 0;
  __nv_bfloat16* out_bf16 = nullptr; __nv_bfloat16* out_bf16_lo = nullptr; long long ld_out16 = 0;
  bool accumulate = false;
  bool acc_first = false; const float* kappa_a = nullptr; const float* kappa_b = nullptr;   // see EpiStore::Params
  const float* bias = nullptr;                                   // [N] added after alpha (nn.Linear bias)
  const __nv_bfloat16* relu_mask = nullptr; long long ld_mask = 0;   // zero the result where relu_mask <= 0
};

int run_gemm(const GemmArgs& g, Bump& ws, cudaStream_t stream) {
  if (g.M <= 0 || g.N <= 0 || g.k_blocks <= 0) return MI_ERR_BAD_ARG;
  Sched sc;
  sc.n_mblk = static_cast<int>(cdiv(g.M, rows_per_mblk()));
  sc.n_ntile = static_cast<int>(cdiv(g.N, mi::TILE_N));
  sc.n_split = sc.n_ntile;           // one tile per unit
  sc.k_blocks = g.k_blocks;
  sc.n_ksplit = g.ksplit < 1 ? 1 : (g.ksplit > sc.k_blocks ? sc.k_blocks : g.ksplit);
  sc.order = g.order;                // 1: all N tiles (and K splits) of an M block run concurrently
  single_segment(sc);
  if (g.seg_len > 0) {
    sc.seg_len = g.seg_len;
    for (int i = 0; i < 4; ++i) { sc.a_seg[i] = g.a_seg[i]; sc.b_seg[i] = g.b_seg[i]; sc.a_moff[i] = g.a_moff[i]; sc.b_noff[i] = g.b_noff[i]; }
  }
  float* partial = nullptr;
  const long long ldp = round_up(g.N, 4);      // split-K partials are compact [M, ldp] blocks
  if (sc.n_ksplit > 1) partial = ws.take<float>(static_cast<size_t>(sc.n_ksplit) * g.M * ldp);
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (ws.dry) return MI_OK;
  if (!g.a.ptr || !g.b.ptr || (!g.out_f32 && !g.out_bf16)) return MI_ERR_BAD_ARG;
  mi::EpiStore::Params ep;
  const bool sk = sc.n_ksplit > 1;
  ep.out_f32 = sk ? partial : g.out_f32;
  ep.out_bf16 = sk ? nullptr : g.out_bf16;
  ep.out_bf16_lo = sk ? nullptr : g.out_bf16_lo;
  ep.ld_out = sk ? ldp : g.ld_out; ep.ld_out16 = g.ld_out16;
  ep.bias = sk ? nullptr : g.bias; ep.relu_mask = sk ? nullptr : g.relu_mask; ep.ld_mask = g.ld_mask;
  ep.acc_first = (!sk && g.acc_first) ? 1 : 0; ep.kappa_a = g.kappa_a; ep.kappa_b = g.kappa_b;
  ep.rows = static_cast<int>(g.M); ep.cols = static_cast<int>(g.N);
  ep.alpha = g.alpha; ep.gamma = g.gamma;
  ep.sub = sk ? nullptr : g.sub; ep.sub_lo = sk ? nullptr : g.sub_lo; ep.ld_sub = g.ld_sub;
  ep.sub_row0 = static_cast<int>(g.sub_row0); ep.sub_rows = static_cast<int>(g.sub_rows < 0 ? g.M : g.sub_rows);
  ep.ksplit_stride = static_cast<long long>(g.M) * ldp;
  ep.accumulate = (!sk && g.accumulate) ? 1 : 0;
  if (g.a_mn && g.b_mn) MI_TRY((launch_engine<mi::EpiStore, true, true>(g.a, g.b, sc, ep, stream)));
  else if (g.a_mn) MI_TRY((launch_engine<mi::EpiStore, true, false>(g.a, g.b, sc, ep, stream)));
  else if (g.b_mn) MI_TRY((launch_engine<mi::EpiStore, false, true>(g.a, g.b, sc, ep, stream)));
  else MI_TRY((launch_engine<mi::EpiStore, false, false>(g.a, g.b, sc, ep, stream)));
  if (sk) {
    if (!g.out_f32 || g.sub || g.bias || g.relu_mask || g.acc_first || g.alpha != 1.f) return MI_ERR_BAD_ARG;
    const long long n = static_cast<long long>(g.M) * g.N;
    reduce_partials_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(partial, sc.n_ksplit, static_cast<long long>(g.M) * ldp, ldp,
                                                                   g.out_f32, g.ld_out, g.M, g.N, g.accumulate ? 1 : 0, t_run_if);
    MI_LAUNCH_CHECK("reduce_partials_kernel");
  }
  return MI_OK;
}

// C = alpha (A B^T - gamma SUB) with optional hi/lo split operands / output (plain K-major operands)
int gemm_impl(const Opnd& A, const Opnd& B, long long M, long long N, long long K,
              float alpha, float gamma, const void* sub, long long ld_sub,
              float* out_f32, long long ld_out, void* out_bf16, long long ld_out16, int out_split, int ksplit,
              Bump& ws, cudaStream_t stream) {
  if (M <= 0 || N <= 0 || K <= 0) return MI_ERR_BAD_ARG;
  GemmArgs g;
  const bool any_split = A.split == 2 || B.split == 2;
  const int kb = static_cast<int>(any_split ? round_up(K, kSplitAlign) / bk() : cdiv(K, bk()));
  g.a = MapSpec{A.p, M, opnd_k_extent(A, K), A.ld};
  g.b = MapSpec{B.p, N, opnd_k_extent(B, K), B.ld};
  g.M = M; g.N = N; g.k_blocks = kb; g.seg_len = kb;
  if (A.split == 2 && B.split == 2) {           // hi*hi + lo*hi + hi*lo
    g.k_blocks = 3 * kb; g.a_seg[1] = kb; g.b_seg[2] = kb;
  } else if (A.split == 2) { g.k_blocks = 2 * kb; g.a_seg[1] = kb; }
  else if (B.split == 2) { g.k_blocks = 2 * kb; g.b_seg[1] = kb; }
  g.ksplit = ksplit;
  g.alpha = alpha; g.gamma = gamma; g.sub = static_cast<const __nv_bfloat16*>(sub); g.ld_sub = ld_sub;
  g.out_f32 = out_f32; g.ld_out = ld_out;
  g.out_bf16 = static_cast<__nv_bfloat16*>(out_bf16); g.ld_out16 = ld_out16;
  g.out_bf16_lo = (out_split == 2 && out_bf16) ? g.out_bf16 + round_up(N, kSplitAlign) : nullptr;
  return run_gemm(g, ws, stream);
}

// C = A B^T with either operand stored K-major ([rows, K]) or MN-major (row-major [K, rows], read in place through
// MN-major UMMA descriptors — no transposed copy); hi/lo operands add the cross terms as K segments.
// ksplit = 0: split-K chosen from the tile count (fp32 output only).
int gemm_mn_impl(const Opnd& A, bool a_mn, const Opnd& B, bool b_mn, long long M, long long N, long long K,
                 float* out_f32, long long ld_out, void* out_bf16, long long ld_out16, int out_split, int ksplit,
                 Bump& ws, cudaStream_t stream) {
  if (M <= 0 || N <= 0 || K <= 0) return MI_ERR_BAD_ARG;
  GemmArgs g;
  const bool a_sp = A.split == 2, b_sp = B.split == 2;
  const bool k_pad = (a_sp && !a_mn) || (b_sp && !b_mn);          // a K-major hi/lo pair fixes the lo offset at round_up(K, 128)
  const int kb = static_cast<int>(k_pad ? round_up(K, kSplitAlign) / bk() : cdiv(K, bk()));
  const long long Mp = round_up(M, kSplitAlign), Np = round_up(N, kSplitAlign);
  g.a_mn = a_mn; g.b_mn = b_mn;
  g.a = a_mn ? MapSpec{A.p, K, a_sp ? Mp + M : M, A.ld} : MapSpec{A.p, M, opnd_k_extent(A, K), A.ld};
  g.b = b_mn ? MapSpec{B.p, K, b_sp ? Np + N : N, B.ld} : MapSpec{B.p, N, opnd_k_extent(B, K), B.ld};
  g.M = M; g.N = N; g.seg_len = kb;
  int seg = 1;
  if (a_sp) { if (a_mn) g.a_moff[seg] = static_cast<int>(Mp); else g.a_seg[seg] = kb; ++seg; }      // A_lo B_hi
  if (b_sp) { if (b_mn) g.b_noff[seg] = static_cast<int>(Np); else g.b_seg[seg] = kb; ++seg; }      // A_hi B_lo
  g.k_blocks = seg * kb;
  if (ksplit == 0) {
    const long long tiles = cdiv(M, rows_per_mblk()) * cdiv(N, mi::TILE_N);
    ksplit = (out_f32 && !out_bf16) ? choose_ksplit(tiles, g.k_blocks) : 1;
  }
  g.ksplit = ksplit;
  g.out_f32 = out_f32; g.ld_out = ld_out;
  g.out_bf16 = static_cast<__nv_bfloat16*>(out_bf16); g.ld_out16 = ld_out16;
  g.out_bf16_lo = (out_split == 2 && out_bf16) ? g.out_bf16 + Np : nullptr;
  return run_gemm(g, ws, stream);
}

int transpose_impl(const void* in, long long ld_in, void* out, long long ld_out, long long R, long long C, cudaStream_t stream) {
  if (!in || !out || R <= 0 || C <= 0) return MI_ERR_BAD_ARG;
  dim3 grid(static_cast<unsigned>(cdiv(C, 64)), static_cast<unsigned>(cdiv(R, 64)));
  transpose_bf16_kernel<<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(in), ld_in,
                                                  static_cast<__nv_bfloat16*>(out), ld_out, R, C);
  MI_LAUNCH_CHECK("transpose_bf16_kernel");
  return MI_OK;
}

// hash pre-pass + padded study ids: everything the epilogue's negatives mask needs
struct MaskBuf { int* sidk_pad; unsigned long long* keys; int* counts; int* members; int4* excl; int* n_same; long long slots; };

MaskBuf take_mask(Bump& ws, long long Bq, long long k_pad, long long Bk) {
  MaskBuf b;
  long long slots = 64;
  while (slots < 2 * Bk) slots *= 2;
  b.slots = slots;
  b.sidk_pad = ws.take<int>(k_pad);
  b.keys = ws.take<unsigned long long>(slots); b.counts = ws.take<int>(slots); b.members = ws.take<int>(slots * mi::kMaxExcl);
  b.excl = ws.take<int4>(Bq); b.n_same = ws.take<int>(Bq);
  return b;
}

int build_mask(const MaskBuf& b, const int* sid_q, const int* sid_k, long long Bq, long long Bk, long long k_pad, cudaStream_t stream) {
  const int* pr = t_run_if;
  pad_int_kernel<<<blocks_for(k_pad, 256), 256, 0, stream>>>(sid_k, b.sidk_pad, Bk, k_pad, -2, pr);
  MI_LAUNCH_CHECK("pad_int_kernel");
  excl_init_kernel<<<blocks_for(b.slots, 256), 256, 0, stream>>>(b.keys, b.counts, b.members, b.slots, pr);
  MI_LAUNCH_CHECK("excl_init_kernel");
  const uint32_t mask = static_cast<uint32_t>(b.slots - 1);
  excl_insert_kernel<<<blocks_for(Bk, 256), 256, 0, stream>>>(sid_k, Bk, b.keys, b.counts, b.members, mask, pr);
  MI_LAUNCH_CHECK("excl_insert_kernel");
  excl_lookup_kernel<<<blocks_for(Bq, 256), 256, 0, stream>>>(sid_q, Bq, b.keys, b.counts, b.members, mask, b.excl, b.n_same, pr);
  MI_LAUNCH_CHECK("excl_lookup_kernel");
  return MI_OK;
}

RedScratch take_red(Bump& ws) {
  RedScratch r;
  r.part = ws.take<double>(kRedBlocks * 8);
  r.ticket = ws.take<unsigned>(1);
  return r;
}
// {max, sum-exp, sums} of the per-row statistics -> scal[8]; the ticket is zeroed here (stream ordered), the kernel resets it
int reduce_rows(const float* row_out, long long rows, double* scal, const RedScratch& red, cudaStream_t stream) {
  MI_CUDA(cudaMemsetAsync(red.ticket, 0, sizeof(unsigned), stream));
  const int nb = static_cast<int>(std::min<long long>(kRedBlocks, std::max<long long>(1, rows / 2048)));
  stats_reduce_mb_kernel<<<nb, 256, 0, stream>>>(reinterpret_cast<const float4*>(row_out), static_cast<int>(rows), scal, red.part,
                                                 red.ticket, t_run_if);
  MI_LAUNCH_CHECK("stats_reduce_mb_kernel");
  return MI_OK;
}

int stats_impl(const Opnd& Q, const Opnd& K, const int* sid_q, const int* sid_k,
               long long q_offset, long long Bq, long long Bk, long long D, float scale,
               float* row_out, double* scal_out, Bump& ws, cudaStream_t stream) {
  if (Bq <= 0 || Bk <= 0 || D <= 0 || (D % 8) != 0) return MI_ERR_BAD_ARG;
  Sched sc;
  sc.n_mblk = static_cast<int>(cdiv(Bq, rows_per_mblk()));
  sc.n_ntile = static_cast<int>(cdiv(Bk, mi::TILE_N));
  sc.n_split = choose_split(sc.n_mblk, sc.n_ntile, num_pairs());
  sc.n_ksplit = 1; sc.order = 0;
  MI_TRY(score_segments(sc, Q, K, D));
  const long long k_pad = static_cast<long long>(sc.n_ntile) * mi::TILE_N;
  const int rows_padded = sc.n_mblk * rows_per_mblk();
  const MaskBuf mb = take_mask(ws, Bq, k_pad, Bk);
  float4* part = ws.take<float4>(static_cast<size_t>(sc.n_split) * mi::kColQuarters * rows_padded);
  float* diag = ws.take<float>(Bq);
  const RedScratch red = take_red(ws);
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (ws.dry) return MI_OK;
  if (!Q.p || !K.p || !sid_q || !sid_k || !row_out || !scal_out || !(scale > 0.f)) return MI_ERR_BAD_ARG;
  MI_TRY(build_mask(mb, sid_q, sid_k, Bq, Bk, k_pad, stream));
  diag_kernel<<<blocks_for(Bq * 32, 256), 256, 0, stream>>>(Q.p, Q.ld, Q.split, K.p, K.ld, K.split, q_offset, Bq, D,
                                                             round_up(D, kSplitAlign), scale, diag, t_run_if);
  MI_LAUNCH_CHECK("diag_kernel");
  mi::EpiStats::Params ep;
  ep.mask = mi::MaskInfo{mb.excl, mb.n_same, sid_q, mb.sidk_pad};
  ep.q_rows = static_cast<int>(Bq); ep.k_cols = static_cast<int>(Bk);
  ep.scale = scale; ep.part = part; ep.rows_padded = rows_padded;
  MI_TRY(launch_engine<mi::EpiStats>(MapSpec{Q.p, Bq, opnd_k_extent(Q, D), Q.ld}, MapSpec{K.p, Bk, opnd_k_extent(K, D), K.ld},
                                     sc, ep, stream));
  stats_merge_kernel<<<blocks_for(Bq, 128), 128, 0, stream>>>(part, sc.n_split * mi::kColQuarters, rows_padded, static_cast<int>(Bq),
                                                              mb.n_same, static_cast<int>(Bk), diag, reinterpret_cast<float4*>(row_out));
  MI_LAUNCH_CHECK("stats_merge_kernel");
  MI_TRY(reduce_rows(row_out, Bq, scal_out, red, stream));
  return MI_OK;
}

// Row AND column statistics of the SQUARE score matrix S = scale Q K^T (same study ids on both sides) from ONE score
// computation (EpiStatsRC) — the symmetric estimator's statistics for 2 B^2 D instead of 4 B^2 D.
// Row AND column statistics of the score block S[q_offset + r, c] = scale <Q_r, K_c>, r < Bq, c < Bk, from ONE pass.
// Square use (Bq == Bk, q_offset = 0; the 1-GPU symmetric estimator): col_out / scal_col receive the columns in the layout of
// the rows.  Row-block use (a rank's rows of the batch-sharded step): col_lse receives, for every column, the log-sum-exp
// over this block's negatives; the caller merges the ranks.  include_pos (row-block use): col_lse also holds the block's
// positive pairs, col_lse[q_offset + r] = logaddexp(col_lse[q_offset + r], S[r, q_offset + r]).
// ev_k_ready / k_local_valid schedule the score tiles as single_pass_impl does: the own column block first, then the wait
// for the other ranks' K rows.  shared_mask: the negatives mask of (sid_q, sid_k), built by the caller.
int stats_rc_impl(const Opnd& Q, const Opnd& K, const int* sid_q, const int* sid_k, long long q_offset, long long Bq, long long Bk,
                  long long D, float scale, float* row_out, double* scal_row, float* col_out, double* scal_col, float* col_lse,
                  Bump& ws, cudaStream_t stream, cudaEvent_t ev_k_ready = nullptr, bool k_local_valid = false,
                  const MaskBuf* shared_mask = nullptr, bool include_pos = false) {
  if (Bq <= 0 || Bk <= 0 || D <= 0 || (D % 8) != 0 || q_offset < 0 || q_offset + Bq > Bk) return MI_ERR_BAD_ARG;
  const bool square = col_lse == nullptr;
  if (square && (Bq != Bk || q_offset != 0 || include_pos) && !ws.dry) return MI_ERR_BAD_ARG;
  Sched sc;
  sc.n_mblk = static_cast<int>(cdiv(Bq, rows_per_mblk()));
  sc.n_ntile = static_cast<int>(cdiv(Bk, mi::TILE_N));
  sc.n_split = choose_split(sc.n_mblk, sc.n_ntile, num_pairs());
  sc.n_ksplit = 1; sc.order = 0;
  MI_TRY(score_segments(sc, Q, K, D));
  const long long k_pad = static_cast<long long>(sc.n_ntile) * mi::TILE_N;
  const int rows_padded = sc.n_mblk * rows_per_mblk();
  const int n_rb = rows_padded / 32;
  const int max_split = sc.n_split;
  const MaskBuf mb = shared_mask != nullptr ? *shared_mask : take_mask(ws, Bq, k_pad, Bk);
  // (x3: up to three launches append their row partials — own columns first, the rest once K has arrived)
  float4* part = ws.take<float4>(3 * static_cast<size_t>(max_split) * mi::kColQuarters * rows_padded);
  float* diag = ws.take<float>(Bq);
  float* colpart = ws.take<float>(static_cast<size_t>(n_rb) * k_pad);
  const RedScratch red = take_red(ws);
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (ws.dry) return MI_OK;
  if (!Q.p || !K.p || !sid_q || !sid_k || !row_out || !scal_row || !(scale > 0.f)) return MI_ERR_BAD_ARG;
  if (square && (!col_out || !scal_col)) return MI_ERR_BAD_ARG;
  if (shared_mask == nullptr) MI_TRY(build_mask(mb, sid_q, sid_k, Bq, Bk, k_pad, stream));
  const long long own_t0 = q_offset / mi::TILE_N, own_t1 = (q_offset + Bq) / mi::TILE_N;
  const bool own_first = ev_k_ready != nullptr && k_local_valid && (q_offset % mi::TILE_N) == 0 && (Bq % mi::TILE_N) == 0 && Bq < Bk;
  if (ev_k_ready != nullptr && !own_first) MI_CUDA(cudaStreamWaitEvent(stream, ev_k_ready, 0));
  diag_kernel<<<blocks_for(Bq * 32, 256), 256, 0, stream>>>(Q.p, Q.ld, Q.split, K.p, K.ld, K.split, q_offset, Bq, D,
                                                             round_up(D, kSplitAlign), scale, diag, t_run_if);
  MI_LAUNCH_CHECK("diag_kernel");
  // a launch covers the N tiles [t0, t1): its row partials are appended, its column partials are its own columns
  int n_part = 0;
  auto score_tiles = [&](long long t0, long long t1) -> int {
    if (t1 <= t0) return MI_OK;
    Sched s = sc;
    s.n_ntile = static_cast<int>(t1 - t0);
    s.n_split = std::min(choose_split(s.n_mblk, s.n_ntile, num_pairs()), max_split);
    MI_TRY(score_segments(s, Q, K, D));
    s.nt_base = static_cast<int>(t0);
    mi::EpiStatsRC::Params ep;
    ep.mask = mi::MaskInfo{mb.excl, mb.n_same, sid_q, mb.sidk_pad};
    ep.q_rows = static_cast<int>(Bq); ep.k_cols = static_cast<int>(Bk);
    ep.scale = scale; ep.part = part + static_cast<size_t>(n_part) * rows_padded; ep.rows_padded = rows_padded;
    ep.colpart = colpart; ep.col_pitch = k_pad;
    MI_TRY(launch_engine<mi::EpiStatsRC>(MapSpec{Q.p, Bq, opnd_k_extent(Q, D), Q.ld}, MapSpec{K.p, Bk, opnd_k_extent(K, D), K.ld},
                                         s, ep, stream));
    n_part += s.n_split * mi::kColQuarters;
    return MI_OK;
  };
  if (own_first) {
    MI_TRY(score_tiles(own_t0, own_t1));                               // this rank's own columns: K rows already here
    MI_CUDA(cudaStreamWaitEvent(stream, ev_k_ready, 0));               // the other ranks' text embeddings
    MI_TRY(score_tiles(0, own_t0));
    MI_TRY(score_tiles(own_t1, sc.n_ntile));
  } else {
    MI_TRY(score_tiles(0, sc.n_ntile));
  }
  stats_merge_kernel<<<blocks_for(Bq, 128), 128, 0, stream>>>(part, n_part, rows_padded, static_cast<int>(Bq),
                                                              mb.n_same, static_cast<int>(Bk), diag, reinterpret_cast<float4*>(row_out));
  MI_LAUNCH_CHECK("stats_merge_kernel");
  MI_TRY(reduce_rows(row_out, Bq, scal_row, red, stream));
  if (square) {
    col_merge_kernel<<<static_cast<unsigned>(cdiv(Bk, 32)), dim3(32, 8), 0, stream>>>(colpart, n_rb, k_pad, static_cast<int>(Bk), mb.n_same,
                                                                                       static_cast<int>(Bq), diag, reinterpret_cast<float4*>(col_out));
    MI_LAUNCH_CHECK("col_merge_kernel");
    MI_TRY(reduce_rows(col_out, Bk, scal_col, red, stream));
  } else {
    col_lse_kernel<<<static_cast<unsigned>(cdiv(Bk, 32)), dim3(32, 8), 0, stream>>>(colpart, n_rb, k_pad, static_cast<int>(Bk), col_lse);
    MI_LAUNCH_CHECK("col_lse_kernel");
    if (include_pos) {
      col_pos_fold_kernel<<<blocks_for(Bq, 256), 256, 0, stream>>>(col_lse + q_offset, diag, Bq);
      MI_LAUNCH_CHECK("col_pos_fold_kernel");
    }
  }
  return MI_OK;
}

// Sampled references sit kRefMargin nats above the sample's log-sum-exp (see ref_merge_kernel).  The sample is a subset of
// the row's columns, so the row's true log-sum-exp can only lie ABOVE the sample's: with the margin a row stays inside the
// safe window while its true log-sum-exp is up to ~117 nats above what the sample saw (row sum <= 1e30), and entries more
// than 87 - 48 = 39 nats below the row's log-sum-exp (relative weight < 1e-17) flush to zero.
constexpr float kRefMargin = 48.f;

// Column sample of the single pass's references: stride such that about g_ref_sample_cols columns are scored per row;
// 1 (every column: exact references, the pass can never leave the safe window) when the sample would not be cheaper
// than ~80 us of tensor time — below that the exact statistics pass costs less than the predicated repeat's empty launches.
long long ref_stride_auto(long long Bq, long long ncols, long long D) {
  const long long target = g_ref_sample_cols.load(std::memory_order_relaxed);
  if (target <= 0) return 1;
  long long stride = ncols / target;
  if (stride < 2) return 1;
  if (2.0 * static_cast<double>(Bq) * static_cast<double>(ncols) * static_cast<double>(D) < 1.0e11 && target >= 2048) return 1;
  return stride;
}

// Per-row softmax references of the single pass (see ref_merge_kernel) from the columns c0 + s * stride, s in [0, ns),
// ns = ceil(nc / stride), of K — one statistics launch over a strided view of K (a TMA map whose row pitch is
// stride * ld; no gather).  `margin` lifts the references above the sample's log-sum-exp (kRefMargin whenever the sampled
// columns are a proper subset of the row's columns, 0 when they are all of them).  Also: diag_out[q] = the positive-pair
// score S[q, q_offset + q]; lam_out[0] = max_q ref_out[q] - margin.
int ref_sample_impl(const Opnd& Q, const Opnd& K, const int* sid_q, const int* sid_k, long long q_offset,
                    long long Bq, long long Bk, long long D, float scale, int include_diag,
                    long long c0, long long nc, long long stride, float margin,
                    float* ref_out, float* diag_out, float* lam_out, Bump& ws, cudaStream_t stream,
                    const MaskBuf* shared_mask = nullptr /* stride 1 over all columns: a mask the caller has built already */) {
  if (Bq <= 0 || Bk <= 0 || D <= 0 || (D % 8) != 0 || stride < 1 || c0 < 0 || nc <= 0 || c0 + nc > Bk) return MI_ERR_BAD_ARG;
  if (shared_mask != nullptr && (stride != 1 || c0 != 0 || nc != Bk)) return MI_ERR_BAD_ARG;
  const long long ns = cdiv(nc, stride);
  Sched sc;
  sc.n_mblk = static_cast<int>(cdiv(Bq, rows_per_mblk()));
  sc.n_ntile = static_cast<int>(cdiv(ns, mi::TILE_N));
  sc.n_split = choose_split(sc.n_mblk, sc.n_ntile, num_pairs());
  sc.n_ksplit = 1; sc.order = 0;
  MI_TRY(score_segments(sc, Q, K, D));
  const long long k_pad = static_cast<long long>(sc.n_ntile) * mi::TILE_N;
  const int rows_padded = sc.n_mblk * rows_per_mblk();
  const MaskBuf mb = shared_mask != nullptr ? *shared_mask : take_mask(ws, Bq, k_pad, ns);
  int* sid_s = ws.take<int>(ns);
  float4* part = ws.take<float4>(static_cast<size_t>(sc.n_split) * mi::kColQuarters * rows_padded);
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (ws.dry) return MI_OK;
  if (!Q.p || !K.p || !sid_q || !sid_k || !ref_out || !diag_out || !(scale > 0.f)) return MI_ERR_BAD_ARG;
  const int* pr = t_run_if;
  const int* sid_cols = sid_k + c0;
  if (stride > 1) {
    gather_int_kernel<<<blocks_for(ns, 256), 256, 0, stream>>>(sid_k + c0, stride, sid_s, ns, pr);
    MI_LAUNCH_CHECK("gather_int_kernel");
    sid_cols = sid_s;
  }
  if (shared_mask == nullptr) MI_TRY(build_mask(mb, sid_q, sid_cols, Bq, ns, k_pad, stream));
  diag_kernel<<<blocks_for(Bq * 32, 256), 256, 0, stream>>>(Q.p, Q.ld, Q.split, K.p, K.ld, K.split, q_offset, Bq, D,
                                                             round_up(D, kSplitAlign), scale, diag_out, pr);
  MI_LAUNCH_CHECK("diag_kernel");
  mi::EpiStats::Params ep;
  ep.mask = mi::MaskInfo{mb.excl, mb.n_same, sid_q, mb.sidk_pad};
  ep.q_rows = static_cast<int>(Bq); ep.k_cols = static_cast<int>(ns);
  ep.scale = scale; ep.part = part; ep.rows_padded = rows_padded;
  MI_TRY(launch_engine<mi::EpiStats>(MapSpec{Q.p, Bq, opnd_k_extent(Q, D), Q.ld},
                                     MapSpec{K.p + c0 * K.ld, ns, opnd_k_extent(K, D), K.ld * stride}, sc, ep, stream));
  ref_merge_kernel<<<blocks_for(Bq, 128), 128, 0, stream>>>(part, sc.n_split * mi::kColQuarters, rows_padded, static_cast<int>(Bq),
                                                            diag_out, include_diag, margin, ref_out, pr);
  MI_LAUNCH_CHECK("ref_merge_kernel");
  if (lam_out != nullptr) {
    // lambda = the largest SAMPLE log-sum-exp (the margin taken out again): e^{S - lambda} is then centred on the global scale
    max_reduce_kernel<<<1, 1024, 0, stream>>>(ref_out, Bq, lam_out, margin, pr);
    MI_LAUNCH_CHECK("max_reduce_kernel");
  }
  return MI_OK;
}

// rows of the dS panel per pass: make the panel GEMM's tile count a multiple of the pair count
long long panel_mblks(long long Bq, long long Bk, long long D, int precision) {
  const int U = num_pairs();
  const int ntD = static_cast<int>(cdiv(D, mi::TILE_N));
  long long mb = U / gcd_i(U, ntD);
  const long long total = cdiv(Bq, rows_per_mblk());
  if (mb > total) mb = total;
  const long long pitch = cdiv(Bk, mi::TILE_N) * mi::TILE_N * (precision == MI_PREC_BF16_STRICT ? 2 : 1);
  const long long cap = 6LL << 30;
  while (mb > 1 && mb * rows_per_mblk() * pitch * 2 > cap) mb = (mb + 1) / 2;
  return mb;
}

// The tensor core adds into its fp32 accumulator with truncation, not round-to-nearest: a chain of n accumulating MMAs
// carries a systematic relative bias of ~n * 2^-25 (measured at B = 65536: 12288 MMAs per output element of the
// dS x Y contraction in strict mode left a 2e-4 bias in dT, which the batch-coherent sum dW = X^T dT amplified to 4e-3).
// Strict ("fp32-accumulate") mode therefore cuts every long contraction into chains of at most kStrictChainBlocks K blocks
// (split-K: partial tiles summed by a separate fp32 round-to-nearest pass).  Fast mode keeps one chain (bound 1e-2).
constexpr int kStrictChainBlocks = 128;
inline int strict_ksplit(int k_blocks) { return static_cast<int>(cdiv(k_blocks, kStrictChainBlocks)); }

struct GradOut {            // fp32 and/or bf16 (split == 2: [hi | lo] rows) destination
  float* f32 = nullptr; long long ld = 0;
  __nv_bfloat16* bf16 = nullptr; long long ld16 = 0; int split = 1;
};

// The fused gradient pass with EXACT references (symmetric InfoNCE, and the mi_score_grad stage op).  For every row panel
// of Q: (1) recompute score tiles and write the bf16 dS panel P (EpiPStore), (2) Ok += alpha (P^T Q[panel] - gamma Q_diag)
// with P read MN-major from the same panel, (3) Oq[panel] = alpha (P K - gamma K_diag) — one score recompute serves both
// gradients; K and Q are read in place as MN-major B operands (no transposed copies).  "diag" is the positive-pair term:
// row q pairs with column q_offset + q.  P is a bounded row panel in `ws`, streamed through HBM panel by panel.
int grad_impl(const Opnd& Q, const Opnd& K, const int* sid_q, const int* sid_k,
              long long q_offset, long long Bq, long long Bk, long long D, float scale,
              const float* refq, float wq, const float* refk, float wk, int include_diag, int precision,
              float alpha, float gamma, const GradOut& oq, const GradOut* ok, Bump& ws, cudaStream_t stream,
              cudaEvent_t ev_after_k = nullptr,
              const MaskBuf* shared_mask = nullptr /* the negatives mask of (sid_q, sid_k), built by the caller */) {
  if (Bq <= 0 || Bk <= 0 || D <= 0 || (D % 8) != 0) return MI_ERR_BAD_ARG;
  typedef __nv_bfloat16 bf;
  const bool strict = precision == MI_PREC_BF16_STRICT;
  const int n_ntile = static_cast<int>(cdiv(Bk, mi::TILE_N));
  const long long k_pad = static_cast<long long>(n_ntile) * mi::TILE_N;
  const int kp = static_cast<int>(k_pad / bk());
  const long long pitch = k_pad * (strict ? 2 : 1);
  const long long Dp = round_up(D, kSplitAlign);
  const bool k_hl = strict && K.split == 2, q_hl = strict && Q.split == 2;
  const long long mb_panel = panel_mblks(Bq, Bk, D, precision);
  const long long panel_rows = mb_panel * rows_per_mblk();
  const MaskBuf mb = shared_mask != nullptr ? *shared_mask : take_mask(ws, Bq, k_pad, Bk);
  float* refk2 = ws.take<float>(k_pad);
  bf* P = ws.take<bf>(static_cast<size_t>(panel_rows) * pitch);
  // strict: the Oq contraction runs as short split-K chains into a raw fp32 panel, finished by an elementwise pass
  const int oq_ksplit = strict ? strict_ksplit(kp * (k_hl ? 3 : 2)) : 1;
  const size_t kpart_elems = oq_ksplit > 1 ? static_cast<size_t>(oq_ksplit) * panel_rows * round_up(D, 4) : 0;
  float* kpart = oq_ksplit > 1 ? ws.take<float>(kpart_elems) : nullptr;
  float* oq_rawp = oq_ksplit > 1 ? ws.take<float>(static_cast<size_t>(panel_rows) * D) : nullptr;
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (ws.dry) return MI_OK;
  if (!Q.p || !K.p || !sid_q || !sid_k || (!oq.f32 && !oq.bf16 && !ok)) return MI_ERR_BAD_ARG;
  const bool use_q = refq != nullptr && wq > 0.f, use_k = refk != nullptr && wk > 0.f;
  if ((!use_q && !use_k) || !(scale > 0.f)) return MI_ERR_BAD_ARG;

  if (shared_mask == nullptr) MI_TRY(build_mask(mb, sid_q, sid_k, Bq, Bk, k_pad, stream));
  if (use_k) {
    make_refk2_kernel<<<blocks_for(k_pad, 256), 256, 0, stream>>>(refk, logf(wk), refk2, Bk, k_pad);
    MI_LAUNCH_CHECK("make_refk2_kernel");
  }
  const Opnd Qe{Q.p, Q.ld, strict ? Q.split : 1}, Ke{K.p, K.ld, strict ? K.split : 1};

  for (long long r0 = 0; r0 < Bq; r0 += panel_rows) {
    const long long rows = (Bq - r0 < panel_rows) ? (Bq - r0) : panel_rows;
    // (1) dS panel
    Sched sc;
    sc.n_mblk = static_cast<int>(cdiv(rows, rows_per_mblk()));
    sc.n_ntile = n_ntile;
    sc.n_split = choose_split(sc.n_mblk, sc.n_ntile, num_pairs());
    sc.n_ksplit = 1; sc.order = 0;
    MI_TRY(score_segments(sc, Qe, Ke, D));
    mi::EpiPStore::Params ep;
    ep.mask = mi::MaskInfo{mb.excl + r0, mb.n_same + r0, sid_q + r0, mb.sidk_pad};
    ep.q_rows = static_cast<int>(rows); ep.k_cols = static_cast<int>(Bk);
    ep.q_offset = q_offset + r0; ep.scale = scale;
    ep.refq = use_q ? refq + r0 : nullptr; ep.ln_wq = use_q ? logf(wq) : 0.f; ep.use_q = use_q ? 1 : 0;
    ep.refk2 = refk2; ep.use_k = use_k ? 1 : 0; ep.include_diag = include_diag;
    MI_TRY(make_tmap_store32(&ep.tmap_p, P, rows, pitch, pitch));
    ep.lo_col0 = strict ? static_cast<int>(k_pad) : 0;
    ep.sum_part = nullptr; ep.rows_padded = 0;
    MI_TRY(launch_engine<mi::EpiPStore>(MapSpec{Qe.p + r0 * Qe.ld, rows, opnd_k_extent(Qe, D), Qe.ld},
                                        MapSpec{Ke.p, Bk, opnd_k_extent(Ke, D), Ke.ld}, sc, ep, stream));
    Bump none(nullptr, 0, false);
    // (2) Ok += alpha (P^T Q[panel] - gamma SUBk), contraction over the panel's rows; P read MN-major
    if (ok) {
      GemmArgs g;
      const int kr = static_cast<int>(cdiv(rows, bk()));
      g.a_mn = true;
      g.a = MapSpec{P, rows, pitch, pitch};            // map rows = K (panel rows), contiguous = M (columns of S)
      g.b_mn = true; g.b = MapSpec{Q.p + r0 * Q.ld, rows, q_hl ? Dp + D : D, Q.ld};
      g.M = Bk; g.N = D; g.seg_len = kr; g.k_blocks = kr;
      if (strict) {                                  // P_hi^T Q_hi + P_lo^T Q_hi (+ P_hi^T Q_lo)
        g.k_blocks = 2 * kr; g.a_moff[1] = static_cast<int>(k_pad);
        if (q_hl) { g.k_blocks = 3 * kr; g.b_noff[2] = static_cast<int>(Dp); }
      }
      g.alpha = alpha; g.gamma = gamma;
      g.accumulate = r0 > 0;
      if (gamma != 0.f) {                            // - gamma Q[k - q_offset] on this panel's own columns
        g.sub = Q.p + r0 * Q.ld; g.ld_sub = Q.ld;
        g.sub_lo = q_hl ? g.sub + Dp : nullptr;
        g.sub_row0 = q_offset + r0; g.sub_rows = rows;
      }
      g.out_f32 = ok->f32; g.ld_out = ok->ld;
      MI_TRY(run_gemm(g, none, stream));
      // the K-side output is complete after the last panel: let the caller start its reduce-scatter here
      if (ev_after_k != nullptr && r0 + panel_rows >= Bq) {
        MI_CUDA(cudaEventRecord(ev_after_k, stream));
        t_reserve_sms = g_overlap_reserve_sms.load(std::memory_order_relaxed);
      }
    }
    // (3) Oq[panel] = alpha (P V - gamma SUB), contraction over the Bk columns
    if (oq.f32 || oq.bf16) {
      GemmArgs g;
      g.a = MapSpec{P, rows, pitch, pitch};
      g.b_mn = true; g.b = MapSpec{K.p, Bk, k_hl ? Dp + D : D, K.ld};
      g.M = rows; g.N = D; g.seg_len = kp; g.k_blocks = kp;
      if (strict) {                                  // P_hi V_hi + P_lo V_hi (+ P_hi V_lo)
        g.k_blocks = 2 * kp; g.a_seg[1] = kp;
        if (k_hl) { g.k_blocks = 3 * kp; g.b_noff[2] = static_cast<int>(Dp); }
      }
      if (oq_ksplit > 1) {
        g.ksplit = oq_ksplit;
        g.out_f32 = oq_rawp; g.ld_out = D;
        Bump kws(kpart, kpart_elems * sizeof(float), false);
        const int st = run_gemm(g, kws, stream);
        t_reserve_sms = 0;
        MI_TRY(st);
        bf* o16 = oq.bf16 ? oq.bf16 + r0 * oq.ld16 : nullptr;
        finalize_q_kernel<<<blocks_capped(rows * D / 8, 256), 256, 0, stream>>>(
            oq_rawp, D, rows, nullptr, nullptr, nullptr, 0, alpha, gamma, K.p + (q_offset + r0) * K.ld, K.ld, k_hl ? 2 : 1, Dp,
            oq.f32 ? oq.f32 + r0 * oq.ld : nullptr, o16, (o16 && oq.split == 2) ? o16 + Dp : nullptr, oq.ld16, t_run_if);
        MI_LAUNCH_CHECK("finalize_q_kernel");
      } else {
      g.alpha = alpha; g.gamma = gamma;
      if (gamma != 0.f) {                            // - gamma K[q_offset + q]
        g.sub = K.p + (q_offset + r0) * K.ld; g.ld_sub = K.ld;
        g.sub_lo = k_hl ? g.sub + Dp : nullptr;
      }
      g.out_f32 = oq.f32 ? oq.f32 + r0 * oq.ld : nullptr; g.ld_out = oq.ld;
      g.out_bf16 = oq.bf16 ? oq.bf16 + r0 * oq.ld16 : nullptr; g.ld_out16 = oq.ld16;
      g.out_bf16_lo = (oq.bf16 && oq.split == 2) ? g.out_bf16 + Dp : nullptr;
      const int st = run_gemm(g, none, stream);
      t_reserve_sms = 0;
      MI_TRY(st);
      }
    }
  }
  return MI_OK;
}

// Optional tail of the single pass on ONE GPU: the loss is finalised as soon as the last panel's row sums are merged
// (the global log-sum-exp is then known on the device), so the last panel's K-side contraction can finish its output
// in the epilogue — Ok = alpha (kappa (Ok_raw) - gamma Q_diag) — instead of a separate read-modify-write pass over [Bk, D].
struct SingleFin {
  double* loss_out; float* lse_f; long long B; int estimator;     // loss_finalize_kernel arguments
  float alpha, gamma; int dv_like;
};

// The rows of Q may become available panel by panel (host-buffer entry point: the image embeddings are still crossing
// PCIe while the first panels are processed).  before_panel(r0, rows) enqueues on the stream whatever makes
// Q[r0, r0 + rows), ref[r0, ...) and diag[r0, ...) valid — and, for r0 == 0, lambda (any constant near the largest
// reference works, it only centres e^{ref - lambda}; later panels are guarded in sum_merge_kernel).
struct PanelFeed { std::function<int(long long, long long)> before_panel; };

// Single-pass form of the forward statistics + gradient pass (dv / infonce / row InfoNCE): ONE score computation.
// ref[q] (caller supplied: ref_sample_impl) is a per-row softmax reference; P~ = incl * e^{S - ref} is written without a
// statistics pass before it, and the same score tiles give (a) the exact row sums l_q = sum_k P~ (=> LSE_q = ref_q + ln l_q,
// the loss) and (b) the bf16 panel P~ whose two contractions, rescaled per row / globally afterwards, are the gradients:
//   dV-side   Oq_raw = P~ K                         final: alpha (c_q Oq_raw - gamma K_diag)
//   dQ-side   Ok_raw = sum_q P~[q,:]^T (w_q Q_q)    final: alpha (kappa Ok_raw - gamma Q_diag)
//   DV: c_q = e^{ref_q - LSE}, w_q = e^{ref_q - lambda}, kappa = e^{lambda - LSE};  row InfoNCE: c_q = w_q = 1/(B l_q), kappa = 1.
// 6 B^2 D executed = the algorithmic count.  Any reference is mathematically valid; flag_out counts the rows whose
// reference left the numerically safe window (see sum_merge_kernel) — the caller then repeats with exact references.
int single_pass_impl(const Opnd& Q, const Opnd& K, const int* sid_q, const int* sid_k,
                     long long q_offset, long long Bq, long long Bk, long long D, float scale,
                     int include_diag, int precision, float inv_bg,
                     const float* ref, const float* lambda, const float* diag,
                     float* row_out, float* oq_raw, float* ok_raw, float* wrow, int* flag_out, Bump& ws, cudaStream_t stream,
                     cudaEvent_t ev_after_k = nullptr, double* scal_out = nullptr, cudaEvent_t ev_after_scal = nullptr,
                     cudaEvent_t ev_k_ready = nullptr, const struct SingleFin* fin = nullptr,
                     const struct PanelFeed* feed = nullptr, bool k_local_valid = false,
                     const MaskBuf* shared_mask = nullptr /* the negatives mask of (sid_q, sid_k), built by the caller */,
                     cudaEvent_t ev_lambda = nullptr /* lambda (an all-reduce in flight) is valid once this event fires: waited for
                                                        right before the first row-sum merge, after the score tiles are enqueued */,
                     bool defer_reduce = false /* do not reduce row_out -> scal_out here: ev_after_scal fires right after the last
                                                  row-sum merge and the CALLER reduces (reduce_rows + flag_to_scal) on another
                                                  stream, so the contractions start without waiting for it */) {
  if (Bq <= 0 || Bk <= 0 || D <= 0 || (D % 8) != 0) return MI_ERR_BAD_ARG;
  typedef __nv_bfloat16 bf;
  const bool strict = (precision & 1) == MI_PREC_BF16_STRICT;
  const int n_ntile = static_cast<int>(cdiv(Bk, mi::TILE_N));
  const long long k_pad = static_cast<long long>(n_ntile) * mi::TILE_N;
  const int kp = static_cast<int>(k_pad / bk());
  const long long pitch = k_pad * (strict ? 2 : 1);
  const long long Dp = round_up(D, kSplitAlign);
  const bool k_hl = strict && K.split == 2;
  const long long mb_panel = panel_mblks(Bq, Bk, D, precision & 1);
  const long long panel_rows = mb_panel * rows_per_mblk();
  const int max_split = n_ntile;
  const MaskBuf mb = shared_mask != nullptr ? *shared_mask : take_mask(ws, Bq, k_pad, Bk);
  const long long ld_qs = strict ? 2 * Dp : D;               // w Q [panel_rows, hi | lo]
  bf* Qs = ok_raw || ws.dry ? ws.take<bf>(static_cast<size_t>(panel_rows) * ld_qs) : nullptr;
  bf* P = ws.take<bf>(static_cast<size_t>(panel_rows) * pitch);
  // (x3: the first panel may be written by up to three launches — own columns first, the rest once K has arrived)
  const size_t part_slices = static_cast<size_t>(max_split > 64 ? 64 : max_split) * mi::kColQuarters;
  float* part = ws.take<float>(3 * part_slices * panel_rows);
  const RedScratch red = take_red(ws);
  const int oq_ksplit = strict ? strict_ksplit(kp * (k_hl ? 3 : 2)) : 1;     // see kStrictChainBlocks
  const size_t kpart_elems = oq_ksplit > 1 ? static_cast<size_t>(oq_ksplit) * panel_rows * round_up(D, 4) : 0;
  float* kpart = oq_ksplit > 1 ? ws.take<float>(kpart_elems) : nullptr;
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (ws.dry) return MI_OK;
  if (!Q.p || !K.p || !sid_q || !sid_k || !ref || !diag || !row_out || !oq_raw || !wrow || !flag_out || !(scale > 0.f) ||
      (!include_diag && !lambda))
    return MI_ERR_BAD_ARG;
  const int* pr = t_run_if;

  if (shared_mask == nullptr) MI_TRY(build_mask(mb, sid_q, sid_k, Bq, Bk, k_pad, stream));
  const Opnd Qe{Q.p, Q.ld, strict ? Q.split : 1}, Ke{K.p, K.ld, strict ? K.split : 1};
  // from here on the K rows are read: wait for the caller's "K complete" event (the all-gather of the text embeddings).
  // When the caller vouches for this rank's own rows (k_local_valid) the wait moves further down: the score tiles of the
  // own column block need nothing else, so they run under the all-gather.
  const long long own_t0 = q_offset / mi::TILE_N, own_t1 = (q_offset + Bq) / mi::TILE_N;
  const bool own_first = ev_k_ready != nullptr && k_local_valid && feed == nullptr &&
                         (q_offset % mi::TILE_N) == 0 && (Bq % mi::TILE_N) == 0 && Bq < Bk;
  if (ev_k_ready != nullptr && !own_first) MI_CUDA(cudaStreamWaitEvent(stream, ev_k_ready, 0));

  for (long long r0 = 0; r0 < Bq; r0 += panel_rows) {
    const long long rows = (Bq - r0 < panel_rows) ? (Bq - r0) : panel_rows;
    if (feed != nullptr) MI_TRY(feed->before_panel(r0, rows));     // this panel's Q rows, references and diag arrive now
    // (1) score tiles -> P~ panel + row sums; a launch covers the N tiles [t0, t1) and appends its partial row sums
    const int n_mblk_p = static_cast<int>(cdiv(rows, rows_per_mblk()));
    const int rows_padded = n_mblk_p * rows_per_mblk();
    int n_part = 0;
    auto score_tiles = [&](long long t0, long long t1) -> int {
      if (t1 <= t0) return MI_OK;
      Sched sc;
      sc.n_mblk = n_mblk_p;
      sc.n_ntile = static_cast<int>(t1 - t0);
      sc.n_split = choose_split(sc.n_mblk, sc.n_ntile, num_pairs());
      if (sc.n_split > 64) sc.n_split = 64;
      sc.n_ksplit = 1; sc.order = 0;
      MI_TRY(score_segments(sc, Qe, Ke, D));
      sc.nt_base = static_cast<int>(t0);
      mi::EpiPStore::Params ep;
      ep.mask = mi::MaskInfo{mb.excl + r0, mb.n_same + r0, sid_q + r0, mb.sidk_pad};
      ep.q_rows = static_cast<int>(rows); ep.k_cols = static_cast<int>(Bk);
      ep.q_offset = q_offset + r0; ep.scale = scale;
      ep.refq = ref + r0; ep.ln_wq = 0.f; ep.use_q = 1;
      ep.refk2 = nullptr; ep.use_k = 0; ep.include_diag = include_diag;
      MI_TRY(make_tmap_store32(&ep.tmap_p, P, rows, pitch, pitch));
      ep.lo_col0 = strict ? static_cast<int>(k_pad) : 0;
      ep.sum_part = part + static_cast<size_t>(n_part) * rows_padded; ep.rows_padded = rows_padded;
      MI_TRY(launch_engine<mi::EpiPStore>(MapSpec{Qe.p + r0 * Qe.ld, rows, opnd_k_extent(Qe, D), Qe.ld},
                                          MapSpec{Ke.p, Bk, opnd_k_extent(Ke, D), Ke.ld}, sc, ep, stream));
      n_part += sc.n_split * mi::kColQuarters;
      return MI_OK;
    };
    if (own_first && r0 == 0) {
      MI_TRY(score_tiles(own_t0, own_t1));                               // this rank's own columns: K rows already here
      MI_CUDA(cudaStreamWaitEvent(stream, ev_k_ready, 0));               // the other ranks' text embeddings
      MI_TRY(score_tiles(0, own_t0));
      MI_TRY(score_tiles(own_t1, n_ntile));
    } else {
      MI_TRY(score_tiles(0, n_ntile));
    }
    if (ev_lambda != nullptr && r0 == 0) MI_CUDA(cudaStreamWaitEvent(stream, ev_lambda, 0));
    sum_merge_kernel<<<blocks_for(rows, 128), 128, 0, stream>>>(part, n_part, rows_padded, static_cast<int>(rows),
                                                                ref + r0, lambda, mb.n_same + r0, static_cast<int>(Bk), diag + r0,
                                                                include_diag, inv_bg, reinterpret_cast<float4*>(row_out) + r0,
                                                                wrow + r0, flag_out, pr);
    MI_LAUNCH_CHECK("sum_merge_kernel");
    if (defer_reduce && r0 + panel_rows >= Bq) {
      if (ev_after_scal != nullptr) MI_CUDA(cudaEventRecord(ev_after_scal, stream));
    } else if (scal_out != nullptr && r0 + panel_rows >= Bq) {
      // every row's statistics are final once the last panel's sums are merged: reduce them NOW (before the two
      // contractions of this panel) so a caller can exchange the scalars of the loss while the GEMMs still run
      MI_TRY(reduce_rows(row_out, Bq, scal_out, red, stream));
      flag_to_scal_kernel<<<1, 1, 0, stream>>>(flag_out, scal_out, pr);
      MI_LAUNCH_CHECK("flag_to_scal_kernel");
      if (ev_after_scal != nullptr) MI_CUDA(cudaEventRecord(ev_after_scal, stream));
      if (fin != nullptr) {
        loss_finalize_kernel<<<1, 32, 0, stream>>>(scal_out, nullptr, fin->B, fin->estimator, fin->loss_out, fin->lse_f,
                                                   fin->dv_like ? lambda : nullptr, pr);
        MI_LAUNCH_CHECK("loss_finalize_kernel");
      }
    }
    Bump none(nullptr, 0, false);
    // (2) Ok_raw += P~^T (w Q)[panel]: contraction over the panel rows, P~ read MN-major
    if (ok_raw) {
      scale_rows_kernel<<<blocks_capped(rows * D / 8, 256), 256, 0, stream>>>(Q.p + r0 * Q.ld, Q.ld, Q.split, Dp, wrow + r0, Qs,
                                                                          strict ? Qs + Dp : nullptr, ld_qs, rows, D, pr);
      MI_LAUNCH_CHECK("scale_rows_kernel");
      GemmArgs g;
      const int kr = static_cast<int>(cdiv(rows, bk()));
      g.a_mn = true;
      g.a = MapSpec{P, rows, pitch, pitch};
      g.b_mn = true; g.b = MapSpec{Qs, rows, strict ? Dp + D : D, ld_qs};
      g.M = Bk; g.N = D; g.seg_len = kr; g.k_blocks = kr;
      if (strict) {                                  // P_hi^T Q_hi + P_lo^T Q_hi + P_hi^T Q_lo
        g.k_blocks = 3 * kr; g.a_moff[1] = static_cast<int>(k_pad);
        g.b_noff[2] = static_cast<int>(Dp);
      }
      g.accumulate = r0 > 0;
      g.out_f32 = ok_raw; g.ld_out = D;
      if (fin != nullptr && scal_out != nullptr && r0 + panel_rows >= Bq) {      // last panel: finish the K-side output here
        g.acc_first = true;
        if (fin->dv_like) { g.kappa_a = lambda; g.kappa_b = fin->lse_f; }
        g.alpha = fin->alpha; g.gamma = fin->gamma;
        g.sub = Q.p; g.ld_sub = Q.ld; g.sub_lo = (strict && Q.split == 2) ? Q.p + Dp : nullptr;
        g.sub_row0 = q_offset; g.sub_rows = Bq;
      }
      MI_TRY(run_gemm(g, none, stream));
      if (ev_after_k != nullptr && r0 + panel_rows >= Bq) {
        MI_CUDA(cudaEventRecord(ev_after_k, stream));
        t_reserve_sms = g_overlap_reserve_sms.load(std::memory_order_relaxed);   // the caller's collective starts here
      }
    }
    // (3) Oq_raw[panel] = P~ K
    {
      GemmArgs g;
      g.a = MapSpec{P, rows, pitch, pitch};
      g.b_mn = true; g.b = MapSpec{K.p, Bk, k_hl ? Dp + D : D, K.ld};
      g.M = rows; g.N = D; g.seg_len = kp; g.k_blocks = kp;
      if (strict) {
        g.k_blocks = 2 * kp; g.a_seg[1] = kp;
        if (k_hl) { g.k_blocks = 3 * kp; g.b_noff[2] = static_cast<int>(Dp); }
      }
      g.out_f32 = oq_raw + r0 * D; g.ld_out = D;
      g.ksplit = oq_ksplit;
      Bump kws(kpart, kpart_elems * sizeof(float), false);
      const int st = run_gemm(g, oq_ksplit > 1 ? kws : none, stream);
      t_reserve_sms = 0;
      MI_TRY(st);
    }
  }
  return MI_OK;
}

// Jensen-Shannon on one GPU (square batch, row q pairs with column q): per row panel ONE score computation (EpiJS) writes
// P = M sigma(S) and the row sums of M softplus(S) (-> row_out in js_rows_kernel's layout, scal_out after the last panel);
// the two contractions give the RAW gradients  oq_raw = P K  and  ok_raw = P^T Q  (accumulated over the panels).  The
// weight 1/N_neg and the positive terms are applied by js_finalize_kernel once N_neg is known.  oq_raw == ok_raw == nullptr:
// the statistics only (EpiJS<false>, no panel).  diag[q] = S[q, q]; with `feed` it is valid for a panel after before_panel.
int js_pass_impl(const Opnd& Q, const Opnd& K, const int* sid, long long B, long long D, float scale, int precision,
                 const float* diag, float* row_out, double* scal_out, float* oq_raw, float* ok_raw, const MaskBuf& mb,
                 Bump& ws, cudaStream_t stream, const PanelFeed* feed = nullptr) {
  if (B <= 0 || D <= 0 || (D % 8) != 0) return MI_ERR_BAD_ARG;
  typedef __nv_bfloat16 bf;
  const bool strict = (precision & 1) == MI_PREC_BF16_STRICT;
  const bool grads = oq_raw != nullptr || ok_raw != nullptr || ws.dry;
  const int n_ntile = static_cast<int>(cdiv(B, mi::TILE_N));
  const long long k_pad = static_cast<long long>(n_ntile) * mi::TILE_N;
  const int kp = static_cast<int>(k_pad / bk());
  const long long pitch = k_pad * (strict ? 2 : 1);
  const long long Dp = round_up(D, kSplitAlign);
  const bool k_hl = strict && K.split == 2, q_hl = strict && Q.split == 2;
  const long long panel_rows = panel_mblks(B, B, D, precision & 1) * rows_per_mblk();
  bf* P = grads ? ws.take<bf>(static_cast<size_t>(panel_rows) * pitch) : nullptr;
  const size_t part_slices = static_cast<size_t>(n_ntile > 64 ? 64 : n_ntile) * mi::kColQuarters;
  float* part = ws.take<float>(part_slices * panel_rows);
  const int oq_ksplit = strict ? strict_ksplit(kp * (k_hl ? 3 : 2)) : 1;     // see kStrictChainBlocks
  const size_t kpart_elems = (grads && oq_ksplit > 1) ? static_cast<size_t>(oq_ksplit) * panel_rows * round_up(D, 4) : 0;
  float* kpart = kpart_elems ? ws.take<float>(kpart_elems) : nullptr;
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (ws.dry) return MI_OK;
  if (!Q.p || !K.p || !sid || !diag || !row_out || !scal_out || !(scale > 0.f)) return MI_ERR_BAD_ARG;
  const Opnd Qe{Q.p, Q.ld, strict ? Q.split : 1}, Ke{K.p, K.ld, strict ? K.split : 1};
  Bump none(nullptr, 0, false);
  for (long long r0 = 0; r0 < B; r0 += panel_rows) {
    const long long rows = (B - r0 < panel_rows) ? (B - r0) : panel_rows;
    if (feed != nullptr) MI_TRY(feed->before_panel(r0, rows));
    // (1) score tiles -> P panel + partial row sums of softplus
    Sched sc;
    sc.n_mblk = static_cast<int>(cdiv(rows, rows_per_mblk()));
    sc.n_ntile = n_ntile;
    sc.n_split = choose_split(sc.n_mblk, sc.n_ntile, num_pairs());
    if (sc.n_split > 64) sc.n_split = 64;
    sc.n_ksplit = 1; sc.order = 0;
    MI_TRY(score_segments(sc, Qe, Ke, D));
    const int rows_padded = sc.n_mblk * rows_per_mblk();
    mi::EpiPStore::Params ep;
    ep.mask = mi::MaskInfo{mb.excl + r0, mb.n_same + r0, sid + r0, mb.sidk_pad};
    ep.q_rows = static_cast<int>(rows); ep.k_cols = static_cast<int>(B);
    ep.q_offset = r0; ep.scale = scale;
    ep.refq = nullptr; ep.ln_wq = 0.f; ep.use_q = 0; ep.refk2 = nullptr; ep.use_k = 0; ep.include_diag = 0;
    ep.lo_col0 = strict ? static_cast<int>(k_pad) : 0;
    ep.sum_part = part; ep.rows_padded = rows_padded;
    const MapSpec ma{Qe.p + r0 * Qe.ld, rows, opnd_k_extent(Qe, D), Qe.ld}, mbk{Ke.p, B, opnd_k_extent(Ke, D), Ke.ld};
    if (grads) {
      MI_TRY(make_tmap_store32(&ep.tmap_p, P, rows, pitch, pitch));
      MI_TRY(launch_engine<mi::EpiJS<true>>(ma, mbk, sc, ep, stream));
    } else {
      std::memset(&ep.tmap_p, 0, sizeof(ep.tmap_p));
      MI_TRY(launch_engine<mi::EpiJS<false>>(ma, mbk, sc, ep, stream));
    }
    js_rows_kernel<<<blocks_for(rows, 128), 128, 0, stream>>>(part, sc.n_split * mi::kColQuarters, rows_padded, static_cast<int>(rows),
                                                              mb.n_same + r0, static_cast<int>(B), diag + r0,
                                                              reinterpret_cast<float4*>(row_out) + r0);
    MI_LAUNCH_CHECK("js_rows_kernel");
    if (r0 + panel_rows >= B) {
      js_reduce_kernel<<<1, kJsRedThreads, 0, stream>>>(reinterpret_cast<const float4*>(row_out), B, scal_out);
      MI_LAUNCH_CHECK("js_reduce_kernel");
    }
    if (!grads) continue;
    // (2) ok_raw += P^T Q[panel]: contraction over the panel rows, P read MN-major
    if (ok_raw) {
      GemmArgs g;
      const int kr = static_cast<int>(cdiv(rows, bk()));
      g.a_mn = true;
      g.a = MapSpec{P, rows, pitch, pitch};
      g.b_mn = true; g.b = MapSpec{Q.p + r0 * Q.ld, rows, q_hl ? Dp + D : D, Q.ld};
      g.M = B; g.N = D; g.seg_len = kr; g.k_blocks = kr;
      if (strict) {                                  // P_hi^T Q_hi + P_lo^T Q_hi (+ P_hi^T Q_lo)
        g.k_blocks = 2 * kr; g.a_moff[1] = static_cast<int>(k_pad);
        if (q_hl) { g.k_blocks = 3 * kr; g.b_noff[2] = static_cast<int>(Dp); }
      }
      g.accumulate = r0 > 0;
      g.out_f32 = ok_raw; g.ld_out = D;
      MI_TRY(run_gemm(g, none, stream));
    }
    // (3) oq_raw[panel] = P K
    if (oq_raw) {
      GemmArgs g;
      g.a = MapSpec{P, rows, pitch, pitch};
      g.b_mn = true; g.b = MapSpec{K.p, B, k_hl ? Dp + D : D, K.ld};
      g.M = rows; g.N = D; g.seg_len = kp; g.k_blocks = kp;
      if (strict) {
        g.k_blocks = 2 * kp; g.a_seg[1] = kp;
        if (k_hl) { g.k_blocks = 3 * kp; g.b_noff[2] = static_cast<int>(Dp); }
      }
      g.out_f32 = oq_raw + r0 * D; g.ld_out = D;
      g.ksplit = oq_ksplit;
      Bump kws(kpart, kpart_elems * sizeof(float), false);
      MI_TRY(run_gemm(g, oq_ksplit > 1 ? kws : none, stream));
    }
  }
  return MI_OK;
}

inline bool single_pass_estimator(int estimator, int precision) {
  return estimator != MI_EST_INFONCE_SYM && (precision & MI_PREC_TWO_PASS) == 0;
}

// How critic_impl deals with a tripped single-pass guard (loss_out[7] != 0 after the sampled-reference pass):
//   predicated: the exact repeat (references from EVERY column) is enqueued behind a device flag — a few empty launches
//               when the guard stayed clear; fully asynchronous and CUDA-graph capturable (the device-pointer ABI);
//   host:       nothing is enqueued; the caller reads loss_out[7] and repeats with MI_PREC_TWO_PASS (the host-buffer ABI,
//               which synchronises anyway).
struct Fallback { bool predicated = true; };

int critic_impl(const void* X_, const void* Y_, const void* W_, const int* sid, long long B, long long D,
                int critic, int estimator, int precision, float inv_tau,
                double* loss_out, float* dX, float* dY, float* dW, Bump& ws, cudaStream_t stream,
                cudaEvent_t ev_dy_final = nullptr, bool* ev_recorded = nullptr,     // event recorded once dY is final (the
                                                                                     // dT / dX / dW work follows it)
                const std::function<int(long long, long long)>* x_ready = nullptr,  // single pass only: X rows arrive per panel
                const Fallback& fb = Fallback()) {
  if (B <= 0 || D <= 0 || (D % 8) != 0) return MI_ERR_BAD_ARG;
  if (estimator < MI_EST_DV || estimator > MI_EST_NWJ) return MI_ERR_BAD_ARG;
  typedef __nv_bfloat16 bf;
  const bf* X = static_cast<const bf*>(X_); const bf* Y = static_cast<const bf*>(Y_); const bf* W = static_cast<const bf*>(W_);
  const bool bilinear = critic == MI_CRITIC_BILINEAR;
  const bool grads = dX != nullptr || dY != nullptr || dW != nullptr;
  const bool plan = ws.dry || grads;
  const bool sym = estimator == MI_EST_INFONCE_SYM;
  const bool js = estimator == MI_EST_JS;           // its own pass (js_pass_impl): no references, no guard
  // NWJ is DV with another final scalar (see loss_finalize_kernel): the same passes, references and guard
  const bool dv_like = estimator == MI_EST_DV || estimator == MI_EST_INFONCE_REF || estimator == MI_EST_NWJ;
  const bool strict = (precision & 1) == MI_PREC_BF16_STRICT;
  // one score computation instead of two (see single_pass_impl); the symmetric estimator needs exact column statistics
  // before its gradient pass and stays on the statistics-pass + gradient-pass path.  MI_PREC_TWO_PASS asks for exact
  // references (stride 1) in the single pass: the same statistics, then the pass can never trip its guard.
  const bool single = !sym && !js && (grads || ws.dry);
  const bool js_grads = js && plan;
  const bool exact_refs = (precision & MI_PREC_TWO_PASS) != 0;
  const int tsplit = (bilinear && strict) ? 2 : 1;        // T = X W kept as a hi/lo bf16 pair in strict mode
  const long long Dp = round_up(D, kSplitAlign);
  const long long ldT = tsplit == 2 ? 2 * Dp : D;
  bf* T = bilinear ? ws.take<bf>(static_cast<size_t>(B) * ldT) : nullptr;
  float* rows_r = ws.take<float>(static_cast<size_t>(B) * 4);
  float* rows_c = sym ? ws.take<float>(static_cast<size_t>(B) * 4) : nullptr;
  double* scal_r = ws.take<double>(8);
  double* scal_c = sym ? ws.take<double>(8) : nullptr;
  float* lse_f = ws.take<float>(1);
  float* ref_r = ws.take<float>(B);
  float* ref_c = sym ? ws.take<float>(B) : nullptr;
  bf* dT16 = (bilinear && plan) ? ws.take<bf>(static_cast<size_t>(B) * ldT) : nullptr;
  float* sp_diag = (single || js) ? ws.take<float>(B) : nullptr;
  float* sp_wrow = single ? ws.take<float>(B) : nullptr;
  float* sp_lambda = single ? ws.take<float>(1) : nullptr;
  int* sp_flags = single ? ws.take<int>(4) : nullptr;     // [0] rows tripped (sampled pass), [1] fallback predicate, [2] rows tripped (repeat)
  double* sp_guard = single ? ws.take<double>(1) : nullptr;
  float* sp_oq = ((single || js_grads) && (bilinear || !dX)) ? ws.take<float>(static_cast<size_t>(B) * D) : nullptr;   // dot: dX doubles as the raw buffer
  float* sp_ok = ((single || js_grads) && !dY) ? ws.take<float>(static_cast<size_t>(B) * D) : nullptr;
  // the negatives mask of the whole batch: built ONCE per call and shared by the exact reference pass and the single pass(es)
  const long long k_pad_all = cdiv(B, mi::TILE_N) * mi::TILE_N;
  MaskBuf all_mask{};
  if (single || js) all_mask = take_mask(ws, B, k_pad_all, B);
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  if (!ws.dry && (!X || !Y || !sid || !loss_out || (bilinear && !W))) return MI_ERR_BAD_ARG;

  const Opnd Xo{X, D, 1}, Yo{Y, D, 1};
  const Opnd To = bilinear ? Opnd{T, ldT, tsplit} : Xo;
  size_t mk = ws.mark();
  const bool streamed = x_ready != nullptr && (single || js_grads) && !ws.dry;
  Bump none(nullptr, 0, false);
  // T[r0 : r0 + rows] = X[r0 : r0 + rows] W  (B operand of the engine is [N, K] = W^T: W itself read MN-major)
  auto project = [&](long long r0, long long rows, Bump& w) -> int {
    GemmArgs g;
    g.a = MapSpec{X + r0 * D, rows, D, D};
    g.b_mn = true; g.b = MapSpec{W, D, D, D};
    g.M = rows; g.N = D; g.k_blocks = static_cast<int>(cdiv(D, bk()));
    g.out_bf16 = T + r0 * ldT; g.ld_out16 = ldT; g.out_bf16_lo = tsplit == 2 ? T + r0 * ldT + Dp : nullptr;
    return run_gemm(g, w, stream);
  };
  if (bilinear) {
    if (!ws.dry && tsplit == 2) {        // zero the gap columns between the hi and lo halves once
      MI_CUDA(cudaMemsetAsync(T, 0, static_cast<size_t>(B) * ldT * sizeof(bf), stream));
      if (dT16) MI_CUDA(cudaMemsetAsync(dT16, 0, static_cast<size_t>(B) * ldT * sizeof(bf), stream));
    }
    if (!streamed) {                     // (streamed: projected panel by panel inside the pass, see PanelFeed)
      if (!ws.dry) MI_TRY(project(0, B, ws));
    }
  }
  if (single) {
    const int incl = dv_like ? 0 : 1;
    const float gam = 1.f / static_cast<float>(B);
    float* oq_raw = sp_oq ? sp_oq : dX;
    float* ok_raw = dY ? dY : sp_ok;
    // the loss is finalised inside the pass and, when dY is wanted, the last panel's contraction finishes dY in its epilogue
    SingleFin fin{loss_out, lse_f, B, estimator, inv_tau, gam, dv_like ? 1 : 0};
    const bool fused_k = dY != nullptr;
    const long long stride0 = exact_refs ? 1 : ref_stride_auto(B, B, D);
    const long long panel_rows = panel_mblks(B, B, D, precision & 1) * rows_per_mblk();
    // one complete pass: references (column sample of the given stride) -> score tiles / statistics / both contractions
    // -> loss and dT.  `flag` counts the rows that tripped the guard of THIS pass.
    if (!ws.dry) MI_TRY(build_mask(all_mask, sid, sid, B, B, k_pad_all, stream));
    auto run_pass = [&](long long stride, int* flag, bool feed_x) -> int {
      if (!ws.dry) MI_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), stream));
      PanelFeed feed;
      if (feed_x) {
        feed.before_panel = [&, stride](long long r0, long long rows) -> int {
          MI_TRY((*x_ready)(r0, rows));
          if (bilinear) MI_TRY(project(r0, rows, none));
          const Opnd Tp{To.p + r0 * To.ld, To.ld, To.split};
          const size_t m2 = ws.mark();
          MI_TRY(ref_sample_impl(Tp, Yo, sid + r0, sid, r0, rows, B, D, inv_tau, incl, 0, B, stride, stride > 1 ? kRefMargin : 0.f,
                                 ref_r + r0, sp_diag + r0, r0 == 0 ? sp_lambda : nullptr, ws, stream));
          ws.release(m2);
          return MI_OK;
        };
      } else {
        MI_TRY(ref_sample_impl(To, Yo, sid, sid, 0, B, B, D, inv_tau, incl, 0, B, stride, stride > 1 ? kRefMargin : 0.f,
                               ref_r, sp_diag, sp_lambda, ws, stream, stride == 1 ? &all_mask : nullptr));
        ws.release(mk);
      }
      MI_TRY(single_pass_impl(To, Yo, sid, sid, 0, B, B, D, inv_tau, incl, precision, gam, ref_r, sp_lambda, sp_diag,
                              rows_r, oq_raw, ok_raw, sp_wrow, flag, ws, stream,
                              fused_k ? ev_dy_final : nullptr, scal_r, nullptr, nullptr, fused_k ? &fin : nullptr,
                              feed_x ? &feed : nullptr, false, &all_mask));
      if (ws.dry) {                      // the per-panel reference sample of the streamed form lives on top of the pass
        const size_t m2 = ws.mark();
        MI_TRY(ref_sample_impl(To, Yo, sid, sid, 0, panel_rows < B ? panel_rows : B, B, D, inv_tau, incl, 0, B, stride, 0.f,
                               ref_r, sp_diag, sp_lambda, ws, stream));
        ws.release(m2);
      }
      ws.release(mk);
      if (ws.dry) return MI_OK;
      if (!fused_k) {
        loss_finalize_kernel<<<1, 32, 0, stream>>>(scal_r, nullptr, B, estimator, loss_out, lse_f, dv_like ? sp_lambda : nullptr, t_run_if);
        MI_LAUNCH_CHECK("loss_finalize_kernel");
      }
      // dT = inv_tau (c G~ Y - Y/B): fp32 (dot critic: this is dX) or the bf16 (hi/lo) operand of the dX / dW GEMMs
      finalize_q_kernel<<<blocks_capped(B * D / 8, 256), 256, 0, stream>>>(oq_raw, D, B, ref_r, sp_wrow, lse_f, dv_like ? 1 : 0, inv_tau, gam,
                                                                        Y, D, 1, Dp, bilinear ? nullptr : dX, bilinear ? dT16 : nullptr,
                                                                        (bilinear && tsplit == 2) ? dT16 + Dp : nullptr, ldT, t_run_if);
      MI_LAUNCH_CHECK("finalize_q_kernel");
      // (dY was finished by the last panel's contraction: see SingleFin)
      return MI_OK;
    };
    MI_TRY(run_pass(stride0, sp_flags, streamed));
    if (fused_k && ev_dy_final && ev_recorded && !ws.dry) *ev_recorded = true;
    if (!ws.dry && stride0 > 1) {
      if (fb.predicated) {
        guard_to_flag_kernel<<<1, 1, 0, stream>>>(loss_out, sp_flags + 1, sp_guard);
        MI_LAUNCH_CHECK("guard_to_flag_kernel");
        {
          PredGuard pg(sp_flags + 1);
          MI_TRY(run_pass(1, sp_flags + 2, false));
        }
        guard_report_kernel<<<1, 1, 0, stream>>>(sp_flags + 1, sp_guard, loss_out);
        MI_LAUNCH_CHECK("guard_report_kernel");
      }
    } else if (ws.dry && stride0 > 1) {
      MI_TRY(run_pass(1, sp_flags, false));
    }
  }
  if (js) {
    if (!ws.dry) MI_TRY(build_mask(all_mask, sid, sid, B, B, k_pad_all, stream));
    // S_ii: one O(B D) row-dot kernel (per panel when the image embeddings arrive panel by panel)
    auto diag_rows = [&](long long r0, long long rows) -> int {
      diag_kernel<<<blocks_for(rows * 32, 256), 256, 0, stream>>>(To.p + r0 * To.ld, To.ld, To.split, Y, D, 1, r0, rows, D, Dp,
                                                                   inv_tau, sp_diag + r0, nullptr);
      MI_LAUNCH_CHECK("diag_kernel");
      return MI_OK;
    };
    PanelFeed feed;
    if (streamed) {
      feed.before_panel = [&](long long r0, long long rows) -> int {
        MI_TRY((*x_ready)(r0, rows));
        if (bilinear) MI_TRY(project(r0, rows, none));
        return diag_rows(r0, rows);
      };
    } else if (!ws.dry) {
      MI_TRY(diag_rows(0, B));
    }
    float* oq_raw = js_grads ? (sp_oq ? sp_oq : dX) : nullptr;
    float* ok_raw = js_grads ? (dY ? dY : sp_ok) : nullptr;
    MI_TRY(js_pass_impl(To, Yo, sid, B, D, inv_tau, precision, sp_diag, rows_r, scal_r, oq_raw, ok_raw, all_mask, ws, stream,
                        streamed ? &feed : nullptr));
    ws.release(mk);
    if (!ws.dry) {
      loss_finalize_kernel<<<1, 32, 0, stream>>>(scal_r, nullptr, B, estimator, loss_out, lse_f, nullptr, nullptr);   // lse_f = 1 / N_neg
      MI_LAUNCH_CHECK("loss_finalize_kernel");
    }
    if (!ws.dry && js_grads) {
      const float inv_b = 1.f / static_cast<float>(B);
      // dY = inv_tau (P^T T / N_neg - sigma(-S_kk) T_k / B), in place
      if (dY) {
        js_finalize_kernel<<<blocks_capped(B * D / 8, 256), 256, 0, stream>>>(dY, D, B, lse_f, sp_diag, inv_b, inv_tau, To.p, To.ld,
                                                                            To.split, Dp, dY, nullptr, nullptr, 0);
        MI_LAUNCH_CHECK("js_finalize_kernel");
        if (ev_dy_final) {
          MI_CUDA(cudaEventRecord(ev_dy_final, stream));
          if (ev_recorded) *ev_recorded = true;
        }
      }
      // dT = inv_tau (P Y / N_neg - sigma(-S_qq) Y_q / B): fp32 (dot critic: this is dX) or the bf16 (hi/lo) operand of dX / dW
      if (bilinear ? (dX || dW) : dX != nullptr) js_finalize_kernel<<<blocks_capped(B * D / 8, 256), 256, 0, stream>>>(oq_raw, D, B, lse_f, sp_diag, inv_b, inv_tau, Y, D, 1, Dp,
                                                                          bilinear ? nullptr : dX, bilinear ? dT16 : nullptr,
                                                                          (bilinear && tsplit == 2) ? dT16 + Dp : nullptr, ldT);
      MI_LAUNCH_CHECK("js_finalize_kernel");
    }
  }
  if ((!single || ws.dry) && !js) {        // statistics pass(es) + gradient pass with exact references (planning covers both paths)
    if (sym) {      // rows and columns from one score computation
      MI_TRY(stats_rc_impl(To, Yo, sid, sid, 0, B, B, D, inv_tau, rows_r, scal_r, rows_c, scal_c, nullptr, ws, stream));
    } else {
      MI_TRY(stats_impl(To, Yo, sid, sid, 0, B, B, D, inv_tau, rows_r, scal_r, ws, stream));
    }
    ws.release(mk);
    if (!ws.dry) {
      loss_finalize_kernel<<<1, 32, 0, stream>>>(scal_r, scal_c, B, estimator, loss_out, lse_f, nullptr, nullptr);
      MI_LAUNCH_CHECK("loss_finalize_kernel");
    }
    if (!plan) return MI_OK;

    if (!ws.dry) {
      if (dv_like) make_ref_kernel<<<blocks_for(B, 256), 256, 0, stream>>>(ref_r, nullptr, 0, lse_f, B);
      else make_ref_kernel<<<blocks_for(B, 256), 256, 0, stream>>>(ref_r, reinterpret_cast<const float4*>(rows_r), 3, nullptr, B);
      MI_LAUNCH_CHECK("make_ref_kernel");
      if (sym) {
        make_ref_kernel<<<blocks_for(B, 256), 256, 0, stream>>>(ref_c, reinterpret_cast<const float4*>(rows_c), 3, nullptr, B);
        MI_LAUNCH_CHECK("make_ref_kernel");
      }
    }
    // G = incl (wq e^{S - refq[row]} + wk e^{S - refk[col]}):  DV: e^{S - LSE} on the negatives;
    // InfoNCE row: (1/B) e^{S - r_i};  symmetric: (1/2B)(e^{S - r_i} + e^{S - c_j}); positives included.
    float wq = 1.f, wk = 0.f;
    const float* refq = ref_r; const float* refk = nullptr;
    if (estimator == MI_EST_INFONCE_ROW) { wq = 1.f / B; }
    else if (sym) { wq = 0.5f / B; wk = 0.5f / B; refk = ref_c; }
    const int incl_diag = dv_like ? 0 : 1;
    const float gamma = 1.f / static_cast<float>(B);

    // one pass: dT = inv_tau (G Y - Y/B)  and  dY = inv_tau (G^T T - T/B)
    GradOut oq, okk;
    if (bilinear) { oq.bf16 = dT16; oq.ld16 = ldT; oq.split = tsplit; }
    else { oq.f32 = dX; oq.ld = D; }
    okk.f32 = dY; okk.ld = D;
    const bool want_q = bilinear ? (dX || dW || ws.dry) : (dX || ws.dry);
    const bool want_k = dY || ws.dry;
    GradOut oq_none;
    if (want_q || want_k) {
      MI_TRY(grad_impl(To, Yo, sid, sid, 0, B, B, D, inv_tau, refq, wq, refk, wk, incl_diag, precision & 1,
                       inv_tau, gamma, want_q ? oq : oq_none, want_k ? &okk : nullptr, ws, stream, want_k ? ev_dy_final : nullptr));
      if (want_k && ev_dy_final && ev_recorded && !ws.dry) *ev_recorded = true;
      ws.release(mk);
    }
  }
  if (bilinear) {
    const Opnd dTo{dT16, ldT, tsplit};
    // dX = dT W^T : B operand [N = d, K = e] is W itself
    if (dX || ws.dry) {
      MI_TRY(gemm_impl(dTo, Opnd{W, D, 1}, B, D, D, 1.f, 0.f, nullptr, 0, dX, D, nullptr, 0, 1, 1, ws, stream));
      ws.release(mk);
    }
    // dW = X^T dT : both operands are row-major [B, D] matrices contracted over their rows (MN-major), split-K over the batch
    if (dW || ws.dry) {
      GemmArgs g;
      const int kb = static_cast<int>(round_up(B, kSplitAlign) / bk());
      g.a_mn = true; g.a = MapSpec{X, B, D, D};
      g.b_mn = true; g.b = MapSpec{dT16, B, tsplit == 2 ? Dp + D : D, ldT};
      g.M = D; g.N = D; g.seg_len = kb; g.k_blocks = kb;
      if (tsplit == 2) { g.k_blocks = 2 * kb; g.b_noff[1] = static_cast<int>(Dp); }
      const long long tiles = cdiv(D, rows_per_mblk()) * cdiv(D, mi::TILE_N);
      // The batch is the contraction dimension: B / 16 accumulating MMAs per output element.  The tensor core's fp32
      // accumulation of such a long, heavily cancelling sum (dW is tiny against the sum of its terms' magnitudes) loses
      // ~1e-3 of the result at B = 65536 with a few hundred K blocks per accumulator (measured: tests/test_gpu_parity.py
      // full-size case); strict mode therefore cuts the chains to <= 16 K blocks and sums the partials in a separate pass.
      const long long ks = choose_ksplit(tiles, g.k_blocks, strict ? cdiv(g.k_blocks, 16) : 1);
      g.ksplit = static_cast<int>(ks);
      g.out_f32 = dW; g.ld_out = D;
      MI_TRY(run_gemm(g, ws, stream));
      ws.release(mk);
    }
  }
  return MI_OK;
}


#include "mlp_critic.cuh"   // the reference's own concat-MLP critic (SURVEY 8f-1)
#include "gdv.cuh"          // Generalised Discrimination Value (SURVEY 8f-3)

int device_check() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); return MI_ERR_NO_DEVICE; }
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) { (void)cudaGetLastError(); return MI_ERR_NO_DEVICE; }
  return major == 10 ? MI_OK : MI_ERR_NO_DEVICE;
}

// second stream + event of the host-buffer entry point (one per device, created on first use)
constexpr int kMaxFeedChunks = 64;
struct CopySide { cudaStream_t stream; cudaEvent_t ev; cudaEvent_t ev_y; cudaEvent_t ev_in; cudaEvent_t ev_x[kMaxFeedChunks]; };
std::mutex g_host_entry_mu[64];      // the host-buffer entry point shares one CopySide per device: one call at a time per device
int copy_side(CopySide* out) {
  static std::mutex mu;
  static CopySide cache[64];
  static bool have[64] = {false};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { (void)cudaGetLastError(); return MI_ERR_CUDA; }
  std::lock_guard<std::mutex> lk(mu);
  if (!have[dev]) {
    MI_CUDA(cudaStreamCreateWithFlags(&cache[dev].stream, cudaStreamNonBlocking));
    MI_CUDA(cudaEventCreateWithFlags(&cache[dev].ev, cudaEventDisableTiming));
    MI_CUDA(cudaEventCreateWithFlags(&cache[dev].ev_y, cudaEventDisableTiming));
    MI_CUDA(cudaEventCreateWithFlags(&cache[dev].ev_in, cudaEventDisableTiming));
    for (int i = 0; i < kMaxFeedChunks; ++i) MI_CUDA(cudaEventCreateWithFlags(&cache[dev].ev_x[i], cudaEventDisableTiming));
    have[dev] = true;
  }
  *out = cache[dev];
  return MI_OK;
}

}  // namespace

#include "sharded.cuh"      // the batch-sharded step with its NCCL collectives as one host call (SURVEY 8e)

// ======================================================================================== C ABI
extern "C" {

const char* mi_status_string(int status) {
  switch (status) {
    case MI_OK: return "ok";
    case MI_ERR_BAD_ARG: return "bad argument (null pointer, non-positive size, D % 8 != 0 or misaligned pointer)";
    case MI_ERR_WORKSPACE: return "workspace too small";
    case MI_ERR_CUDA: return "CUDA error";
    case MI_ERR_NO_DEVICE: return "no sm_100 (Blackwell) device: this library has no CPU fallback";
    case MI_ERR_NO_NEGATIVES: return "no negative pairs (all study ids equal)";
    case MI_GUARD_TRIPPED: return "single-pass guard tripped: results are not valid, repeat the step with exact references";
    default: return "unknown status";
  }
}
const char* mi_last_cuda_error(void) { return g_cuda_err; }
int mi_abi_version(void) { return 5; }
int mi_device_check(void) { return device_check(); }
int64_t mi_launch_count(void) { return g_launches.load(); }
void mi_set_profiling(int on) { g_profiling = on != 0; }
// ms[k], launches[k] for k = 0 (score statistics), 1 (dS panel), 2 (GEMM), 3 (MLP single pass), 4 (MLP fused dZ1),
// 5 (MLP two-pass epilogues); drains the records (synchronises them).  mi_profile_read: the first three kinds.
int mi_profile_read_kinds(double* ms, int64_t* launches, int n_kinds) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (int k = 0; k < n_kinds; ++k) { ms[k] = 0.0; launches[k] = 0; }
  for (auto& r : g_prof) {
    float t = 0.f;
    MI_CUDA(cudaEventSynchronize(r.e1));
    MI_CUDA(cudaEventElapsedTime(&t, r.e0, r.e1));
    if (r.kind < n_kinds) { ms[r.kind] += t; launches[r.kind] += 1; }
    cudaEventDestroy(r.e0); cudaEventDestroy(r.e1);
  }
  g_prof.clear();
  return MI_OK;
}
int mi_profile_read(double* ms, int64_t* launches) { return mi_profile_read_kinds(ms, launches, 3); }
void mi_set_ref_sample_columns(int64_t n) { g_ref_sample_cols.store(n, std::memory_order_relaxed); }
void mi_set_overlap_reserve_sms(int n) { g_overlap_reserve_sms.store((n > 0 && n < 128) ? (n & ~1) : 0, std::memory_order_relaxed); }
void mi_set_mlp_panel_pairs(int64_t pairs) {      // bounded: pair indices inside a panel are 32-bit
  g_mlp_max_pairs = pairs > 0 ? (pairs < (1LL << 27) ? pairs : (1LL << 27)) : (1LL << 20);
}
void mi_set_mlp_mode(int mode) { g_mlp_mode.store(mode < 0 ? 3 : (mode & 3), std::memory_order_relaxed); }
int mi_get_mlp_mode(void) { return g_mlp_mode.load(std::memory_order_relaxed); }
void mi_set_cta_group(int g) { g_cta_group.store((g == 1) ? 1 : 2, std::memory_order_relaxed); }
int mi_get_cta_group(void) { return cta_group(); }

int mi_gemm_bf16(const void* A, int64_t lda, int a_split, const void* B, int64_t ldb, int b_split,
                 int64_t M, int64_t N, int64_t K, float alpha, float gamma, const void* sub, int64_t ld_sub,
                 float* out_f32, int64_t ld_out, void* out_bf16, int64_t ld_out16, int out_split,
                 mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(nullptr, 0, false);
  return gemm_impl(Opnd{static_cast<const __nv_bfloat16*>(A), lda, a_split == 2 ? 2 : 1},
                   Opnd{static_cast<const __nv_bfloat16*>(B), ldb, b_split == 2 ? 2 : 1}, M, N, K, alpha, gamma, sub, ld_sub,
                   out_f32, ld_out, out_bf16, ld_out16, out_split, 1, ws, reinterpret_cast<cudaStream_t>(stream));
}

size_t mi_gemm_bf16_mn_workspace_bytes(int64_t M, int64_t N, int64_t K, int a_split, int a_mn, int b_split, int b_mn) {
  Bump ws(nullptr, 0, true);
  if (gemm_mn_impl(Opnd{nullptr, 8, a_split == 2 ? 2 : 1}, a_mn != 0, Opnd{nullptr, 8, b_split == 2 ? 2 : 1}, b_mn != 0, M, N, K,
                   reinterpret_cast<float*>(16), N, nullptr, 0, 1, 0, ws, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_gemm_bf16_mn(const void* A, int64_t lda, int a_split, int a_mn, const void* B, int64_t ldb, int b_split, int b_mn,
                    int64_t M, int64_t N, int64_t K, float* out_f32, int64_t ld_out, void* out_bf16, int64_t ld_out16, int out_split,
                    void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(workspace, workspace_bytes, false);
  return gemm_mn_impl(Opnd{static_cast<const __nv_bfloat16*>(A), lda, a_split == 2 ? 2 : 1}, a_mn != 0,
                      Opnd{static_cast<const __nv_bfloat16*>(B), ldb, b_split == 2 ? 2 : 1}, b_mn != 0, M, N, K,
                      out_f32, ld_out, out_bf16, ld_out16, out_split, 0, ws, reinterpret_cast<cudaStream_t>(stream));
}

int mi_transpose_bf16(const void* in, int64_t ld_in, void* out, int64_t ld_out, int64_t R, int64_t C, mi_stream_t stream) {
  MI_TRY(device_check());
  return transpose_impl(in, ld_in, out, ld_out, R, C, reinterpret_cast<cudaStream_t>(stream));
}

int mi_cast_f32_to_bf16(const float* in, void* out, int64_t n, mi_stream_t stream) {
  MI_TRY(device_check());
  if (!in || !out || n <= 0) return MI_ERR_BAD_ARG;
  cast_f32_bf16_kernel<<<blocks_for(cdiv(n, 4), 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      in, static_cast<__nv_bfloat16*>(out), n);
  MI_LAUNCH_CHECK("cast_f32_bf16_kernel");
  return MI_OK;
}

size_t mi_score_stats_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D) {
  Bump ws(nullptr, 0, true);
  if (stats_impl(Opnd{nullptr, D, 1}, Opnd{nullptr, D, 1}, nullptr, nullptr, 0, Bq, Bk, D, 1.f, nullptr, nullptr, ws, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_score_stats(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                   const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                   int64_t Bq, int64_t Bk, int64_t D, float scale, float* row_out, double* scal_out,
                   void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(workspace, workspace_bytes, false);
  return stats_impl(Opnd{static_cast<const __nv_bfloat16*>(Q), ldq, q_split == 2 ? 2 : 1},
                    Opnd{static_cast<const __nv_bfloat16*>(K), ldk, k_split == 2 ? 2 : 1},
                    sid_q, sid_k, q_offset, Bq, Bk, D, scale, row_out, scal_out, ws, reinterpret_cast<cudaStream_t>(stream));
}

size_t mi_score_stats_rc_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D) {
  Bump ws(nullptr, 0, true);
  float dummy = 0.f;
  if (stats_rc_impl(Opnd{nullptr, D, 1}, Opnd{nullptr, D, 1}, nullptr, nullptr, 0, Bq, Bk, D, 1.f, nullptr, nullptr, nullptr, nullptr,
                    &dummy, ws, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_score_stats_rc_ex(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                         const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                         int64_t Bq, int64_t Bk, int64_t D, float scale, float* row_out, double* scal_out, float* col_lse_out,
                         void* event_k_ready, int k_local_valid, int include_pos,
                         void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  if (!col_lse_out) return MI_ERR_BAD_ARG;
  Bump ws(workspace, workspace_bytes, false);
  return stats_rc_impl(Opnd{static_cast<const __nv_bfloat16*>(Q), ldq, q_split == 2 ? 2 : 1},
                       Opnd{static_cast<const __nv_bfloat16*>(K), ldk, k_split == 2 ? 2 : 1},
                       sid_q, sid_k, q_offset, Bq, Bk, D, scale, row_out, scal_out, nullptr, nullptr, col_lse_out, ws,
                       reinterpret_cast<cudaStream_t>(stream), reinterpret_cast<cudaEvent_t>(event_k_ready), k_local_valid != 0,
                       nullptr, include_pos != 0);
}
int mi_score_stats_rc(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                      const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                      int64_t Bq, int64_t Bk, int64_t D, float scale, float* row_out, double* scal_out, float* col_lse_out,
                      void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  return mi_score_stats_rc_ex(Q, ldq, q_split, K, ldk, k_split, sid_q, sid_k, q_offset, Bq, Bk, D, scale, row_out, scal_out,
                              col_lse_out, nullptr, 0, 0, workspace, workspace_bytes, stream);
}

size_t mi_score_grad_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D, int precision) {
  Bump ws(nullptr, 0, true);
  GradOut oq, ok;
  // planned for the largest variant: hi/lo operands and both outputs
  const int sp = precision == MI_PREC_BF16_STRICT ? 2 : 1;
  if (grad_impl(Opnd{nullptr, D, sp}, Opnd{nullptr, D, 1}, nullptr, nullptr, 0, Bq, Bk, D, 1.f, nullptr, 1.f, nullptr, 0.f, 0, precision,
                1.f, 0.f, oq, &ok, ws, nullptr) != MI_OK) return 0;
  const size_t a = ws.peak;
  Bump ws2(nullptr, 0, true);
  if (grad_impl(Opnd{nullptr, D, 1}, Opnd{nullptr, D, sp}, nullptr, nullptr, 0, Bq, Bk, D, 1.f, nullptr, 1.f, nullptr, 0.f, 0, precision,
                1.f, 0.f, oq, &ok, ws2, nullptr) != MI_OK) return 0;
  return (a > ws2.peak ? a : ws2.peak) + 256;
}
int mi_score_grad(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                  const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                  int64_t Bq, int64_t Bk, int64_t D, float scale,
                  const float* refq, float wq, const float* refk, float wk, int include_diag, int precision,
                  float alpha, float gamma,
                  float* outq_f32, void* outq_bf16, int64_t ld_outq16, int outq_split, float* outk_f32,
                  void* event_after_outk, void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  if (q_offset < 0 || q_offset + Bq > Bk) return MI_ERR_BAD_ARG;
  Bump ws(workspace, workspace_bytes, false);
  GradOut oq, ok;
  oq.f32 = outq_f32; oq.ld = D;
  oq.bf16 = static_cast<__nv_bfloat16*>(outq_bf16); oq.ld16 = ld_outq16; oq.split = outq_split == 2 ? 2 : 1;
  ok.f32 = outk_f32; ok.ld = D;
  return grad_impl(Opnd{static_cast<const __nv_bfloat16*>(Q), ldq, q_split == 2 ? 2 : 1},
                   Opnd{static_cast<const __nv_bfloat16*>(K), ldk, k_split == 2 ? 2 : 1},
                   sid_q, sid_k, q_offset, Bq, Bk, D, scale, refq, wq, refk, wk, include_diag, precision,
                   alpha, gamma, oq, outk_f32 ? &ok : nullptr, ws, reinterpret_cast<cudaStream_t>(stream),
                   reinterpret_cast<cudaEvent_t>(event_after_outk));
}

size_t mi_score_ref_sample_workspace_bytes(int64_t Bq, int64_t n_cols, int64_t D, int64_t stride) {
  Bump ws(nullptr, 0, true);
  if (stride < 1) stride = ref_stride_auto(Bq, n_cols, D);
  // planned for a hi/lo Q (the larger K loop does not change the workspace, only the mask / partial buffers matter)
  if (ref_sample_impl(Opnd{nullptr, D, 1}, Opnd{nullptr, D, 1}, nullptr, nullptr, 0, Bq, n_cols, D, 1.f, 0, 0, n_cols, stride, 0.f,
                      nullptr, nullptr, nullptr, ws, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_score_ref_sample(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                        const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                        int64_t Bq, int64_t Bk, int64_t D, float scale, int include_diag,
                        int64_t col0, int64_t n_cols, int64_t stride, int subset,
                        float* ref_out, float* diag_out, float* lambda_out,
                        void* workspace, size_t workspace_bytes, mi_stream_t stream_) {
  MI_TRY(device_check());
  if (q_offset < 0 || q_offset + Bq > Bk) return MI_ERR_BAD_ARG;
  if (stride < 1) stride = ref_stride_auto(Bq, n_cols, D);
  const float margin = (stride > 1 || subset != 0) ? kRefMargin : 0.f;
  Bump ws(workspace, workspace_bytes, false);
  return ref_sample_impl(Opnd{static_cast<const __nv_bfloat16*>(Q), ldq, q_split == 2 ? 2 : 1},
                         Opnd{static_cast<const __nv_bfloat16*>(K), ldk, k_split == 2 ? 2 : 1},
                         sid_q, sid_k, q_offset, Bq, Bk, D, scale, include_diag, col0, n_cols, stride, margin,
                         ref_out, diag_out, lambda_out, ws, reinterpret_cast<cudaStream_t>(stream_));
}
int64_t mi_ref_sample_stride(int64_t Bq, int64_t n_cols, int64_t D) { return ref_stride_auto(Bq, n_cols, D); }

size_t mi_score_single_pass_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D, int precision) {
  Bump ws(nullptr, 0, true);
  const int sp = (precision & 1) ? 2 : 1;
  if (single_pass_impl(Opnd{nullptr, D, sp}, Opnd{nullptr, D, 1}, nullptr, nullptr, 0, Bq, Bk, D, 1.f, 0, precision, 1.f,
                       nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, ws, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_row_norm_max(const void* A, int64_t lda, int a_split, int64_t rows, int64_t D, float* norm_out, float* max_out, mi_stream_t stream_) {
  MI_TRY(device_check());
  if (!A || !norm_out || !max_out || rows <= 0 || D <= 0) return MI_ERR_BAD_ARG;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  row_norm_kernel<<<blocks_for(rows * 32, 256), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(A), lda, a_split == 2 ? 2 : 1,
                                                                   round_up(D, kSplitAlign), rows, D, norm_out);
  MI_LAUNCH_CHECK("row_norm_kernel");
  max_reduce_kernel<<<1, 1024, 0, stream>>>(norm_out, rows, max_out, 0.f, nullptr);
  MI_LAUNCH_CHECK("max_reduce_kernel");
  return MI_OK;
}
int mi_score_single_pass(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                         const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                         int64_t Bq, int64_t Bk, int64_t D, float scale, int include_diag, int precision, float inv_bg,
                         const float* ref, const float* lambda, const float* diag,
                         float* row_out, double* scal_out, float* oq_raw, float* ok_raw,
                         float* wrow, int32_t* flag_out, void* event_after_outk,
                         void* event_after_scal, void* event_k_ready, int k_local_valid,
                         void* workspace, size_t workspace_bytes, mi_stream_t stream_) {
  MI_TRY(device_check());
  if (q_offset < 0 || q_offset + Bq > Bk || !scal_out || !flag_out) return MI_ERR_BAD_ARG;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  Bump ws(workspace, workspace_bytes, false);
  MI_CUDA(cudaMemsetAsync(flag_out, 0, sizeof(int), stream));
  MI_TRY(single_pass_impl(Opnd{static_cast<const __nv_bfloat16*>(Q), ldq, q_split == 2 ? 2 : 1},
                          Opnd{static_cast<const __nv_bfloat16*>(K), ldk, k_split == 2 ? 2 : 1},
                          sid_q, sid_k, q_offset, Bq, Bk, D, scale, include_diag, precision, inv_bg, ref, lambda, diag,
                          row_out, oq_raw, ok_raw, wrow, flag_out, ws, stream,
                          reinterpret_cast<cudaEvent_t>(event_after_outk), scal_out, reinterpret_cast<cudaEvent_t>(event_after_scal),
                          reinterpret_cast<cudaEvent_t>(event_k_ready), nullptr, nullptr, k_local_valid != 0));
  return MI_OK;
}
int mi_merge_scalars(const double* scal_all, int world, int64_t B_global, int estimator, const float* lambda,
                     double* loss_out, float* lse_out, double* scratch8, mi_stream_t stream_) {
  MI_TRY(device_check());
  if (!scal_all || world <= 0 || !loss_out || !lse_out || !scratch8 || estimator < MI_EST_DV || estimator > MI_EST_INFONCE_ROW)
    return MI_ERR_BAD_ARG;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  merge_scal_kernel<<<1, 32, 0, stream>>>(scal_all, world, scratch8);
  MI_LAUNCH_CHECK("merge_scal_kernel");
  loss_finalize_kernel<<<1, 32, 0, stream>>>(scratch8, nullptr, B_global, estimator, loss_out, lse_out, lambda, nullptr);
  MI_LAUNCH_CHECK("loss_finalize_kernel");
  return MI_OK;
}
int64_t mi_merge_sym_stats_scratch_doubles(int64_t B_global) { return B_global > 0 ? merge_sym_scratch_doubles(B_global) : 0; }
int mi_merge_sym_stats(const double* scal_all, const float* col_all, int64_t col_pitch, int world, int64_t B_global,
                       double* loss_out, float* c_out, double* scratch, mi_stream_t stream) {
  MI_TRY(device_check());
  if (!scal_all || !col_all || world <= 0 || B_global <= 0 || col_pitch < B_global || !loss_out || !c_out || !scratch)
    return MI_ERR_BAD_ARG;
  return merge_sym_impl(scal_all, 8, col_all, col_pitch, world, B_global, loss_out, c_out, scratch,
                        reinterpret_cast<cudaStream_t>(stream));
}
int mi_single_finalize_q(const float* oq_raw, int64_t rows, int64_t D, const float* ref, const float* wrow, const float* lse,
                         int dv_like, float alpha, float gamma, const void* kdiag, int64_t ldk, int k_split,
                         float* out_f32, void* out_bf16, int64_t ld16, int out_split, mi_stream_t stream_) {
  MI_TRY(device_check());
  if (!oq_raw || !ref || !wrow || !kdiag || rows <= 0 || D <= 0 || (D % 8) != 0 || (dv_like && !lse) || (!out_f32 && !out_bf16)) return MI_ERR_BAD_ARG;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const long long Dp = round_up(D, kSplitAlign);
  __nv_bfloat16* ob = static_cast<__nv_bfloat16*>(out_bf16);
  finalize_q_kernel<<<blocks_capped(rows * D / 8, 256), 256, 0, stream>>>(oq_raw, D, rows, ref, wrow, lse, dv_like, alpha, gamma,
                                                                       static_cast<const __nv_bfloat16*>(kdiag), ldk, k_split == 2 ? 2 : 1, Dp,
                                                                       out_f32, ob, (ob && out_split == 2) ? ob + Dp : nullptr, ld16, nullptr);
  MI_LAUNCH_CHECK("finalize_q_kernel");
  return MI_OK;
}
int mi_single_finalize_k(float* ok, int64_t rows, int64_t D, const float* lambda, const float* lse, int dv_like,
                         float alpha, float gamma, const void* qdiag, int64_t ldq, int q_split, mi_stream_t stream_) {
  MI_TRY(device_check());
  if (!ok || !qdiag || rows <= 0 || D <= 0 || (dv_like && (!lse || !lambda))) return MI_ERR_BAD_ARG;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if ((D % 8) != 0) return MI_ERR_BAD_ARG;
  finalize_k_kernel<<<blocks_capped(rows * D / 8, 256), 256, 0, stream>>>(ok, D, rows, lambda, lse, dv_like, alpha, gamma,
                                                                   static_cast<const __nv_bfloat16*>(qdiag), ldq, q_split == 2 ? 2 : 1,
                                                                   round_up(D, kSplitAlign), 0, rows);
  MI_LAUNCH_CHECK("finalize_k_kernel");
  return MI_OK;
}

size_t mi_critic_workspace_bytes(int64_t B, int64_t D, int critic, int estimator, int precision, int need_grads) {
  Bump ws(nullptr, 0, true);
  (void)need_grads;   // planned for the larger (gradient) case always; forward-only calls simply use less
  if (critic_impl(nullptr, nullptr, nullptr, nullptr, B, D, critic, estimator, precision, 1.f, nullptr, nullptr, nullptr,
                  nullptr, ws, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_critic_loss_fwd_bwd(const void* X, const void* Y, const void* W, const int32_t* sid,
                           int64_t B, int64_t D, int critic, int estimator, int precision, float inv_tau,
                           double* loss_out, float* dX, float* dY, float* dW,
                           void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(workspace, workspace_bytes, false);
  return critic_impl(X, Y, W, sid, B, D, critic, estimator, precision, inv_tau, loss_out, dX, dY, dW, ws,
                     reinterpret_cast<cudaStream_t>(stream));
}

size_t mi_critic_host_scratch_bytes(int64_t B, int64_t D, int critic, int estimator, int precision, int need_grads) {
  const size_t core = mi_critic_workspace_bytes(B, D, critic, estimator, precision, need_grads);
  if (core == 0) return 0;
  Bump ws(nullptr, 0, true);
  ws.take<float>(static_cast<size_t>(B) * D); ws.take<float>(static_cast<size_t>(B) * D);     // staging fp32 X, Y
  ws.take<float>(static_cast<size_t>(D) * D);                                                  // staging fp32 W
  ws.take<__nv_bfloat16>(static_cast<size_t>(B) * D); ws.take<__nv_bfloat16>(static_cast<size_t>(B) * D);
  ws.take<__nv_bfloat16>(static_cast<size_t>(D) * D);
  ws.take<int>(B); ws.take<double>(8);
  ws.take<float>(static_cast<size_t>(B) * D); ws.take<float>(static_cast<size_t>(B) * D); ws.take<float>(static_cast<size_t>(D) * D);
  return ws.peak + 256 + core;
}
// in_bf16: the host embeddings / W are bf16 (copied straight into the operand buffers, no cast);
// grads_on_device: dX_host / dY_host / dW_host are DEVICE pointers — the gradients stay where the encoders' backward consumes them
static int host_entry_impl(const void* X_host_, const void* Y_host_, const void* W_host_, const int32_t* sid_host, bool in_bf16,
                           int64_t B, int64_t D, int critic, int estimator, int precision, float inv_tau,
                           double* loss_out_host, float* dX_host, float* dY_host, float* dW_host, bool grads_on_device,
                           void* dev_scratch, size_t dev_scratch_bytes, mi_stream_t stream_) {
  MI_TRY(device_check());
  const float* X_host = static_cast<const float*>(X_host_); const float* Y_host = static_cast<const float*>(Y_host_);
  const float* W_host = static_cast<const float*>(W_host_);
  const __nv_bfloat16* X_hb = static_cast<const __nv_bfloat16*>(X_host_); const __nv_bfloat16* Y_hb = static_cast<const __nv_bfloat16*>(Y_host_);
  const __nv_bfloat16* W_hb = static_cast<const __nv_bfloat16*>(W_host_);
  if (!X_host || !Y_host || !sid_host || !loss_out_host || !dev_scratch || B <= 0 || D <= 0) return MI_ERR_BAD_ARG;
  const bool bilinear = critic == MI_CRITIC_BILINEAR;
  if (bilinear && !W_host) return MI_ERR_BAD_ARG;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  typedef __nv_bfloat16 bf;
  Bump ws(dev_scratch, dev_scratch_bytes, false);
  const size_t nBD = static_cast<size_t>(B) * D, nDD = static_cast<size_t>(D) * D;
  float* X32 = ws.take<float>(nBD); float* Y32 = ws.take<float>(nBD); float* W32 = ws.take<float>(nDD);
  bf* X16 = ws.take<bf>(nBD); bf* Y16 = ws.take<bf>(nBD); bf* W16 = ws.take<bf>(nDD);
  int* sid = ws.take<int>(B); double* loss = ws.take<double>(8);
  float* dX = ws.take<float>(nBD); float* dY = ws.take<float>(nBD); float* dW = ws.take<float>(nDD);
  if (grads_on_device) { dX = dX_host; dY = dY_host; dW = dW_host; }
  if (!ws.ok()) return MI_ERR_WORKSPACE;
  ws.off = (ws.off + 255) & ~static_cast<size_t>(255);
  uint8_t* core = ws.base + ws.off;
  const size_t core_bytes = dev_scratch_bytes - ws.off;
  // Input side: the text embeddings go first; the image embeddings follow in row panels on a second stream, each with
  // its own event, and the single pass consumes them panel by panel (cast + projection + references inside the pass)
  // while the rest is still crossing PCIe.  Output side: dY is final before the last panel's dT contraction and the
  // dX / dW GEMMs, its copy back starts from an in-pass event on the second stream.
  // The second stream and its events are per device: calls on the same device are serialised here (the call
  // synchronises before it returns, so nothing is lost).
  int dev = 0;
  MI_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> entry_lock(g_host_entry_mu[dev & 63]);
  CopySide side;
  const bool have_side = copy_side(&side) == MI_OK;
  // every exit below this point leaves no copy in flight into / out of the caller's buffers
  auto fail = [&](int st) -> int {
    if (have_side) (void)cudaStreamSynchronize(side.stream);
    (void)cudaStreamSynchronize(stream);
    return st;
  };
#define MI_HOST_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(set_cuda_err(e__, #call)); } while (0)
#define MI_HOST_TRY(call) do { int s__ = (call); if (s__ != MI_OK) return fail(s__); } while (0)
  const long long chunk_rows = panel_mblks(B, B, D, precision & 1) * rows_per_mblk();
  const long long n_chunks = cdiv(B, chunk_rows);
  const bool want_grads = dX_host || dY_host || (dW_host && bilinear);
  const bool streamed = have_side && want_grads && single_pass_estimator(estimator, precision) && n_chunks <= kMaxFeedChunks;
  if (have_side) {      // the second stream starts after whatever the caller's stream still does with dev_scratch
    MI_HOST_CUDA(cudaEventRecord(side.ev_in, stream));
    MI_HOST_CUDA(cudaStreamWaitEvent(side.stream, side.ev_in, 0));
  }
  MI_HOST_CUDA(cudaMemcpyAsync(sid, sid_host, static_cast<size_t>(B) * 4, cudaMemcpyHostToDevice, stream));
  if (bilinear) {
    if (in_bf16) {
      MI_HOST_CUDA(cudaMemcpyAsync(W16, W_hb, nDD * 2, cudaMemcpyHostToDevice, stream));
    } else {
      MI_HOST_CUDA(cudaMemcpyAsync(W32, W_host, nDD * 4, cudaMemcpyHostToDevice, stream));
      MI_HOST_TRY(mi_cast_f32_to_bf16(W32, W16, static_cast<int64_t>(nDD), stream_));
    }
  }
  std::function<int(long long, long long)> x_ready;
  if (streamed) {
    if (in_bf16) MI_HOST_CUDA(cudaMemcpyAsync(Y16, Y_hb, nBD * 2, cudaMemcpyHostToDevice, side.stream));
    else MI_HOST_CUDA(cudaMemcpyAsync(Y32, Y_host, nBD * 4, cudaMemcpyHostToDevice, side.stream));
    MI_HOST_CUDA(cudaEventRecord(side.ev_y, side.stream));
    for (long long c = 0; c < n_chunks; ++c) {
      const long long r0 = c * chunk_rows, rows = (B - r0 < chunk_rows) ? (B - r0) : chunk_rows;
      if (in_bf16) MI_HOST_CUDA(cudaMemcpyAsync(X16 + r0 * D, X_hb + r0 * D, static_cast<size_t>(rows) * D * 2, cudaMemcpyHostToDevice, side.stream));
      else MI_HOST_CUDA(cudaMemcpyAsync(X32 + r0 * D, X_host + r0 * D, static_cast<size_t>(rows) * D * 4, cudaMemcpyHostToDevice, side.stream));
      MI_HOST_CUDA(cudaEventRecord(side.ev_x[c], side.stream));
    }
    MI_HOST_CUDA(cudaStreamWaitEvent(stream, side.ev_y, 0));
    if (!in_bf16) MI_HOST_TRY(mi_cast_f32_to_bf16(Y32, Y16, static_cast<int64_t>(nBD), stream_));
    x_ready = [&](long long r0, long long rows) -> int {
      if (r0 % chunk_rows != 0) return MI_ERR_BAD_ARG;                // the pass walks the same panels
      MI_CUDA(cudaStreamWaitEvent(stream, side.ev_x[r0 / chunk_rows], 0));
      if (in_bf16) return MI_OK;
      return mi_cast_f32_to_bf16(X32 + r0 * D, X16 + r0 * D, static_cast<int64_t>(rows * D), stream_);
    };
  } else if (in_bf16) {
    MI_HOST_CUDA(cudaMemcpyAsync(X16, X_hb, nBD * 2, cudaMemcpyHostToDevice, stream));
    MI_HOST_CUDA(cudaMemcpyAsync(Y16, Y_hb, nBD * 2, cudaMemcpyHostToDevice, stream));
  } else {
    MI_HOST_CUDA(cudaMemcpyAsync(X32, X_host, nBD * 4, cudaMemcpyHostToDevice, stream));
    MI_HOST_CUDA(cudaMemcpyAsync(Y32, Y_host, nBD * 4, cudaMemcpyHostToDevice, stream));
    MI_HOST_TRY(mi_cast_f32_to_bf16(X32, X16, static_cast<int64_t>(nBD), stream_));
    MI_HOST_TRY(mi_cast_f32_to_bf16(Y32, Y16, static_cast<int64_t>(nBD), stream_));
  }
  const bool early = dY_host != nullptr && have_side && !grads_on_device;
  // Pass 0: sampled references, no device-side fallback (the host decides: this call synchronises anyway).
  // Pass 1 (only if the guard tripped): exact references, inputs already on the device.
  double guard0 = 0.0;
  for (int attempt = 0; attempt < 2; ++attempt) {
    bool recorded = false;
    Fallback fb; fb.predicated = false;
    Bump cws(core, core_bytes, false);
    MI_HOST_TRY(critic_impl(X16, Y16, bilinear ? W16 : nullptr, sid, B, D, critic, estimator,
                            attempt == 0 ? precision : (precision | MI_PREC_TWO_PASS), inv_tau, loss,
                            dX_host ? dX : nullptr, dY_host ? dY : nullptr, (dW_host && bilinear) ? dW : nullptr, cws, stream,
                            early ? side.ev : nullptr, &recorded, (streamed && attempt == 0) ? &x_ready : nullptr, fb));
    if (dY_host && !grads_on_device) {
      cudaStream_t cs = stream;
      if (early && recorded) {
        MI_HOST_CUDA(cudaStreamWaitEvent(side.stream, side.ev, 0));
        cs = side.stream;
      }
      MI_HOST_CUDA(cudaMemcpyAsync(dY_host, dY, nBD * 4, cudaMemcpyDeviceToHost, cs));
    }
    MI_HOST_CUDA(cudaMemcpyAsync(loss_out_host, loss, 8 * sizeof(double), cudaMemcpyDeviceToHost, stream));
    if (dX_host && !grads_on_device) MI_HOST_CUDA(cudaMemcpyAsync(dX_host, dX, nBD * 4, cudaMemcpyDeviceToHost, stream));
    if (dW_host && bilinear && !grads_on_device) MI_HOST_CUDA(cudaMemcpyAsync(dW_host, dW, nDD * 4, cudaMemcpyDeviceToHost, stream));
    MI_HOST_CUDA(cudaStreamSynchronize(stream));
    if (have_side) MI_HOST_CUDA(cudaStreamSynchronize(side.stream));
    if (attempt == 1) {          // same report as the device entry: [7] = rows that tripped the sampled pass
      if (loss_out_host[7] != 0.0) loss_out_host[0] = std::nan("");   // impossible by construction (l = 1 for every row)
      loss_out_host[7] = guard0;
      break;
    }
    if (!(loss_out_host[7] != 0.0)) break;
    guard0 = loss_out_host[7];
  }
#undef MI_HOST_CUDA
#undef MI_HOST_TRY
  return MI_OK;
}

int mi_critic_loss_fwd_bwd_host(const float* X_host, const float* Y_host, const float* W_host, const int32_t* sid_host,
                                int64_t B, int64_t D, int critic, int estimator, int precision, float inv_tau,
                                double* loss_out_host, float* dX_host, float* dY_host, float* dW_host,
                                void* dev_scratch, size_t dev_scratch_bytes, mi_stream_t stream) {
  return host_entry_impl(X_host, Y_host, W_host, sid_host, false, B, D, critic, estimator, precision, inv_tau, loss_out_host,
                         dX_host, dY_host, dW_host, false, dev_scratch, dev_scratch_bytes, stream);
}
int mi_critic_loss_fwd_bwd_from_host(const void* X_host, const void* Y_host, const void* W_host, const int32_t* sid_host, int host_dtype,
                                     int64_t B, int64_t D, int critic, int estimator, int precision, float inv_tau,
                                     double* loss_out_host, float* dX_dev, float* dY_dev, float* dW_dev,
                                     void* dev_scratch, size_t dev_scratch_bytes, mi_stream_t stream) {
  if (host_dtype != 0 && host_dtype != 1) return MI_ERR_BAD_ARG;
  return host_entry_impl(X_host, Y_host, W_host, sid_host, host_dtype == 1, B, D, critic, estimator, precision, inv_tau, loss_out_host,
                         dX_dev, dY_dev, dW_dev, true, dev_scratch, dev_scratch_bytes, stream);
}

int mi_dist_ctx_create(void* nccl_comm, mi_dist_ctx** out) {
  MI_TRY(device_check());
  if (!nccl_comm || !out) return MI_ERR_BAD_ARG;
  const NcclApi& nc = nccl_api();
  if (!nc.ok) { std::snprintf(g_cuda_err, sizeof(g_cuda_err), "libnccl.so.2 not found in the process"); return MI_ERR_CUDA; }
  mi_dist_ctx* c = new mi_dist_ctx();
  c->comm = nccl_comm;
  MI_NCCL(nc.comm_count(nccl_comm, &c->world));
  MI_NCCL(nc.comm_rank(nccl_comm, &c->rank));
  MI_CUDA(cudaGetDevice(&c->device));
  MI_CUDA(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
  MI_CUDA(cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking));
  cudaEvent_t* evs[] = {&c->ev_in, &c->ev_lamloc, &c->ev_sid, &c->ev_y, &c->ev_lam, &c->ev_s, &c->ev_k, &c->ev_m, &c->ev_rs,
                        &c->ev_dwg, &c->ev_dw, &c->ev_drain, &c->ev_mask, &c->ev_start};
  for (cudaEvent_t* e : evs) MI_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  MI_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&c->guard_host), sizeof(double), cudaHostAllocDefault));
  c->guard_host[0] = 0.0;
  *out = c;
  return MI_OK;
}
void mi_dist_ctx_destroy(mi_dist_ctx* c) {
  if (!c) return;
  (void)cudaStreamSynchronize(c->comm_stream);
  (void)cudaStreamSynchronize(c->aux_stream);
  cudaEvent_t evs[] = {c->ev_in, c->ev_lamloc, c->ev_sid, c->ev_y, c->ev_lam, c->ev_s, c->ev_k, c->ev_m, c->ev_rs, c->ev_dwg, c->ev_dw,
                       c->ev_drain, c->ev_mask, c->ev_start};
  for (cudaEvent_t e : evs) (void)cudaEventDestroy(e);
  (void)cudaStreamDestroy(c->comm_stream);
  (void)cudaStreamDestroy(c->aux_stream);
  (void)cudaFreeHost(c->guard_host);
  delete c;
}
int mi_dist_ctx_info(const mi_dist_ctx* c, int* rank, int* world) {
  if (!c || !rank || !world) return MI_ERR_BAD_ARG;
  *rank = c->rank; *world = c->world;
  return MI_OK;
}
size_t mi_sharded_critic_workspace_bytes(int64_t B_local, int world, int64_t D, int critic, int estimator, int precision) {
  Bump ws(nullptr, 0, true);
  if (sharded_impl(nullptr, world, 0, nullptr, nullptr, nullptr, nullptr, B_local, D, critic, estimator, precision, 1.f, nullptr, nullptr,
                   nullptr, nullptr, ws, 0, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_sharded_critic_loss_fwd_bwd(mi_dist_ctx* ctx, const void* X_local, const void* Y_local, const void* W, const int32_t* sid_local,
                                   int64_t B_local, int64_t D, int critic, int estimator, int precision, float inv_tau,
                                   double* loss_out, float* dX, float* dY, float* dW,
                                   void* workspace, size_t workspace_bytes, int check_guard, mi_stream_t stream) {
  MI_TRY(device_check());
  if (!ctx) return MI_ERR_BAD_ARG;
  Bump ws(workspace, workspace_bytes, false);
  return sharded_impl(ctx, ctx->world, ctx->rank, X_local, Y_local, W, sid_local, B_local, D, critic, estimator, precision, inv_tau,
                      loss_out, dX, dY, dW, ws, check_guard, reinterpret_cast<cudaStream_t>(stream));
}

size_t mi_mlp_critic_workspace_bytes(int64_t B, int64_t D, int64_t H1, int64_t H2, int precision) {
  Bump ws(nullptr, 0, true);
  MlpParams prm{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  MlpGrads gr{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  if (mlp_impl(nullptr, nullptr, prm, nullptr, MlpDims{B, D, H1, H2}, MI_EST_DV, precision, nullptr, nullptr, gr, ws, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_mlp_critic_loss_fwd_bwd(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                               const float* W3, const float* b3, const int32_t* sid,
                               int64_t B, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                               double* loss_out, float* S_out, float* dX, float* dY, float* dW1, float* db1, float* dW2, float* db2,
                               float* dW3, float* db3, void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(workspace, workspace_bytes, false);
  return mlp_impl(X, Y, MlpParams{W1, b1, W2, b2, W3, b3}, sid, MlpDims{B, D, H1, H2}, estimator, precision, loss_out, S_out,
                  MlpGrads{dX, dY, dW1, db1, dW2, db2, dW3, db3}, ws, reinterpret_cast<cudaStream_t>(stream));
}

// ---- the MLP critic over a row block: the stage ops of the batch-sharded step (DESIGN 8.4)
// (the size queries plan every stage of both sequences: the path is chosen per step)
size_t mi_mlp_block_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D, int64_t H1, int64_t H2, int precision) {
  const MlpBlock blk{Bq, Bk, 0, Bk, nullptr, nullptr};
  const MlpDims d{Bk, D, H1, H2};
  size_t peak = 0;
  const int stages[5][2] = {{kMlpStageRef, 0}, {kMlpStageFwd, 0}, {kMlpStageFwd, 1}, {kMlpStageBwd, 0}, {kMlpStageBwd, 1}};
  for (const auto& st : stages) {
    Bump ws(nullptr, 0, true), keep(nullptr, 0, true);
    MlpBlockIO io{};
    io.two_pass = st[1];
    // the reference stage keeps nothing: its state comes from the workspace
    if (mlp_block_impl(st[0], nullptr, nullptr, MlpParams{}, blk, d, MI_EST_DV, precision, io, ws, st[0] == kMlpStageRef ? ws : keep,
                       nullptr) != MI_OK)
      return 0;
    if (ws.peak > peak) peak = ws.peak;
  }
  Bump ws(nullptr, 0, true);
  if (mlp_input_grad_impl(nullptr, nullptr, nullptr, 1, Bq, D, H1, precision, nullptr, nullptr, nullptr, ws, nullptr) != MI_OK) return 0;
  if (ws.peak > peak) peak = ws.peak;
  return peak + 256;
}
size_t mi_mlp_block_state_bytes(int64_t Bq, int64_t Bk, int64_t D, int64_t H1, int64_t H2, int precision) {
  Bump ws(nullptr, 0, true), keep(nullptr, 0, true);
  if (mlp_block_impl(kMlpStageFwd, nullptr, nullptr, MlpParams{}, MlpBlock{Bq, Bk, 0, Bk, nullptr, nullptr}, MlpDims{Bk, D, H1, H2},
                     MI_EST_DV, precision, MlpBlockIO{}, ws, keep, nullptr) != MI_OK) return 0;
  return keep.peak + 256;
}
int mi_mlp_block_ref_logit(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                           const float* W3, const float* b3, int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2,
                           int precision, float* ref_out, void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(workspace, workspace_bytes, false);
  MlpBlockIO io{};
  io.ref_out = ref_out;
  return mlp_block_impl(kMlpStageRef, X, Y, MlpParams{W1, b1, W2, b2, W3, b3}, MlpBlock{Bq, Bk, q_offset, Bk, nullptr, nullptr},
                        MlpDims{Bk, D, H1, H2}, MI_EST_DV, precision, io, ws, ws, reinterpret_cast<cudaStream_t>(stream));
}
int mi_mlp_block_fwd_rc(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                        const float* W3, const float* b3, const int32_t* sid_q, const int32_t* sid_k,
                        int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                        const float* ref, int two_pass, double* scal_out, float* col_lse_out, void* state, size_t state_bytes,
                        void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(workspace, workspace_bytes, false), keep(state, state_bytes, false);
  MlpBlockIO io{};
  io.ref = ref; io.two_pass = two_pass; io.scal_out = scal_out; io.col_lse_out = col_lse_out;
  return mlp_block_impl(kMlpStageFwd, X, Y, MlpParams{W1, b1, W2, b2, W3, b3}, MlpBlock{Bq, Bk, q_offset, Bk, sid_q, sid_k},
                        MlpDims{Bk, D, H1, H2}, estimator, precision, io, ws, keep, reinterpret_cast<cudaStream_t>(stream));
}
int mi_mlp_block_fwd(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                     const float* W3, const float* b3, const int32_t* sid_q, const int32_t* sid_k,
                     int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                     const float* ref, int two_pass, double* scal_out, void* state, size_t state_bytes,
                     void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  return mi_mlp_block_fwd_rc(X, Y, W1, b1, W2, b2, W3, b3, sid_q, sid_k, Bq, Bk, q_offset, D, H1, H2, estimator, precision, ref,
                             two_pass, scal_out, nullptr, state, state_bytes, workspace, workspace_bytes, stream);
}
int mi_mlp_block_merge(const double* scal_all, int world, int64_t B_global, int estimator, int two_pass, double* loss_out, double* merged,
                       mi_stream_t stream_) {
  MI_TRY(device_check());
  const bool sym = estimator == MI_EST_INFONCE_SYM;
  if (!scal_all || world <= 0 || B_global <= 0 || !loss_out || !merged || (sym && !two_pass) ||
      (estimator != MI_EST_DV && estimator != MI_EST_INFONCE_REF && estimator != MI_EST_INFONCE_ROW && !sym)) return MI_ERR_BAD_ARG;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  merge_scal_kernel<<<1, 32, 0, stream>>>(scal_all, world, merged);
  MI_LAUNCH_CHECK("merge_scal_kernel");
  // symmetric InfoNCE: the slots of infonce_row (slot 0 = loss_row, slot 5 = 0); the caller completes 0 and 5 from the
  // merged columns
  loss_finalize_kernel<<<1, 32, 0, stream>>>(merged, nullptr, B_global, sym ? MI_EST_INFONCE_ROW : estimator, loss_out, nullptr, nullptr,
                                             nullptr);
  MI_LAUNCH_CHECK("loss_finalize_kernel");
  if (!two_pass) {
    mlp_block_guard_kernel<<<1, 1, 0, stream>>>(merged, loss_out);
    MI_LAUNCH_CHECK("mlp_block_guard_kernel");
  }
  return MI_OK;
}
int mi_mlp_block_bwd_rc(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                        const float* W3, const float* b3, const int32_t* sid_q, const int32_t* sid_k,
                        int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                        int two_pass, const double* loss, const double* merged, const float* col_lse, void* state, size_t state_bytes,
                        float* dX, float* dC_part, float* dW1, float* db1, float* dW2, float* db2, float* dW3, float* db3,
                        void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(workspace, workspace_bytes, false), keep(state, state_bytes, false);
  MlpBlockIO io{};
  io.two_pass = two_pass; io.loss = loss; io.merged = merged; io.col_lse = col_lse; io.dC_part = dC_part;
  io.gr = MlpGrads{dX, nullptr, dW1, db1, dW2, db2, dW3, db3};
  return mlp_block_impl(kMlpStageBwd, X, Y, MlpParams{W1, b1, W2, b2, W3, b3}, MlpBlock{Bq, Bk, q_offset, Bk, sid_q, sid_k},
                        MlpDims{Bk, D, H1, H2}, estimator, precision, io, ws, keep, reinterpret_cast<cudaStream_t>(stream));
}
int mi_mlp_block_bwd(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                     const float* W3, const float* b3, const int32_t* sid_q, const int32_t* sid_k,
                     int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                     int two_pass, const double* loss, const double* merged, void* state, size_t state_bytes,
                     float* dX, float* dC_part, float* dW1, float* db1, float* dW2, float* db2, float* dW3, float* db3,
                     void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  return mi_mlp_block_bwd_rc(X, Y, W1, b1, W2, b2, W3, b3, sid_q, sid_k, Bq, Bk, q_offset, D, H1, H2, estimator, precision, two_pass,
                             loss, merged, nullptr, state, state_bytes, dX, dC_part, dW1, db1, dW2, db2, dW3, db3, workspace,
                             workspace_bytes, stream);
}
size_t mi_mlp_input_grad_workspace_bytes(int64_t R, int64_t D, int64_t H1, int precision) {
  Bump ws(nullptr, 0, true);
  if (mlp_input_grad_impl(nullptr, nullptr, nullptr, 0, R, D, H1, precision, nullptr, nullptr, nullptr, ws, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_mlp_input_grad(const float* dZ, const float* In, const float* W1, int side, int64_t R, int64_t D, int64_t H1, int precision,
                      float* dIn, float* dW1, float* db1, void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(workspace, workspace_bytes, false);
  return mlp_input_grad_impl(dZ, In, W1, side, R, D, H1, precision, dIn, dW1, db1, ws, reinterpret_cast<cudaStream_t>(stream));
}

// ---- introspection of the host-side scheduling decisions (CPU tests; no device needed)
int mi_plan_ksplit(int64_t tiles, int k_blocks, int64_t min_ks) { return choose_ksplit(tiles, k_blocks, min_ks); }
// The work items of the fused dZ1 kernel (EpiMlpDa, Sched::order 2) for a panel of `rr` image rows: item t is
// out[3 t .. 3 t + 2] = {unit, M block, N tile} in the order a CTA pair walks them.  Returns the number of items
// (> max_items: nothing beyond max_items was written).
int64_t mi_plan_mlp_walk(int64_t rr, int64_t B, int64_t H1, int32_t* out, int64_t max_items) {
  if (rr <= 0 || B <= 0 || H1 <= 0) return MI_ERR_BAD_ARG;
  const long long Bp = round_up(B, rows_per_mblk());
  Sched sc;
  single_segment(sc);
  sc.order = 2;
  sc.n_ntile = static_cast<int>(cdiv(H1, mi::TILE_N));
  sc.grp = static_cast<int>(Bp / rows_per_mblk()); sc.n_il = static_cast<int>(rr);
  mlp_da_chunks(rr, static_cast<long long>(sc.n_ntile) * sc.grp, sc.chunk_len, sc.n_chunks);
  sc.n_mblk = sc.grp * sc.n_il; sc.n_split = 1; sc.n_ksplit = 1; sc.k_blocks = 1;
  int64_t n = 0;
  for (int u = 0; u < mi::num_units(sc); ++u) {
    const mi::Unit un = mi::decode_unit<true>(sc, u);
    for (int it = 0; it < un.n_items; ++it, ++n) {
      if (n < max_items && out != nullptr) {
        out[3 * n] = u; out[3 * n + 1] = un.m + it * un.m_step; out[3 * n + 2] = un.nt0;
      }
    }
  }
  return n;
}

size_t mi_gdv_workspace_bytes(int64_t Np, int64_t Nn, int64_t D, int precision) {
  Bump ws(nullptr, 0, true);
  if (gdv_impl(nullptr, nullptr, Np, Nn, D, precision, nullptr, ws, nullptr) != MI_OK) return 0;
  return ws.peak + 256;
}
int mi_gdv(const float* pos, const float* neg, int64_t Np, int64_t Nn, int64_t D, int precision, double* out,
           void* workspace, size_t workspace_bytes, mi_stream_t stream) {
  MI_TRY(device_check());
  Bump ws(workspace, workspace_bytes, false);
  return gdv_impl(pos, neg, Np, Nn, D, precision, out, ws, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
