// Persistent, warp-specialised tcgen05 / TMA tile engine for sm_100a.
//
// One kernel skeleton computes accumulator tiles  ACC[128*kCG x 256] = A[rows, K] * B[cols, K]^T
// (bf16 operands, K-major, fp32 accumulate in TMEM) and hands every tile to an epilogue policy:
//
//   EpiStats   online (max, sum-exp) row statistics of the masked score matrix  — S is never stored
//   EpiPStore  recomputes score tiles and writes the bf16 dS panel  P = incl * (a e^{S-rq} + b e^{S-rk})
//   EpiStore   plain GEMM epilogue  C = alpha * (ACC - gamma * SUB)
//
// Roles (640 threads): warp 0 lane 0 = TMA producer, warp 1 lane 0 = MMA issuer (leader CTA only when
// kCG == 2), warp 2 = TMEM allocator, warps 4..19 = epilogue (warp%4 selects the 32-lane TMEM
// quarter, (warp-4)/4 the 64-column quarter of the tile).  Pipelines: smem ring full/empty (TMA <-> MMA)
// and a 2-deep TMEM accumulator ring tmem_full/tmem_empty (MMA <-> epilogue), so the epilogue of
// tile t overlaps the MMAs of tile t+1.  With kCG == 2 a CTA pair (cluster 2x1) shares the B operand:
// each CTA loads its own 128 A rows and one 128-row half of the 256-row B tile, the leader issues
// cta_group::2 MMAs with M = 256 and commits are multicast to both CTAs.
#pragma once
#include <type_traits>
#include "ptx.cuh"

namespace mi {

constexpr int BLOCK_M = 128;   // accumulator rows per CTA (TMEM lanes)
constexpr int TILE_N = 256;    // accumulator columns per tile
constexpr int ATOM_K = 64;     // 64 bf16 = 128 B = one swizzle-128B row (TMA box width)
constexpr int UMMA_K = 16;
constexpr int kNumThreads = 640;
constexpr int kEpiWarp0 = 4;
constexpr int kNumEpiWarps = 16;    // 4 per SM sub-partition: enough warps in flight to hide TMEM / MUFU / smem latency
constexpr int kTmemCols = 512;

// K block per pipeline stage: 128 for CTA pairs (8 MMAs per barrier round trip, 3 stages of 64 KB),
// 64 for the single-CTA variant (4 stages of 48 KB).
__host__ __device__ constexpr int block_k(int cg) { return cg == 2 ? 128 : 64; }

template <int kCG>
struct Cfg {
  static constexpr int kBK = block_k(kCG);
  static constexpr int kAtoms = kBK / ATOM_K;                      // 64-wide swizzle atoms per stage
  static constexpr int kStages = (kCG == 1) ? 4 : 3;
  static constexpr int kAAtomBytes = BLOCK_M * ATOM_K * 2;         // 16 KB: 128 rows x 128 B
  static constexpr int kABytes = kAAtomBytes * kAtoms;
  static constexpr int kBRows = TILE_N / kCG;                      // B rows this CTA loads
  static constexpr int kBAtomBytes = kBRows * ATOM_K * 2;
  static constexpr int kBBytes = kBAtomBytes * kAtoms;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024;  // + slack for 1024 B alignment
  template <class Epi> static constexpr int smem_bytes() { return kSmemBytes + Epi::kEpiSmemBytes; }
};

// Work decomposition.  A "unit" is (m block, N-range split, K split); a CTA (pair) walks units
// u = pair, pair + n_pairs, ... and inside a unit walks its N tiles, each over its K blocks.
// kSegs: the length of the K-segment table.  Host code plans with Sched (six entries); the fast / strict kernels take
// SchedT<4> — the kernel parameter of the parent layout, so their register allocation is unchanged — and only the
// MLP critic's fp32 mode (six segments) launches kernels that take the six-entry table.
constexpr int kMaxSegs = 6;
template <int kSegs>
struct SchedT {
  int n_mblk;     // M blocks of 128*kCG rows
  int n_ntile;    // N tiles of 256 columns
  int n_split;    // contiguous N-range splits per M block
  int n_ksplit;   // K splits (split-K GEMM), 1 otherwise
  int nt_base;    // first N tile of this launch (a launch may cover a sub-range of the columns)
  int order;      // 0: m fastest (concurrent units share the N range), 1: ksplit, split fastest,
                  // 2: "column walk" (below)
  int k_blocks;   // number of K blocks (block_k wide) per tile, all segments
  // K segments: block kb belongs to segment kb / seg_len and reads A at K block a_seg[seg] + kb % seg_len,
  // B at b_seg[seg] + kb % seg_len.  One segment = plain GEMM; more = sums of products of hi/lo splits,
  // e.g. [P_hi | P_lo] x [V ; V] or [T_hi | T_lo] x [Y ; Y] (fp32-accumulate "strict" mode), or the six terms of two
  // three-piece operands (the MLP critic's fp32 mode).
  int seg_len;
  int a_seg[kSegs];
  int b_seg[kSegs];
  int a_moff[kSegs];  // MN-major A only: M-coordinate offset of the segment (e.g. the lo half of a [hi | lo] panel)
  int b_noff[kSegs];  // MN-major B only: N-coordinate offset of the segment
  // Device-side launch predicate: when non-null and *run_if == 0 the whole grid returns at once.  The exact
  // fallback of the single pass is enqueued behind such a flag, so it costs a few empty launches unless needed.
  const int* run_if;
  // order 2: the M blocks form a grid [n_il][grp] (m = il * grp + jb).  A unit is (N tile, jb, chunk of chunk_len
  // consecutive il) and its items are the M blocks il * grp + jb of the chunk, all on the SAME N tile: the rows of
  // consecutive items are `grp` M blocks apart, so an epilogue thread meets the same (jb-local row, column) cell of
  // every il and can sum over il in registers (EpiMlpDa).
  int grp, chunk_len, n_chunks, n_il;
};
using Sched = SchedT<kMaxSegs>;

// A unit's work items: item `it` is the accumulator tile (M block m + it * m_step, N tile nt0 + it * nt_step).
struct Unit { int m, s, ks, nt0, nt1, kb0, kb1, n_items, m_step, nt_step; };

template <int kSegs>
__host__ __device__ __forceinline__ int num_units(const SchedT<kSegs>& sc) {
  return sc.order == 2 ? sc.n_ntile * sc.grp * sc.n_chunks : sc.n_mblk * sc.n_split * sc.n_ksplit;
}
template <int kSegs>
__device__ __forceinline__ int sel_seg(const int (&a)[kSegs], int i) {
  if constexpr (kSegs == 4) return i == 0 ? a[0] : i == 1 ? a[1] : i == 2 ? a[2] : a[3];
  else return i == 0 ? a[0] : i == 1 ? a[1] : i == 2 ? a[2] : i == 3 ? a[3] : i == 4 ? a[4] : a[5];
}

template <bool kWalk, int kSegs>
__host__ __device__ __forceinline__ Unit decode_unit(const SchedT<kSegs>& sc, int u) {
  Unit r;
  if (kWalk && sc.order == 2) {
    const int nt = u % sc.n_ntile; int t = u / sc.n_ntile;      // the N tiles of an M block run concurrently (A tile from L2)
    const int jb = t % sc.grp, il0 = (t / sc.grp) * sc.chunk_len;
    r.m = il0 * sc.grp + jb; r.s = 0; r.ks = 0;
    r.nt0 = sc.nt_base + nt; r.nt1 = r.nt0 + 1;
    r.kb0 = 0; r.kb1 = sc.k_blocks;
    r.n_items = sc.n_il - il0 < sc.chunk_len ? sc.n_il - il0 : sc.chunk_len;
    r.m_step = sc.grp; r.nt_step = 0;
    return r;
  }
  if (sc.order == 0) {
    r.m = u % sc.n_mblk; int t = u / sc.n_mblk;
    r.s = t % sc.n_split; r.ks = t / sc.n_split;
  } else {
    r.ks = u % sc.n_ksplit; int t = u / sc.n_ksplit;
    r.s = t % sc.n_split; r.m = t / sc.n_split;
  }
  r.nt0 = sc.nt_base + (int)(((long long)r.s * sc.n_ntile) / sc.n_split);
  r.nt1 = sc.nt_base + (int)(((long long)(r.s + 1) * sc.n_ntile) / sc.n_split);
  r.kb0 = (int)(((long long)r.ks * sc.k_blocks) / sc.n_ksplit);
  r.kb1 = (int)(((long long)(r.ks + 1) * sc.k_blocks) / sc.n_ksplit);
  r.n_items = r.nt1 - r.nt0; r.m_step = 0; r.nt_step = 1;
  return r;
}

// kAMN: the A operand is stored M-contiguous ("MN-major": A[m,k] at base[k*ld + m], i.e. the transpose
// of a row-major [K, M] matrix).  Its 128(M) x kBK(K) tile is fetched as 64(K) x 64(M) boxes — for each
// 64-wide M half the K rows are contiguous — and described to the MMA with the MN-major SWIZZLE_128B
// canonical layout (LBO = bytes between the M halves, SBO = 1 KB between 8-row K groups).
// kBMN: the same for the B operand (B[n,k] at base[k*ld + n]): per 64-wide N group the K rows are contiguous.
template <int kCG, class Epi, bool kAMN, bool kBMN, int kSegs>
__global__ void __launch_bounds__(kNumThreads, 1)
tile_engine_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   const SchedT<kSegs> sc, const __grid_constant__ typename Epi::Params ep) {
  using C = Cfg<kCG>;
  if (sc.run_if != nullptr && *sc.run_if == 0) return;      // grid-uniform: both CTAs of a pair leave together
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[C::kStages];
  __shared__ __align__(8) uint64_t empty_bar[C::kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;

  const uint32_t warp = threadIdx.x >> 5;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t cta_rank = (kCG == 2) ? ptx::cluster_ctarank() : 0u;
  const bool leader = (cta_rank == 0);
  const int pair_id = blockIdx.x / kCG;
  const int n_pairs = gridDim.x / kCG;
  const int n_units = num_units(sc);

  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  const uint32_t tiles_addr = (raw_addr + 1023u) & ~1023u;
  uint8_t* epi_smem = smem_raw + (tiles_addr - raw_addr) + C::kStages * C::kStageBytes;   // Epi staging, if any

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_a);
    ptx::prefetch_tmap(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) { ptx::mbar_init(&full_bar[s], 1); ptx::mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { ptx::mbar_init(&tmem_full_bar[a], 1); ptx::mbar_init(&tmem_empty_bar[a], kNumEpiWarps * kCG); }
    ptx::fence_barrier_init();
  }
  __syncwarp();
  if (warp == 2) {
    ptx::tmem_alloc<kCG>(&tmem_base_slot, kTmemCols);
    ptx::tmem_relinquish<kCG>();
  }
  ptx::tc_fence_before();
  if constexpr (kCG == 2) ptx::cluster_sync(); else __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;
  const uint32_t full0 = ptx::smem_u32(&full_bar[0]);
  const uint32_t empty0 = ptx::smem_u32(&empty_bar[0]);

  // Role loops run warp-uniformly (all 32 lanes walk the same schedule and poll the same barriers);
  // only the TMA / MMA / commit instructions themselves are issued by lane 0.  This keeps the loop
  // state in uniform registers instead of paying a divergent-to-uniform move per operand.
  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    uint32_t stage = 0, phase = 0;
    const uint32_t full0_lead = (kCG == 2) ? ptx::mapa(full0, 0) : full0;
    const uint64_t ta = reinterpret_cast<uint64_t>(&tmap_a), tb = reinterpret_cast<uint64_t>(&tmap_b);
    for (int u = pair_id; u < n_units; u += n_pairs) {
      const Unit un = decode_unit<Epi::kWalk>(sc, u);
      const int n_items = Epi::kWalk ? un.n_items : un.nt1 - un.nt0;
      for (int it = 0; it < n_items; ++it) {
        const int a_row = ((Epi::kWalk ? un.m + it * un.m_step : un.m) * kCG + (int)cta_rank) * BLOCK_M;
        const int b_row = (Epi::kWalk ? un.nt0 : un.nt0 + it) * TILE_N + (int)cta_rank * C::kBRows;
        int seg = un.kb0 / sc.seg_len, w = un.kb0 - seg * sc.seg_len;
        int a_k = (sel_seg(sc.a_seg, seg) + w) * C::kBK, b_k = (sel_seg(sc.b_seg, seg) + w) * C::kBK;
        int a_m = a_row + sel_seg(sc.a_moff, seg);
        int b_n = b_row + sel_seg(sc.b_noff, seg);
        for (int kb = un.kb0; kb < un.kb1; ++kb) {
          ptx::mbar_wait_addr(empty0 + stage * 8u, phase ^ 1u, 1);
          if (lane == 0) {
            const uint32_t sa = tiles_addr + stage * C::kStageBytes;
            const uint32_t sb = sa + C::kABytes;
            const uint32_t bar = full0_lead + stage * 8u;
            if (kCG == 1 || leader) ptx::mbar_arrive_expect_tx_addr(full0 + stage * 8u, kCG * C::kStageBytes);
#pragma unroll
            for (int t = 0; t < C::kAtoms; ++t) {
              if constexpr (kAMN) {
                // per 64-wide M half: kBK contiguous K rows of 128 B
                ptx::tma_load_2d_addr<kCG>(sa + t * (ATOM_K * 128), ta, bar, a_m, a_k + t * ATOM_K);
                ptx::tma_load_2d_addr<kCG>(sa + C::kABytes / 2 + t * (ATOM_K * 128), ta, bar, a_m + 64, a_k + t * ATOM_K);
              } else {
                ptx::tma_load_2d_addr<kCG>(sa + t * C::kAAtomBytes, ta, bar, a_k + t * ATOM_K, a_row);
              }
              if constexpr (kBMN) {
#pragma unroll
                for (int h = 0; h < C::kBRows / 64; ++h)
                  ptx::tma_load_2d_addr<kCG>(sb + h * (C::kBK * 128) + t * (ATOM_K * 128), tb, bar, b_n + 64 * h, b_k + t * ATOM_K);
              } else {
                ptx::tma_load_2d_addr<kCG>(sb + t * C::kBAtomBytes, tb, bar, b_k + t * ATOM_K, b_row);
              }
            }
          }
          __syncwarp();
          a_k += C::kBK; b_k += C::kBK;
          if (++w == sc.seg_len) {
            w = 0; ++seg;
            a_k = sel_seg(sc.a_seg, seg) * C::kBK; b_k = sel_seg(sc.b_seg, seg) * C::kBK; a_m = a_row + sel_seg(sc.a_moff, seg);
            b_n = b_row + sel_seg(sc.b_noff, seg);
          }
          if (++stage == (uint32_t)C::kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (leader) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(BLOCK_M * kCG, TILE_N) | (kAMN ? (1u << 15) : 0u) | (kBMN ? (1u << 16) : 0u);
      const uint32_t tfull0 = ptx::smem_u32(&tmem_full_bar[0]);
      const uint32_t tempty0 = ptx::smem_u32(&tmem_empty_bar[0]);
      // descriptor templates (everything but the 14-bit start address)
      const uint64_t da_hi = kAMN ? ptx::make_smem_desc_mn128(0, C::kABytes / 2) : ptx::make_smem_desc_k128(0);
      const uint64_t db_hi = kBMN ? ptx::make_smem_desc_mn128(0, C::kBK * 128) : ptx::make_smem_desc_k128(0);
      uint32_t stage = 0, phase = 0, tile_cnt = 0;
      for (int u = pair_id; u < n_units; u += n_pairs) {
        const Unit un = decode_unit<Epi::kWalk>(sc, u);
        const int n_items = Epi::kWalk ? un.n_items : un.nt1 - un.nt0;
        for (int it = 0; it < n_items; ++it) {
          const uint32_t as = tile_cnt & 1u, aphase = (tile_cnt >> 1) & 1u;
          ptx::mbar_wait_addr(tempty0 + as * 8u, aphase ^ 1u, 2);
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + as * TILE_N;
          uint32_t acc = 0;
          for (int kb = un.kb0; kb < un.kb1; ++kb) {
            ptx::mbar_wait_addr(full0 + stage * 8u, phase, 3);
            ptx::tc_fence_after();
            if (lane == 0) {
              const uint32_t sa16 = (tiles_addr + stage * C::kStageBytes) >> 4;     // 16 B units
              const uint64_t da = da_hi | (uint64_t)sa16;
              const uint64_t db = db_hi | (uint64_t)(sa16 + (C::kABytes >> 4));
#pragma unroll
              for (int k = 0; k < C::kBK / UMMA_K; ++k) {
                // K-major: 16 bf16 = 32 B inside the 128 B swizzle row (+2), next 64-wide atom after 4 steps;
                // MN-major: 16 K rows = two 1 KB swizzle atoms (+128)
                const uint32_t a_adv = kAMN ? (uint32_t)(128 * k)
                                            : (uint32_t)((k / 4) * (C::kAAtomBytes >> 4) + (k % 4) * 2);
                const uint32_t b_adv = kBMN ? (uint32_t)(128 * k)
                                            : (uint32_t)((k / 4) * (C::kBAtomBytes >> 4) + (k % 4) * 2);
                ptx::umma_bf16<kCG>(d_tmem, da + a_adv, db + b_adv, idesc, (k == 0) ? acc : 1u);
              }
              ptx::umma_commit_addr<kCG>(empty0 + stage * 8u, 0x3);   // smem slot reusable once these MMAs retire
            }
            __syncwarp();
            acc = 1u;
            if (++stage == (uint32_t)C::kStages) { stage = 0; phase ^= 1u; }
          }
          if (lane == 0) ptx::umma_commit_addr<kCG>(tfull0 + as * 8u, 0x3);   // accumulator ready for the epilogue
          __syncwarp();
          ++tile_cnt;
        }
      }
    }
  } else if (warp >= kEpiWarp0) {
    // ------------------------------------------------------------ epilogue (16 warps)
    const uint32_t quarter = warp & 3u;                 // TMEM lanes 32*quarter .. +31 (hardware: warp % 4)
    const uint32_t colq = (warp - kEpiWarp0) >> 2;        // 64-column quarter of the 256-column tile
    uint32_t tile_cnt = 0;
    typename Epi::State st;
    Epi::init(ep, st);
    st.stage_smem = epi_smem + (warp - kEpiWarp0) * (Epi::kEpiSmemBytes / kNumEpiWarps);
    for (int u = pair_id; u < n_units; u += n_pairs) {
      const Unit un = decode_unit<Epi::kWalk>(sc, u);
      const int row0 = (un.m * kCG + (int)cta_rank) * BLOCK_M + (int)(quarter * 32u + lane);
      const int n_items = Epi::kWalk ? un.n_items : un.nt1 - un.nt0;
      Epi::unit_begin(ep, st, un, row0, (int)colq);
      if constexpr (Epi::kJoint) {
        // The unit's (<= 2) N tiles are ONE logical tile: a first pass over both accumulator stages forms a per-row
        // quantity that needs every column (Epi::pass1 ... Epi::mid, which may synchronise the 16 epilogue warps), the
        // second pass re-reads the stages from TMEM, hands them back and runs Epi::chunk.
        const uint32_t lane_addr = tmem_base + ((quarter * 32u) << 16) + colq * 64u;
        for (int it = 0; it < n_items; ++it) {
          const uint32_t tc = tile_cnt + (uint32_t)it, as = tc & 1u, aphase = (tc >> 1) & 1u;
          ptx::mbar_wait(&tmem_full_bar[as], aphase, 4);
          ptx::tc_fence_after();
          {   // both 32-column chunks in flight before the wait: the first pass is short, TMEM latency would dominate it
            uint32_t v0[32], v1[32];
            ptx::tmem_ld_32x32(lane_addr + as * TILE_N, v0);
            ptx::tmem_ld_32x32(lane_addr + as * TILE_N + 32u, v1);
            ptx::tmem_ld_wait();
            const int col = (un.nt0 + it) * TILE_N + (int)(colq * 64u);
            Epi::pass1(ep, st, col, v0);
            Epi::pass1(ep, st, col + 32, v1);
          }
        }
        Epi::mid(ep, st, un, row0, (int)colq, epi_smem);
        for (int it = 0; it < n_items; ++it) {
          const uint32_t as = (tile_cnt + (uint32_t)it) & 1u;
          const uint32_t base = lane_addr + as * TILE_N;
          const int col = (un.nt0 + it) * TILE_N + (int)(colq * 64u);
          // 16-column pieces; the next piece's TMEM read is in flight while the current one is processed
          uint32_t va[16], vb[16];
          ptx::tmem_ld_32x16(base, va);
          ptx::tmem_ld_wait();
          ptx::tmem_ld_32x16(base + 16u, vb);
          Epi::template chunk16<0>(ep, st, un, row0, col, va);
          ptx::tmem_ld_wait();
          ptx::tmem_ld_32x16(base + 32u, va);
          Epi::template chunk16<1>(ep, st, un, row0, col + 16, vb);
          ptx::tmem_ld_wait();
          ptx::tmem_ld_32x16(base + 48u, vb);
          Epi::template chunk16<2>(ep, st, un, row0, col + 32, va);
          ptx::tmem_ld_wait();
          {   // the stage's last read is in registers: hand it back to the MMA issuer
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if constexpr (kCG == 1) ptx::mbar_arrive(&tmem_empty_bar[as]);
              else ptx::mbar_arrive_remote(&tmem_empty_bar[as], 0);
            }
          }
          Epi::template chunk16<3>(ep, st, un, row0, col + 48, vb);
        }
        tile_cnt += (uint32_t)n_items;
      } else {
        for (int it = 0; it < n_items; ++it) {
          const int row = Epi::kWalk ? row0 + it * un.m_step * (kCG * BLOCK_M) : row0;
          const int nt = Epi::kWalk ? un.nt0 : un.nt0 + it;
          const uint32_t as = tile_cnt & 1u, aphase = (tile_cnt >> 1) & 1u;
          if constexpr (Epi::kChunk16) Epi::item_begin(ep, st, row, nt * TILE_N + (int)(colq * 64u));   // loads issued before the wait
          ptx::mbar_wait(&tmem_full_bar[as], aphase, 4);
          ptx::tc_fence_after();
          if constexpr (Epi::kChunk16) {
            auto quarter16 = [&](auto qc) {
              constexpr int c = decltype(qc)::value;
              const uint32_t col_in_tile = colq * 64u + (uint32_t)c * 16u;
              uint32_t v[16];
              ptx::tmem_ld_32x16(tmem_base + ((quarter * 32u) << 16) + as * TILE_N + col_in_tile, v);
              ptx::tmem_ld_wait();
              if (c == 3) {
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                  if constexpr (kCG == 1) ptx::mbar_arrive(&tmem_empty_bar[as]);
                  else ptx::mbar_arrive_remote(&tmem_empty_bar[as], 0);
                }
              }
              Epi::template chunk16<c>(ep, st, un, row, nt * TILE_N + (int)col_in_tile, v);
            };
            quarter16(std::integral_constant<int, 0>{}); quarter16(std::integral_constant<int, 1>{});
            quarter16(std::integral_constant<int, 2>{}); quarter16(std::integral_constant<int, 3>{});
          } else
#pragma unroll 1
          for (int c = 0; c < 2; ++c) {
            const uint32_t col_in_tile = colq * 64u + (uint32_t)c * 32u;
            const uint32_t taddr = tmem_base + ((quarter * 32u) << 16) + as * TILE_N + col_in_tile;
            uint32_t v[32];
            ptx::tmem_ld_32x32(taddr, v);
            ptx::tmem_ld_wait();
            if (c == 1) {
              // this warp's last read of the accumulator stage is in registers: hand the stage back to the MMA
              // issuer BEFORE the chunk is processed, so the MMAs of tile t+2 never wait for epilogue math / stores
              ptx::tc_fence_before();
              __syncwarp();
              if (lane == 0) {
                if constexpr (kCG == 1) ptx::mbar_arrive(&tmem_empty_bar[as]);
                else ptx::mbar_arrive_remote(&tmem_empty_bar[as], 0);
              }
            }
            Epi::chunk(ep, st, un, row, nt * TILE_N + (int)col_in_tile, v);
          }
          ++tile_cnt;
        }
      }
      Epi::unit_end(ep, st, un, row0, (int)colq);
    }
    Epi::finish(ep, st, (int)colq);
  }

  // ---------------------------------------------------------------- teardown
  ptx::tc_fence_before();
  if constexpr (kCG == 2) ptx::cluster_sync(); else __syncthreads();
  if (warp == 2) ptx::tmem_dealloc<kCG>(tmem_base, kTmemCols);
}

// =====================================================================================
// Epilogue policies
// =====================================================================================
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr int kColQuarters = 4;      // epilogue column quarters per tile (partials per N split)
constexpr int kMaxExcl = 4;          // same-study columns listed per row; more -> per-element compare path

__device__ __forceinline__ float neg_inf() { return __int_as_float(0xff800000); }

// The negatives mask (main_utils.py:105: study_id[i] != study_id[j]) is sparse: a row is excluded only
// from the few columns that share its study.  A hash pre-pass lists those columns per row
// (excl[row] = up to 4 column indices, -1 padded; n_same[row] = their exact number, own sample
// included), so the epilogue builds a 32-bit exclusion mask per 32-column chunk from 4 compares
// instead of loading and comparing 32 study ids.  Rows with more than 4 listed columns (n_same > 4)
// switch their whole warp to the exact per-element compare path.
struct MaskInfo {
  const int4* excl;      // [rows]
  const int* n_same;     // [rows]
  const int* sid_q;      // [rows]            (per-element path only)
  const int* sid_k;      // [n_ntile * 256]   (padded; per-element path only)
};
struct MaskState { int4 ex; int sidq; bool slow; };

__device__ __forceinline__ void mask_begin(const MaskInfo& mi, MaskState& ms, int row, int q_rows) {
  const bool ok = row < q_rows;
  ms.ex = ok ? __ldg(mi.excl + row) : make_int4(-1, -1, -1, -1);
  const int n = ok ? __ldg(mi.n_same + row) : 0;
  ms.sidq = ok ? __ldg(mi.sid_q + row) : -1;
  ms.slow = __any_sync(0xffffffffu, n > kMaxExcl);
}
// bit c set <=> column col0 + c is excluded for this row (same study, or beyond the last column)
__device__ __forceinline__ uint32_t chunk_mask(const MaskInfo& mi, const MaskState& ms, int col0, int k_cols) {
  uint32_t m = 0;
  if (!ms.slow) {
    const uint32_t d0 = (uint32_t)(ms.ex.x - col0), d1 = (uint32_t)(ms.ex.y - col0);
    const uint32_t d2 = (uint32_t)(ms.ex.z - col0), d3 = (uint32_t)(ms.ex.w - col0);
    if (d0 < 32u) m |= 1u << d0;
    if (d1 < 32u) m |= 1u << d1;
    if (d2 < 32u) m |= 1u << d2;
    if (d3 < 32u) m |= 1u << d3;
  } else {
    const int4* sk4 = reinterpret_cast<const int4*>(mi.sid_k + col0);
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const int4 sk = __ldg(sk4 + g);
      m |= (sk.x == ms.sidq ? 1u : 0u) << (4 * g);
      m |= (sk.y == ms.sidq ? 1u : 0u) << (4 * g + 1);
      m |= (sk.z == ms.sidq ? 1u : 0u) << (4 * g + 2);
      m |= (sk.w == ms.sidq ? 1u : 0u) << (4 * g + 3);
    }
  }
  const int limit = k_cols - col0;                    // columns >= k_cols do not exist
  if (limit < 32) m |= (limit <= 0) ? 0xffffffffu : ~((1u << limit) - 1u);
  return m;
}

// ---- score statistics: per row online (max, sum-exp) over the negatives (the positive-pair scores
//      S[q, q_offset+q] are O(B D) work and come from a separate dot-product kernel)
struct EpiStats {
  static constexpr bool kJoint = false;
  static constexpr bool kWalk = false;
  static constexpr bool kChunk16 = false;
  static constexpr int kEpiSmemBytes = 0;
  struct Params {
    MaskInfo mask;
    int q_rows, k_cols;
    float scale;           // S = scale * acc, scale > 0
    float4* part;          // [n_split][4][rows_padded]  {max (log2 units), sum, 0, 0}
    int rows_padded;
  };
  struct State { uint8_t* stage_smem; MaskState ms; float m, s; };

  static __device__ __forceinline__ void init(const Params&, State&) {}
  static __device__ __forceinline__ void finish(const Params&, State&, int) {}
  static __device__ __forceinline__ void unit_begin(const Params& p, State& st, const Unit&, int row, int) {
    st.m = neg_inf(); st.s = 0.f;
    mask_begin(p.mask, st.ms, row, p.q_rows);
  }
  static __device__ __forceinline__ void chunk(const Params& p, State& st, const Unit&, int row, int col0,
                                               uint32_t (&v)[32]) {
    const float c2 = p.scale * kLog2e;
    const uint32_t mk = chunk_mask(p.mask, st.ms, col0, p.k_cols);
    if (mk != 0u) {                                    // rare: knock the excluded columns out
#pragma unroll
      for (int c = 0; c < 32; ++c) if ((mk >> c) & 1u) v[c] = 0xff800000u;   // -inf
    }
    // max over the chunk (4 independent chains), in accumulator units (scale > 0)
    float m0 = __uint_as_float(v[0]), m1 = __uint_as_float(v[1]), m2 = __uint_as_float(v[2]), m3 = __uint_as_float(v[3]);
#pragma unroll
    for (int c = 4; c < 32; c += 4) {
      m0 = fmaxf(m0, __uint_as_float(v[c])); m1 = fmaxf(m1, __uint_as_float(v[c + 1]));
      m2 = fmaxf(m2, __uint_as_float(v[c + 2])); m3 = fmaxf(m3, __uint_as_float(v[c + 3]));
    }
    const float cm = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)) * c2;
    const float m_new = fmaxf(st.m, cm);
    if (m_new > neg_inf()) {
      float s0 = st.s * ptx::ex2(st.m - m_new), s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
        s0 += ptx::ex2(fmaf(__uint_as_float(v[c]), c2, -m_new));
        s1 += ptx::ex2(fmaf(__uint_as_float(v[c + 1]), c2, -m_new));
        s2 += ptx::ex2(fmaf(__uint_as_float(v[c + 2]), c2, -m_new));
        s3 += ptx::ex2(fmaf(__uint_as_float(v[c + 3]), c2, -m_new));
      }
      st.s = (s0 + s1) + (s2 + s3); st.m = m_new;
    }
  }
  static __device__ __forceinline__ void unit_end(const Params& p, State& st, const Unit& un, int row, int colq) {
    p.part[((size_t)un.s * kColQuarters + colq) * p.rows_padded + row] = make_float4(st.m, st.s, 0.f, 0.f);
  }
};

// ---- row AND column statistics from one score computation (symmetric InfoNCE: both softmax directions).
//      Rows: the lane-local online (max, sum-exp) of EpiStats.  Columns: each warp transposes its 32 x 32 chunk through
//      2 KB of shared memory, 16 columns at a time (conflict-free: 16 B groups XOR-swizzled by the row), so that a lane
//      holds 16 rows of ONE column and max / sum-exp are lane-local again; the two row halves meet in one shuffle.
//      Output: colpart[row block of 32][column] = log2-sum-exp2 of the column over those 32 rows (-inf if all excluded),
//      merged over the row blocks by a small kernel.  S itself is never stored.
struct EpiStatsRC {
  static constexpr bool kJoint = false;
  static constexpr bool kWalk = false;
  static constexpr bool kChunk16 = false;
  static constexpr int kEpiSmemBytes = kNumEpiWarps * 2048;
  struct Params {
    MaskInfo mask;
    int q_rows, k_cols;
    float scale;           // S = scale * acc, scale > 0
    float4* part;          // [n_split][4][rows_padded]  {max (log2 units), sum, 0, 0}
    int rows_padded;
    float* colpart;        // [rows_padded / 32][col_pitch]
    long long col_pitch;
  };
  struct State { uint8_t* stage_smem; MaskState ms; float m, s; };

  static __device__ __forceinline__ void init(const Params&, State&) {}
  static __device__ __forceinline__ void finish(const Params&, State&, int) {}
  static __device__ __forceinline__ void unit_begin(const Params& p, State& st, const Unit&, int row, int) {
    st.m = neg_inf(); st.s = 0.f;
    mask_begin(p.mask, st.ms, row, p.q_rows);
  }
  static __device__ __forceinline__ void chunk(const Params& p, State& st, const Unit&, int row, int col0,
                                               uint32_t (&v)[32]) {
    const float c2 = p.scale * kLog2e;
    const int lane = (int)(threadIdx.x & 31);
    uint32_t mk = chunk_mask(p.mask, st.ms, col0, p.k_cols);
    if (row >= p.q_rows) mk = 0xffffffffu;             // rows beyond the matrix (zero-filled by TMA) take no part
    if (mk != 0u) {
#pragma unroll
      for (int c = 0; c < 32; ++c) if ((mk >> c) & 1u) v[c] = 0xff800000u;   // -inf
    }
    // ---- rows: lane-local online softmax statistics (as EpiStats)
    float m0 = __uint_as_float(v[0]), m1 = __uint_as_float(v[1]), m2 = __uint_as_float(v[2]), m3 = __uint_as_float(v[3]);
#pragma unroll
    for (int c = 4; c < 32; c += 4) {
      m0 = fmaxf(m0, __uint_as_float(v[c])); m1 = fmaxf(m1, __uint_as_float(v[c + 1]));
      m2 = fmaxf(m2, __uint_as_float(v[c + 2])); m3 = fmaxf(m3, __uint_as_float(v[c + 3]));
    }
    const float cm = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)) * c2;
    const float m_new = fmaxf(st.m, cm);
    if (m_new > neg_inf()) {
      float s0 = st.s * ptx::ex2(st.m - m_new), s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
        s0 += ptx::ex2(fmaf(__uint_as_float(v[c]), c2, -m_new));
        s1 += ptx::ex2(fmaf(__uint_as_float(v[c + 1]), c2, -m_new));
        s2 += ptx::ex2(fmaf(__uint_as_float(v[c + 2]), c2, -m_new));
        s3 += ptx::ex2(fmaf(__uint_as_float(v[c + 3]), c2, -m_new));
      }
      st.s = (s0 + s1) + (s2 + s3); st.m = m_new;
    }
    // ---- columns: transpose 16 columns at a time.  Element (r, c) of the half lives at word
    //      r * 16 + 4 * ((c >> 2) ^ ((r >> 1) & 3)) + (c & 3); lane (cc = lane & 15, rh = lane >> 4) reads rows 2t + rh.
    float* sm = reinterpret_cast<float*>(st.stage_smem);
    const int sw = (lane >> 1) & 3;
    const int cc = lane & 15, rh = lane >> 4;
    const int rb = (row - lane) >> 5;                  // 32-row block of this warp
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
      for (int g = 0; g < 4; ++g)
        *reinterpret_cast<uint4*>(sm + lane * 16 + 4 * (g ^ sw)) =
            make_uint4(v[16 * h + 4 * g], v[16 * h + 4 * g + 1], v[16 * h + 4 * g + 2], v[16 * h + 4 * g + 3]);
      __syncwarp();
      float x[16];
#pragma unroll
      for (int t = 0; t < 16; ++t) x[t] = sm[(2 * t + rh) * 16 + 4 * ((cc >> 2) ^ (t & 3)) + (cc & 3)];
      __syncwarp();
      float a0 = fmaxf(x[0], x[1]), a1 = fmaxf(x[2], x[3]), a2 = fmaxf(x[4], x[5]), a3 = fmaxf(x[6], x[7]);
      a0 = fmaxf(a0, fmaxf(x[8], x[9])); a1 = fmaxf(a1, fmaxf(x[10], x[11]));
      a2 = fmaxf(a2, fmaxf(x[12], x[13])); a3 = fmaxf(a3, fmaxf(x[14], x[15]));
      const float mh = fmaxf(fmaxf(a0, a1), fmaxf(a2, a3)) * c2;          // this half's column max (log2 units)
      const float mo = __shfl_xor_sync(0xffffffffu, mh, 16);
      const float mc = fmaxf(mh, mo);                                      // column max over the warp's 32 rows
      float s0 = 0.f, s1 = 0.f;
      if (mc > neg_inf()) {
#pragma unroll
        for (int t = 0; t < 16; t += 2) {
          s0 += ptx::ex2(fmaf(x[t], c2, -mc));
          s1 += ptx::ex2(fmaf(x[t + 1], c2, -mc));
        }
      }
      float sc = s0 + s1;
      sc += __shfl_xor_sync(0xffffffffu, sc, 16);
      if (rh == 0) {
        const float l2 = (mc > neg_inf() && sc > 0.f) ? mc + __log2f(sc) : neg_inf();
        p.colpart[(size_t)rb * p.col_pitch + col0 + 16 * h + cc] = l2;
      }
    }
  }
  static __device__ __forceinline__ void unit_end(const Params& p, State& st, const Unit& un, int row, int colq) {
    p.part[((size_t)un.s * kColQuarters + colq) * p.rows_padded + row] = make_float4(st.m, st.s, 0.f, 0.f);
  }
};

// ---- dS panel: P[row, col] = incl * ( wq e^{S - refq[row]} + wk e^{S - refk[col]} ), bf16 (hi [+ lo])
// Each epilogue warp stages its 32 rows x 32 columns (2 KB, 16 B chunks XOR-swizzled by the row = TMA SWIZZLE_64B) in
// shared memory and ONE lane hands the tile to the TMA engine (cp.async.bulk.tensor store): no per-thread global stores,
// no address arithmetic, rows beyond the panel clipped by the tensor map.
struct EpiPStore {
  static constexpr bool kJoint = false;
  static constexpr bool kWalk = false;
  static constexpr bool kChunk16 = false;
  static constexpr int kEpiSmemBytes = kNumEpiWarps * 2048;
  struct Params {
    alignas(64) CUtensorMap tmap_p;   // the panel [q_rows, pitch] bf16, box 32 x 32, SWIZZLE_64B
    MaskInfo mask;
    int q_rows, k_cols;
    long long q_offset;
    float scale;
    const float* refq;      // [q_rows] natural-log reference per row (used when use_q)
    float ln_wq;            // ln(weight) of the row term
    int use_q;
    const float* refk2;     // [n_ntile*256] (padded) column reference, log2 units, weight folded in
    int use_k;
    int include_diag;       // 1: the positive pair is part of the softmax (InfoNCE), 0: negatives only (DV)
    int lo_col0;            // strict mode: the residual panel starts at this column of the same rows (0: none)
    // single-pass mode: refq is a per-row UPPER BOUND of the scores, so P <= 1 needs no running max; the
    // row sums of P (fp32, before rounding) are the statistics: sum_part[n_split][4][rows_padded]
    float* sum_part;
    int rows_padded;
  };
  struct State { uint8_t* stage_smem; MaskState ms; float rq2; float s; };

  static __device__ __forceinline__ void init(const Params&, State&) {}
  static __device__ __forceinline__ void finish(const Params&, State&, int) {
    if ((threadIdx.x & 31) == 0) ptx::tma_store_wait_all();          // this lane issued the warp's stores
  }
  static __device__ __forceinline__ void unit_begin(const Params& p, State& st, const Unit&, int row, int) {
    st.s = 0.f;
    mask_begin(p.mask, st.ms, row, p.q_rows);
    const float r = (p.use_q && row < p.q_rows) ? __ldg(p.refq + row) : 0.f;
    st.rq2 = (r - p.ln_wq) * kLog2e;
  }
  // stage this thread's 32 packed bf16 (16 words = 4 x 16 B) into its row of the warp's 32 x 64 B tile (the TMA
  // SWIZZLE_64B pattern: 16 B chunk index ^= (row >> 1) & 3), then lane 0 issues the tile store at (col, row0)
  static __device__ __forceinline__ void stage_and_store(const Params& p, uint8_t* smem, int lane, const uint32_t (&w)[16],
                                                         int col, int row0) {
    if (lane == 0) ptx::tma_store_wait_read();         // the previous store of this warp has drained the buffer
    __syncwarp();
    const int sw = (lane >> 1) & 3;
#pragma unroll
    for (int g = 0; g < 4; ++g)
      *reinterpret_cast<uint4*>(smem + lane * 64 + ((g ^ sw) * 16)) = make_uint4(w[4 * g], w[4 * g + 1], w[4 * g + 2], w[4 * g + 3]);
    ptx::fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0 && row0 < p.q_rows) {
      ptx::tma_store_2d(&p.tmap_p, ptx::smem_u32(smem), col, row0);
      ptx::tma_store_commit();
    }
  }
  static __device__ __forceinline__ void chunk(const Params& p, State& st, const Unit&, int row, int col0,
                                               uint32_t (&v)[32]) {
    const float c2 = p.scale * kLog2e;
    const int lane = (int)(threadIdx.x & 31);
    uint32_t mk = chunk_mask(p.mask, st.ms, col0, p.k_cols);
    if (p.include_diag) {                              // the positive pair stays in
      const long long dcol = p.q_offset + row - col0;
      if (dcol >= 0 && dcol < 32) mk &= ~(1u << (int)dcol);
    }
    // v[c] <- p value (fp32 bits), in place
    if (p.use_q && !p.use_k) {
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] = __float_as_uint(ptx::ex2(fmaf(__uint_as_float(v[c]), c2, -st.rq2)));
    } else {
      const float4* rk4 = reinterpret_cast<const float4*>(p.refk2 + col0);
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const float4 rk = __ldg(rk4 + g);
        const float rks[4] = {rk.x, rk.y, rk.z, rk.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = 4 * g + j;
          const float a = __uint_as_float(v[c]);
          float val = ptx::ex2(fmaf(a, c2, -rks[j]));
          if (p.use_q) val += ptx::ex2(fmaf(a, c2, -st.rq2));
          v[c] = __float_as_uint(val);
        }
      }
    }
    if (mk != 0u) {
#pragma unroll
      for (int c = 0; c < 32; ++c) if ((mk >> c) & 1u) v[c] = 0u;
    }
    if (p.sum_part != nullptr) {
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
        s0 += __uint_as_float(v[c]); s1 += __uint_as_float(v[c + 1]);
        s2 += __uint_as_float(v[c + 2]); s3 += __uint_as_float(v[c + 3]);
      }
      st.s += (s0 + s1) + (s2 + s3);
    }
    uint32_t hi[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) hi[c] = ptx::pack_bf16(__uint_as_float(v[2 * c]), __uint_as_float(v[2 * c + 1]));
    const int row0 = row - lane;                       // first row of this warp
    stage_and_store(p, st.stage_smem, lane, hi, col0, row0);
    if (p.lo_col0 > 0) {                               // strict mode: residual panel, lo_col0 columns to the right
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        const float h0 = __uint_as_float(hi[c] << 16), h1 = __uint_as_float(hi[c] & 0xffff0000u);
        hi[c] = ptx::pack_bf16(__uint_as_float(v[2 * c]) - h0, __uint_as_float(v[2 * c + 1]) - h1);
      }
      stage_and_store(p, st.stage_smem, lane, hi, col0 + p.lo_col0, row0);
    }
  }
  static __device__ __forceinline__ void unit_end(const Params& p, State& st, const Unit& un, int row, int colq) {
    if (p.sum_part != nullptr) p.sum_part[((size_t)un.s * kColQuarters + colq) * p.rows_padded + row] = st.s;
  }
};

__device__ __forceinline__ float rcp_approx(float x) {
  float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
}
// log1p(e) for e in [0, 1]: degree-8 polynomial e * p(e) on the FMA pipe, |error| < 2e-7 in fp32 (fitted to log1p on [0, 1])
__device__ __forceinline__ float log1p_unit(float e) {
  float p = -0.006472604814916849f;
  p = fmaf(p, e, 0.03617211803793907f);
  p = fmaf(p, e, -0.09547846019268036f);
  p = fmaf(p, e, 0.16779260337352753f);
  p = fmaf(p, e, -0.2408052682876587f);
  p = fmaf(p, e, 0.331819087266922f);
  p = fmaf(p, e, -0.49987688660621643f);
  p = fmaf(p, e, 0.999996542930603f);
  return p * e;
}

// ---- Jensen-Shannon dS panel: P[row, col] = M sigma(S) (bf16 hi [+ lo], stored as EpiPStore does) and the fp32 row sums of
//      M softplus(S) (sum_part; the loss).  Per score: one MUFU.EX2 (e = e^{-|S|}), one MUFU.RCP (r = 1 / (1 + e)),
//      sigma(S) = r (S >= 0) or e r, softplus(S) = max(S, 0) + log1p(e) with log1p as a polynomial on the FMA pipe.  Safe for
//      any finite S (e in [0, 1]).  The weights lie in (0, 1): no reference, no running maximum, no guard.
//      kStore = false: the row sums only (forward-only calls), no panel.  Params as EpiPStore (refq / refk2 / include_diag unused).
template <bool kStore>
struct EpiJS {
  static constexpr bool kJoint = false;
  static constexpr bool kWalk = false;
  static constexpr bool kChunk16 = false;
  static constexpr int kEpiSmemBytes = kStore ? kNumEpiWarps * 2048 : 0;
  using Params = EpiPStore::Params;
  struct State { uint8_t* stage_smem; MaskState ms; float s; };

  static __device__ __forceinline__ void init(const Params&, State&) {}
  static __device__ __forceinline__ void finish(const Params&, State&, int) {
    if (kStore && (threadIdx.x & 31) == 0) ptx::tma_store_wait_all();
  }
  static __device__ __forceinline__ void unit_begin(const Params& p, State& st, const Unit&, int row, int) {
    st.s = 0.f;
    mask_begin(p.mask, st.ms, row, p.q_rows);
  }
  static __device__ __forceinline__ void chunk(const Params& p, State& st, const Unit&, int row, int col0,
                                               uint32_t (&v)[32]) {
    const float sc = p.scale, c2 = -p.scale * kLog2e;   // scale > 0: |S| log2 e = |acc| scale log2 e
    const int lane = (int)(threadIdx.x & 31);
    const uint32_t mk = chunk_mask(p.mask, st.ms, col0, p.k_cols);
    const bool split = kStore && p.lo_col0 > 0;        // strict mode: residual panel, lo_col0 columns to the right
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    uint32_t hi[16], lo[16];
    // pairs of scores, packed as soon as they are formed (v dies as hi / lo fill: no spills at 96 registers)
#pragma unroll
    for (int c = 0; c < 32; c += 2) {
      float sig[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const float a = __uint_as_float(v[c + j]);
        const float e = ptx::ex2(fabsf(a) * c2);
        float sp = fmaf(fmaxf(a, 0.f), sc, log1p_unit(e));
        if constexpr (kStore) {
          const float r = rcp_approx(1.f + e);
          sig[j] = a >= 0.f ? r : e * r;
        }
        if ((mk >> (c + j)) & 1u) { sig[j] = 0.f; sp = 0.f; }
        s[(c + j) & 3] += sp;
      }
      if constexpr (kStore) {
        const uint32_t h = ptx::pack_bf16(sig[0], sig[1]);
        hi[c / 2] = h;
        if (split) lo[c / 2] = ptx::pack_bf16(sig[0] - __uint_as_float(h << 16), sig[1] - __uint_as_float(h & 0xffff0000u));
      }
    }
    st.s += (s[0] + s[1]) + (s[2] + s[3]);
    if constexpr (kStore) {
      const int row0 = row - lane;
      EpiPStore::stage_and_store(p, st.stage_smem, lane, hi, col0, row0);
      if (split) EpiPStore::stage_and_store(p, st.stage_smem, lane, lo, col0 + p.lo_col0, row0);
    }
  }
  static __device__ __forceinline__ void unit_end(const Params& p, State& st, const Unit& un, int row, int colq) {
    p.sum_part[((size_t)un.s * kColQuarters + colq) * p.rows_padded + row] = st.s;
  }
};

// ---- plain GEMM epilogue: C = alpha * (ACC - gamma * SUB) [+ C_prev]
struct EpiStore {
  static constexpr bool kJoint = false;
  static constexpr bool kWalk = false;
  static constexpr bool kChunk16 = false;
  static constexpr int kEpiSmemBytes = 0;
  struct Params {
    float* out_f32;            // optional
    __nv_bfloat16* out_bf16;   // optional
    __nv_bfloat16* out_bf16_lo;  // optional residual bf16(C - hi) (hi/lo split output), same pitch
    long long ld_out;          // pitch of out_f32
    long long ld_out16;        // pitch of out_bf16 / out_bf16_lo
    int rows, cols;
    float alpha, gamma;
    const __nv_bfloat16* sub;  // optional [sub_rows, ld_sub]
    const __nv_bfloat16* sub_lo;  // optional residual of SUB (SUB = sub + sub_lo), same pitch
    long long ld_sub;
    int sub_row0, sub_rows;    // SUB row r applies to output row sub_row0 + r, r in [0, sub_rows)
    long long ksplit_stride;   // elements between split-K partial outputs (fp32 only)
    int accumulate;            // out_f32 += result (panel-by-panel accumulation)
    int acc_first;             // with `accumulate`: C = alpha * (kappa * (ACC + C_prev) - gamma SUB) — the last panel of an
    const float* kappa_a;      // accumulation finishes the result; kappa = exp(kappa_a[0] - kappa_b[0]) (device scalars) or 1
    const float* kappa_b;
    const float* bias;         // optional [cols]: C = alpha * (ACC - gamma SUB) + bias   (nn.Linear bias)
    const __nv_bfloat16* relu_mask;  // optional [rows, ld_mask]: C = 0 where relu_mask <= 0  (backward of a ReLU whose
    long long ld_mask;               //                          output is relu_mask)
  };
  struct State { uint8_t* stage_smem; };
  static __device__ __forceinline__ void init(const Params&, State&) {}
  static __device__ __forceinline__ void finish(const Params&, State&, int) {}
  static __device__ __forceinline__ void unit_begin(const Params&, State&, const Unit&, int, int) {}
  static __device__ __forceinline__ void chunk(const Params& p, State&, const Unit& un, int row, int col0,
                                               uint32_t (&v)[32]) {
    if (row >= p.rows || col0 >= p.cols) return;
    float o[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) o[c] = __uint_as_float(v[c]);
    const bool full = (col0 + 32 <= p.cols);
    const bool acc_first = p.acc_first != 0 && p.out_f32 != nullptr;
    if (acc_first) {
      const float* d = p.out_f32 + (size_t)un.ks * p.ksplit_stride + (size_t)row * p.ld_out + col0;
      const float kappa = p.kappa_a != nullptr ? expf(__ldg(p.kappa_a) - __ldg(p.kappa_b)) : 1.f;
      if (p.accumulate) {
        if (full) {
          const float4* d4 = reinterpret_cast<const float4*>(d);
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float4 prev = d4[g];
            o[4 * g] += prev.x; o[4 * g + 1] += prev.y; o[4 * g + 2] += prev.z; o[4 * g + 3] += prev.w;
          }
        } else {
          for (int c = 0; c < 32; ++c) if (col0 + c < p.cols) o[c] += d[c];
        }
      }
#pragma unroll
      for (int c = 0; c < 32; ++c) o[c] *= kappa;
    }
    const int srow = row - p.sub_row0;
    if (p.sub != nullptr && srow >= 0 && srow < p.sub_rows) {
      const __nv_bfloat16* s = p.sub + (size_t)srow * p.ld_sub + col0;
      if (full) {
        const uint4* s4 = reinterpret_cast<const uint4*>(s);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const uint4 q = __ldg(s4 + g);
          const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            o[g * 8 + 2 * j]     -= p.gamma * __uint_as_float(w[j] << 16);
            o[g * 8 + 2 * j + 1] -= p.gamma * __uint_as_float(w[j] & 0xffff0000u);
          }
        }
      } else {
        for (int c = 0; c < 32; ++c) if (col0 + c < p.cols) o[c] -= p.gamma * __bfloat162float(s[c]);
      }
      if (p.sub_lo != nullptr) {
        const __nv_bfloat16* sl = p.sub_lo + (size_t)srow * p.ld_sub + col0;
        for (int c = 0; c < 32; ++c) if (col0 + c < p.cols) o[c] -= p.gamma * __bfloat162float(sl[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < 32; ++c) o[c] *= p.alpha;
    if (p.bias != nullptr) {
      if (full) {
        const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const float4 b = __ldg(b4 + g);
          o[4 * g] += b.x; o[4 * g + 1] += b.y; o[4 * g + 2] += b.z; o[4 * g + 3] += b.w;
        }
      } else {
        for (int c = 0; c < 32; ++c) if (col0 + c < p.cols) o[c] += p.bias[col0 + c];
      }
    }
    if (p.relu_mask != nullptr) {
      const __nv_bfloat16* m = p.relu_mask + (size_t)row * p.ld_mask + col0;
      if (full) {
        const uint4* m4 = reinterpret_cast<const uint4*>(m);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const uint4 q = __ldg(m4 + g);
          const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {       // bf16 > 0  <=>  sign clear and magnitude non-zero
            if (!(__uint_as_float(w[j] << 16) > 0.f)) o[g * 8 + 2 * j] = 0.f;
            if (!(__uint_as_float(w[j] & 0xffff0000u) > 0.f)) o[g * 8 + 2 * j + 1] = 0.f;
          }
        }
      } else {
        for (int c = 0; c < 32; ++c) if (col0 + c < p.cols && !(__bfloat162float(m[c]) > 0.f)) o[c] = 0.f;
      }
    }
    if (p.out_f32 != nullptr) {
      float* d = p.out_f32 + (size_t)un.ks * p.ksplit_stride + (size_t)row * p.ld_out + col0;
      if (full) {
        float4* d4 = reinterpret_cast<float4*>(d);
        if (p.accumulate && !acc_first) {
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float4 prev = d4[g];
            o[4 * g] += prev.x; o[4 * g + 1] += prev.y; o[4 * g + 2] += prev.z; o[4 * g + 3] += prev.w;
          }
        }
#pragma unroll
        for (int g = 0; g < 8; ++g) d4[g] = make_float4(o[4 * g], o[4 * g + 1], o[4 * g + 2], o[4 * g + 3]);
      } else {
        for (int c = 0; c < 32; ++c) if (col0 + c < p.cols) { if (p.accumulate && !acc_first) o[c] += d[c]; d[c] = o[c]; }
      }
    }
    if (p.out_bf16 != nullptr) {
      __nv_bfloat16* d = p.out_bf16 + (size_t)row * p.ld_out16 + col0;
      uint32_t hi[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) hi[c] = ptx::pack_bf16(o[2 * c], o[2 * c + 1]);
      if (full) {
        uint4* d4 = reinterpret_cast<uint4*>(d);
#pragma unroll
        for (int g = 0; g < 4; ++g) d4[g] = make_uint4(hi[4 * g], hi[4 * g + 1], hi[4 * g + 2], hi[4 * g + 3]);
      } else {
        for (int c = 0; c < 32; ++c) if (col0 + c < p.cols) d[c] = __float2bfloat16(o[c]);
      }
      if (p.out_bf16_lo != nullptr) {
        __nv_bfloat16* dl = p.out_bf16_lo + (size_t)row * p.ld_out16 + col0;
        uint32_t lo[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const float h0 = __uint_as_float(hi[c] << 16), h1 = __uint_as_float(hi[c] & 0xffff0000u);
          lo[c] = ptx::pack_bf16(o[2 * c] - h0, o[2 * c + 1] - h1);
        }
        if (full) {
          uint4* d4 = reinterpret_cast<uint4*>(dl);
#pragma unroll
          for (int g = 0; g < 4; ++g) d4[g] = make_uint4(lo[4 * g], lo[4 * g + 1], lo[4 * g + 2], lo[4 * g + 3]);
        } else {
          for (int c = 0; c < 32; ++c)
            if (col0 + c < p.cols) dl[c] = __float2bfloat16(o[c] - __bfloat162float(__float2bfloat16(o[c])));
        }
      }
    }
  }
  static __device__ __forceinline__ void unit_end(const Params&, State&, const Unit&, int, int) {}
};

// =====================================================================================
// Concat-MLP critic (the reference's make_mlp(2D, [H1, H2]), model.py:18-32): the accumulator tile is
// Z2[pair, n] = sum_k H1act[pair, k] W2[n, k]; rows are (image i, text j) pairs, columns the H2 hidden units.
// =====================================================================================
// column sums over the 32 lanes (rows) of a warp: in: v[c] = this row's value of column c; out: lane l holds
// sum over rows of column l.  Butterfly that halves the live values per step: 31 shuffles instead of 160.
__device__ __forceinline__ float warp_column_sums(float (&v)[32], int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int c = 0; c < s; ++c) {
      // lanes with bit s keep the upper half [s, 2s), the others the lower half [0, s)
      const float send = up ? v[c] : v[c + s];
      const float keep = up ? v[c + s] : v[c];
      v[c] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
  return v[0];      // column index = lane (bit s of the lane selected the half at every step)
}

// the same for 16 columns: lanes l and l ^ 16 both end with the sum over the 32 rows of column (l & 15)
__device__ __forceinline__ float warp_column_sums16(float (&v)[16], int lane) {
#pragma unroll
  for (int s = 8; s >= 1; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int c = 0; c < s; ++c) {
      const float send = up ? v[c] : v[c + s];
      const float keep = up ? v[c + s] : v[c];
      v[c] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 16);
}

// ---- forward: logit[pair] = b3 + sum_n w3[n] relu(Z2[pair, n] + b2[n]); each epilogue warp owns a 64-column
//      quarter of every 256-column tile, so it writes one partial per (pair, column quarter)
struct EpiMlpFwd {
  static constexpr bool kJoint = false;
  static constexpr bool kWalk = false;
  static constexpr bool kChunk16 = false;
  static constexpr int kEpiSmemBytes = 0;
  struct Params {
    const float* b2;       // [n_ntile * 256] zero padded
    const float* w3;       // [n_ntile * 256] zero padded
    float* part;           // [kColQuarters][rows_padded]
    int rows_padded;
  };
  struct State { uint8_t* stage_smem; float acc; };
  static __device__ __forceinline__ void init(const Params&, State&) {}
  static __device__ __forceinline__ void finish(const Params&, State&, int) {}
  static __device__ __forceinline__ void unit_begin(const Params&, State& st, const Unit&, int, int) { st.acc = 0.f; }
  static __device__ __forceinline__ void chunk(const Params& p, State& st, const Unit&, int, int col0, uint32_t (&v)[32]) {
    const float4* b4 = reinterpret_cast<const float4*>(p.b2 + col0);
    const float4* w4 = reinterpret_cast<const float4*>(p.w3 + col0);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const float4 b = __ldg(b4 + g), w = __ldg(w4 + g);
      a0 = fmaf(w.x, fmaxf(__uint_as_float(v[4 * g]) + b.x, 0.f), a0);
      a1 = fmaf(w.y, fmaxf(__uint_as_float(v[4 * g + 1]) + b.y, 0.f), a1);
      a2 = fmaf(w.z, fmaxf(__uint_as_float(v[4 * g + 2]) + b.z, 0.f), a2);
      a3 = fmaf(w.w, fmaxf(__uint_as_float(v[4 * g + 3]) + b.w, 0.f), a3);
    }
    st.acc += (a0 + a1) + (a2 + a3);
  }
  static __device__ __forceinline__ void unit_end(const Params& p, State& st, const Unit&, int row, int colq) {
    p.part[(size_t)colq * p.rows_padded + row] = st.acc;
  }
};

// ---- backward through layer 3 / ReLU 2:  dZ2[pair, n] = g[pair] w3[n] [Z2 + b2 > 0]  (bf16 hi [+ lo]) for the
//      dW2 / dH1 contractions;  dw3[n] += sum_pairs g relu(Z2 + b2),  db2[n] += sum_pairs dZ2  (column sums over
//      the warp's rows, kept per lane across the whole launch, one atomicAdd per column at the end).
struct EpiMlpDzParams {
  const float* b2;       // [n_ntile * 256] zero padded
  const float* w3;       // [n_ntile * 256] zero padded
  const float* g;        // [rows] dL/dlogit of the pair
  int rows, cols;
  __nv_bfloat16* dz;     // [rows, pitch]
  __nv_bfloat16* dz_lo;  // residual half (strict), second piece (fp32 mode) or nullptr
  __nv_bfloat16* dz_lo2; // third piece (fp32 mode) or nullptr
  long long pitch;
  float* dw3;            // [n_ntile * 256] accumulators (atomicAdd)
  float* db2;
};
// kThird: fp32 mode (three-piece dZ2 stores); the fast / strict instantiation carries none of that code
template <bool kThird>
struct EpiMlpDzT {
  static constexpr bool kJoint = false;
  static constexpr bool kWalk = false;
  static constexpr bool kChunk16 = false;
  static constexpr int kEpiSmemBytes = 0;
  static constexpr int kMaxTiles = 2;       // H2 <= 512
  using Params = EpiMlpDzParams;
  struct State { uint8_t* stage_smem; float g; float sw[kMaxTiles][2]; float sb[kMaxTiles][2]; };
  static __device__ __forceinline__ void init(const Params&, State& st) {
#pragma unroll
    for (int t = 0; t < kMaxTiles; ++t) { st.sw[t][0] = st.sw[t][1] = 0.f; st.sb[t][0] = st.sb[t][1] = 0.f; }
  }
  static __device__ __forceinline__ void unit_begin(const Params& p, State& st, const Unit&, int row, int) {
    st.g = row < p.rows ? __ldg(p.g + row) : 0.f;
  }
  static __device__ __forceinline__ void chunk(const Params& p, State& st, const Unit&, int row, int col0, uint32_t (&v)[32]) {
    const int lane = (int)(threadIdx.x & 31);
    const float4* b4 = reinterpret_cast<const float4*>(p.b2 + col0);
    const float4* w4 = reinterpret_cast<const float4*>(p.w3 + col0);
    float dz[32];
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const float4 b = __ldg(b4 + g), w = __ldg(w4 + g);
      const float bb[4] = {b.x, b.y, b.z, b.w}, ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float z = __uint_as_float(v[4 * g + j]) + bb[j];
        dz[4 * g + j] = z > 0.f ? st.g * ww[j] : 0.f;                       // padded columns: w3 = 0
        v[4 * g + j] = __float_as_uint(z > 0.f ? st.g * z : 0.f);             // g relu(z2): the dw3 summand
      }
    }
    if (row < p.rows && col0 < p.cols) {
      uint32_t hi[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) hi[c] = ptx::pack_bf16(dz[2 * c], dz[2 * c + 1]);
      const bool full = col0 + 32 <= p.cols;
      __nv_bfloat16* d = p.dz + (size_t)row * p.pitch + col0;
      if (full) {
        uint4* d4 = reinterpret_cast<uint4*>(d);
#pragma unroll
        for (int g = 0; g < 4; ++g) d4[g] = make_uint4(hi[4 * g], hi[4 * g + 1], hi[4 * g + 2], hi[4 * g + 3]);
      } else {
        for (int c = 0; c < 32; ++c) if (col0 + c < p.cols) d[c] = __float2bfloat16(dz[c]);
      }
      if (p.dz_lo != nullptr) {
        __nv_bfloat16* dl = p.dz_lo + (size_t)row * p.pitch + col0;
        uint32_t lo[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const float h0 = __uint_as_float(hi[c] << 16), h1 = __uint_as_float(hi[c] & 0xffff0000u);
          lo[c] = ptx::pack_bf16(dz[2 * c] - h0, dz[2 * c + 1] - h1);
        }
        if (full) {
          uint4* d4 = reinterpret_cast<uint4*>(dl);
#pragma unroll
          for (int g = 0; g < 4; ++g) d4[g] = make_uint4(lo[4 * g], lo[4 * g + 1], lo[4 * g + 2], lo[4 * g + 3]);
        } else {
          for (int c = 0; c < 32; ++c)
            if (col0 + c < p.cols) dl[c] = __float2bfloat16(dz[c] - __bfloat162float(__float2bfloat16(dz[c])));
        }
        if (kThird && p.dz_lo2 != nullptr) {          // fp32 mode: the third piece (dz - hi) - lo, both differences exact
          __nv_bfloat16* d2 = p.dz_lo2 + (size_t)row * p.pitch + col0;
          if (full) {
            uint32_t l2[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) {
              const float r0 = dz[2 * c] - __uint_as_float(hi[c] << 16), r1 = dz[2 * c + 1] - __uint_as_float(hi[c] & 0xffff0000u);
              l2[c] = ptx::pack_bf16(r0 - __uint_as_float(lo[c] << 16), r1 - __uint_as_float(lo[c] & 0xffff0000u));
            }
            uint4* d4 = reinterpret_cast<uint4*>(d2);
#pragma unroll
            for (int g = 0; g < 4; ++g) d4[g] = make_uint4(l2[4 * g], l2[4 * g + 1], l2[4 * g + 2], l2[4 * g + 3]);
          } else {
            for (int c = 0; c < 32; ++c)
              if (col0 + c < p.cols) {
                const float r = dz[c] - __bfloat162float(__float2bfloat16(dz[c]));
                d2[c] = __float2bfloat16(r - __bfloat162float(__float2bfloat16(r)));
              }
          }
        }
      }
    }
    // column sums over this warp's 32 pairs (rows beyond p.rows carry g = 0)
    const float cb = warp_column_sums(dz, lane);
    float hw[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) hw[c] = __uint_as_float(v[c]);
    const float cw = warp_column_sums(hw, lane);
    const int t = col0 >> 8, h = (col0 >> 5) & 1;
#pragma unroll
    for (int tt = 0; tt < kMaxTiles; ++tt)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh)
        if (tt == t && hh == h) { st.sb[tt][hh] += cb; st.sw[tt][hh] += cw; }
  }
  static __device__ __forceinline__ void unit_end(const Params&, State&, const Unit&, int, int) {}
  static __device__ __forceinline__ void finish(const Params& p, State& st, int colq) {
    const int lane = (int)(threadIdx.x & 31);
#pragma unroll
    for (int t = 0; t < kMaxTiles; ++t)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int col = t * TILE_N + colq * 64 + h * 32 + lane;
        if (col < p.cols && (st.sb[t][h] != 0.f || st.sw[t][h] != 0.f)) {
          atomicAdd(p.db2 + col, st.sb[t][h]);
          atomicAdd(p.dw3 + col, st.sw[t][h]);
        }
      }
  }
};
using EpiMlpDz = EpiMlpDzT<false>;
using EpiMlpDz3 = EpiMlpDzT<true>;

// ---- single pass (dv-like estimators): forward AND the backward through layer 3 / ReLU 2 from ONE Z2 accumulator.
//      The softmax weights of the negatives are taken relative to a reference logit `ref` that is fixed BEFORE the
//      pass (g~ = incl e^{S - ref}; every gradient is linear in g~, the caller multiplies by e^{ref - LSE} at the end),
//      so nothing has to wait for the global log-sum-exp and Z2 is never recomputed.
//      Rows are pairs in the padded panel order p = il * Bp + j (Bp = B rounded up to the M block): an M block has ONE
//      image row i = r0 + il and consecutive text columns j.  The image rows may be a block of a larger batch (sharded
//      step): local row i is global row q_off + i, so its positive pair is text column j = q_off + i.  Joint policy: pass1 forms this warp's share of the logit
//      (64 of the up to 512 columns per tile), `mid` adds the four column quarters through shared memory (one named
//      barrier of the 16 epilogue warps per unit, double-buffered slots), derives g~ and the row statistics, and the
//      second pass is EpiMlpDz's chunk with that g~.
constexpr float kMlpSpScale = 1.6940658945086007e-21f;    // 2^-69: g~ = e^{S - max_sample} 2^-69
constexpr double kMlpSpMargin = 47.82715406979468;        // 69 ln 2
struct EpiMlpSpParams {
  const float* b2;       // [n_ntile * 256] zero padded
  const float* w3;       // [n_ntile * 256] zero padded
  const float* b3;       // [1]
  const float* ref;      // [1] maximum logit of the sample (the reference logit is this + kMlpSpMargin)
  const int* sid_q;      // [rows] study ids of the image rows (negatives: sid_q[i] != sid_k[j], main_utils.py:105)
  const int* sid_k;      // [B] study ids of the text rows
  int B, Bp, r0, rr;     // text rows, padded text rows, first image row of the panel, image rows in the panel
  int q_off;             // global index of local image row 0
  int cols;              // H2
  __nv_bfloat16* dz;     // [rr * Bp, pitch]  g~ w3 [Z2 + b2 > 0]
  __nv_bfloat16* dz_lo;  // residual half (strict), second piece (fp32 mode) or nullptr
  __nv_bfloat16* dz_lo2; // third piece (fp32 mode) or nullptr
  long long pitch;
  float* dw3;            // [n_ntile * 256] accumulators (atomicAdd), in g~ units
  float* db2;
  float* rowsum;         // [rows] += sum_j g~          (atomicAdd)
  float* rowcnt;         // [rows] += number of negatives of the row
  float* diag_out;       // [rows] logit of the positive pair
  float* S_out;          // optional [rows, B]: every logit
};
// kThird: fp32 mode (three-piece dZ2 stores); the fast / strict instantiation carries none of that code
template <bool kThird>
struct EpiMlpSpT {
  static constexpr bool kJoint = true;
  static constexpr bool kWalk = false;
  static constexpr bool kChunk16 = false;
  static constexpr int kEpiSmemBytes = 2 * kColQuarters * BLOCK_M * 4;     // 2 slots x [4 column quarters][128 rows] fp32
  static constexpr int kMaxTiles = 2;       // H2 <= 512
  using Params = EpiMlpSpParams;
  struct State { uint8_t* stage_smem; float acc; float g; int slot; float sw[kMaxTiles][2]; float sb[kMaxTiles][2]; };
  static __device__ __forceinline__ void init(const Params&, State& st) {
    st.slot = 0;
#pragma unroll
    for (int t = 0; t < kMaxTiles; ++t) { st.sw[t][0] = st.sw[t][1] = 0.f; st.sb[t][0] = st.sb[t][1] = 0.f; }
  }
  static __device__ __forceinline__ void unit_begin(const Params&, State& st, const Unit&, int, int) { st.acc = 0.f; }
  static __device__ __forceinline__ void pass1(const Params& p, State& st, int col0, uint32_t (&v)[32]) {
    const float4* b4 = reinterpret_cast<const float4*>(p.b2 + col0);
    const float4* w4 = reinterpret_cast<const float4*>(p.w3 + col0);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const float4 b = __ldg(b4 + g), w = __ldg(w4 + g);
      a0 = fmaf(w.x, fmaxf(__uint_as_float(v[4 * g]) + b.x, 0.f), a0);
      a1 = fmaf(w.y, fmaxf(__uint_as_float(v[4 * g + 1]) + b.y, 0.f), a1);
      a2 = fmaf(w.z, fmaxf(__uint_as_float(v[4 * g + 2]) + b.z, 0.f), a2);
      a3 = fmaf(w.w, fmaxf(__uint_as_float(v[4 * g + 3]) + b.w, 0.f), a3);
    }
    st.acc += (a0 + a1) + (a2 + a3);
  }
  static __device__ __forceinline__ void mid(const Params& p, State& st, const Unit&, int row, int colq, uint8_t* epi_smem) {
    const int lane = (int)(threadIdx.x & 31);
    const int r = (int)(((threadIdx.x >> 5) & 3u) * 32u) + lane;            // row inside the CTA's 128
    float* slot = reinterpret_cast<float*>(epi_smem) + st.slot * (kColQuarters * BLOCK_M);
    slot[colq * BLOCK_M + r] = st.acc;
    ptx::named_bar_sync(1, kNumEpiWarps * 32);
    // every warp adds the quarters in the same order: the four threads of a row agree bit for bit
    const float S = __ldg(p.b3) + ((slot[r] + slot[BLOCK_M + r]) + (slot[2 * BLOCK_M + r] + slot[3 * BLOCK_M + r]));
    st.slot ^= 1;       // the next unit writes the other slot; this one is rewritten two barriers from now
    const int il = row / p.Bp, j = row - il * p.Bp, i = p.r0 + il;
    const bool valid = j < p.B && il < p.rr;
    const bool incl = valid && __ldg(p.sid_q + i) != __ldg(p.sid_k + j);
    // e^{S - ref} with ref = (sample maximum) + 69 ln 2: the subtraction stays near the logits (no absolute rounding at
    // the size of the margin) and the margin is an exact power of two
    const float g = incl ? expf(S - __ldg(p.ref)) * kMlpSpScale : 0.f;
    st.g = g;
    if (colq == 0) {
      if (valid) {
        if (p.S_out != nullptr) p.S_out[(size_t)i * p.B + j] = S;
        if (j == p.q_off + i) p.diag_out[i] = S;
      }
      float gs = g;
#pragma unroll
      for (int o = 16; o; o >>= 1) gs += __shfl_xor_sync(0xffffffffu, gs, o);
      const int cnt = __popc(__ballot_sync(0xffffffffu, incl));
      if (lane == 0 && il < p.rr && cnt > 0) {        // the warp's 32 rows share the image row i
        atomicAdd(p.rowsum + i, gs);
        atomicAdd(p.rowcnt + i, (float)cnt);
      }
    }
  }
  // second pass over 16 columns (kQ = piece of the thread's 64 columns)
  template <int kQ>
  static __device__ __forceinline__ void chunk16(const Params& p, State& st, const Unit&, int row, int col0, uint32_t (&v)[16]) {
    const int lane = (int)(threadIdx.x & 31);
    const float4* b4 = reinterpret_cast<const float4*>(p.b2 + col0);
    const float4* w4 = reinterpret_cast<const float4*>(p.w3 + col0);
    float dz[16], hw[16];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const float4 b = __ldg(b4 + g), w = __ldg(w4 + g);
      const float bb[4] = {b.x, b.y, b.z, b.w}, ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float z = __uint_as_float(v[4 * g + j]) + bb[j];
        dz[4 * g + j] = z > 0.f ? st.g * ww[j] : 0.f;                       // padded columns: w3 = 0
        hw[4 * g + j] = z > 0.f ? st.g * z : 0.f;                           // g relu(z2): the dw3 summand
      }
    }
    if (col0 < p.cols) {                                    // every row of the panel exists (padded pairs carry g~ = 0)
      uint32_t hi[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) hi[c] = ptx::pack_bf16(dz[2 * c], dz[2 * c + 1]);
      const bool full = col0 + 16 <= p.cols;
      __nv_bfloat16* d = p.dz + (size_t)row * p.pitch + col0;
      if (full) {
        uint4* d4 = reinterpret_cast<uint4*>(d);
        d4[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        d4[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
      } else {
        for (int c = 0; c < 16; ++c) if (col0 + c < p.cols) d[c] = __float2bfloat16(dz[c]);
      }
      if (p.dz_lo != nullptr) {
        __nv_bfloat16* dl = p.dz_lo + (size_t)row * p.pitch + col0;
        uint32_t lo[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float h0 = __uint_as_float(hi[c] << 16), h1 = __uint_as_float(hi[c] & 0xffff0000u);
          lo[c] = ptx::pack_bf16(dz[2 * c] - h0, dz[2 * c + 1] - h1);
        }
        if (full) {
          uint4* d4 = reinterpret_cast<uint4*>(dl);
          d4[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          d4[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
        } else {
          for (int c = 0; c < 16; ++c)
            if (col0 + c < p.cols) dl[c] = __float2bfloat16(dz[c] - __bfloat162float(__float2bfloat16(dz[c])));
        }
        if (kThird && p.dz_lo2 != nullptr) {          // fp32 mode: the third piece (dz - hi) - lo, both differences exact
          __nv_bfloat16* d2 = p.dz_lo2 + (size_t)row * p.pitch + col0;
          if (full) {
            uint32_t l2[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float r0 = dz[2 * c] - __uint_as_float(hi[c] << 16), r1 = dz[2 * c + 1] - __uint_as_float(hi[c] & 0xffff0000u);
              l2[c] = ptx::pack_bf16(r0 - __uint_as_float(lo[c] << 16), r1 - __uint_as_float(lo[c] & 0xffff0000u));
            }
            uint4* d4 = reinterpret_cast<uint4*>(d2);
#pragma unroll
            for (int g = 0; g < 2; ++g) d4[g] = make_uint4(l2[4 * g], l2[4 * g + 1], l2[4 * g + 2], l2[4 * g + 3]);
          } else {
            for (int c = 0; c < 16; ++c)
              if (col0 + c < p.cols) {
                const float r = dz[c] - __bfloat162float(__float2bfloat16(dz[c]));
                d2[c] = __float2bfloat16(r - __bfloat162float(__float2bfloat16(r)));
              }
          }
        }
      }
    }
    // column sums over this warp's 32 pairs; a warp whose rows are all excluded (g~ = 0) has nothing to add.
    // Lanes l and l ^ 16 receive the same column (l & 15); lane l keeps it when its upper bit names this piece's
    // half of the 32-column group, so that lane l ends up owning column l of the group (as finish() expects).
    if (__any_sync(0xffffffffu, st.g != 0.f)) {
      const float cb = warp_column_sums16(dz, lane);
      const float cw = warp_column_sums16(hw, lane);
      if ((lane >> 4) == (kQ & 1)) {
        const int t = col0 >> 8;
#pragma unroll
        for (int tt = 0; tt < kMaxTiles; ++tt)
          if (tt == t) { st.sb[tt][kQ >> 1] += cb; st.sw[tt][kQ >> 1] += cw; }
      }
    }
  }
  static __device__ __forceinline__ void unit_end(const Params&, State&, const Unit&, int, int) {}
  static __device__ __forceinline__ void finish(const Params& p, State& st, int colq) {
    const int lane = (int)(threadIdx.x & 31);
#pragma unroll
    for (int t = 0; t < kMaxTiles; ++t)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int col = t * TILE_N + colq * 64 + h * 32 + lane;
        if (col < p.cols && (st.sb[t][h] != 0.f || st.sw[t][h] != 0.f)) {
          atomicAdd(p.db2 + col, st.sb[t][h]);
          atomicAdd(p.dw3 + col, st.sw[t][h]);
        }
      }
  }
};
using EpiMlpSp = EpiMlpSpT<false>;
using EpiMlpSp3 = EpiMlpSpT<true>;

// ---- backward through ReLU 1 with both reductions fused:  dZ1 = (dZ2 W2) . [H > 0]  is never stored;
//      dA[i, k] += sum_j dZ1[(i, j), k]  (column sums over the warp's 32 rows: one image row per M block) and
//      dC[j, k] += sum_i dZ1[(i, j), k]  (order-2 schedule: a unit walks the image rows of ONE (text block, N tile), so each
//      thread adds its (j, 64 columns) cells in registers and flushes them once per unit).
//      The ReLU mask comes as bits (one 32-bit word per pair and 32 columns, written by the H generator).
struct EpiMlpDa {
  static constexpr bool kJoint = false;
  static constexpr bool kWalk = true;
  static constexpr bool kChunk16 = true;      // 16-column accumulator reads: 64 running sums + a chunk fit the register file
  static constexpr int kEpiSmemBytes = kNumEpiWarps * 2048;   // staging of the dC flush
  struct Params {
    const uint32_t* mask;  // [rr * Bp][wpr]
    int wpr;               // mask words per pair = ceil(H1 / 32) rounded up to an even number (8 B loads)
    int B, Bp, r0, rr;     // text rows, padded text rows, first image row of the panel, image rows in the panel
    int cols;              // H1
    float* dA;             // [image rows, cols]   (atomicAdd)
    float* dC;             // [B, cols]            (atomicAdd)
  };
  struct State { uint8_t* stage_smem; float dc[64]; uint32_t mw0, mw1; int il; };
  static __device__ __forceinline__ void init(const Params&, State&) {}
  static __device__ __forceinline__ void finish(const Params&, State&, int) {}
  static __device__ __forceinline__ void unit_begin(const Params&, State& st, const Unit&, int, int) {
#pragma unroll
    for (int c = 0; c < 64; ++c) st.dc[c] = 0.f;
  }
  // before the accumulator is awaited: the item's image row and the thread's 64 mask bits (two words, 8 B aligned)
  static __device__ __forceinline__ void item_begin(const Params& p, State& st, int row, int col0) {
    st.il = row / p.Bp;
    st.mw0 = 0u; st.mw1 = 0u;
    if (st.il < p.rr) {
      const uint32_t* m = p.mask + (size_t)row * p.wpr + (col0 >> 5);
      if (col0 < p.cols) { const uint2 w = __ldg(reinterpret_cast<const uint2*>(m)); st.mw0 = w.x; st.mw1 = w.y; }   // wpr is even
    }
  }
  // kQ = which 16-column quarter of the thread's 64 columns (compile time: the running sums stay in registers)
  template <int kQ>
  static __device__ __forceinline__ void chunk16(const Params& p, State& st, const Unit&, int, int col0, uint32_t (&v)[16]) {
    const int lane = (int)(threadIdx.x & 31);
    const uint32_t mw = ((kQ & 2) ? st.mw1 : st.mw0) >> ((kQ & 1) * 16);
    float x[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      x[c] = ((mw >> c) & 1u) ? __uint_as_float(v[c]) : 0.f;
      st.dc[16 * kQ + c] += x[c];
    }
    const float cs = warp_column_sums16(x, lane);
    if (lane < 16 && st.il < p.rr && col0 + lane < p.cols) atomicAdd(p.dA + (size_t)(p.r0 + st.il) * p.cols + col0 + lane, cs);
  }
  // Flush of the unit's running sums.  A lane owns ONE text row, so a direct red per column would touch 32 rows 4 KB apart
  // per instruction; instead each 16-column quarter goes through the warp's 2 KB of shared memory ([32 rows][16] floats,
  // 16 B groups XOR-swizzled by the row as in EpiStatsRC) and is sent out as 64 B row segments: a half warp per row.
  static __device__ __forceinline__ void unit_end(const Params& p, State& st, const Unit& un, int row, int colq) {
    const int lane = (int)(threadIdx.x & 31);
    const int j0 = (row - lane) % p.Bp;                 // text row of lane 0 (the warp's 32 rows are consecutive text rows)
    const int c0 = un.nt0 * TILE_N + colq * 64;
    float* sm = reinterpret_cast<float*>(st.stage_smem);
    const int sw = (lane >> 1) & 3;
    const int cc = lane & 15, rh = lane >> 4;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      __syncwarp();
#pragma unroll
      for (int g = 0; g < 4; ++g)
        *reinterpret_cast<float4*>(sm + lane * 16 + 4 * (g ^ sw)) =
            make_float4(st.dc[16 * q + 4 * g], st.dc[16 * q + 4 * g + 1], st.dc[16 * q + 4 * g + 2], st.dc[16 * q + 4 * g + 3]);
      __syncwarp();
      const int col = c0 + 16 * q + cc;
#pragma unroll
      for (int t = 0; t < 16; ++t) {
        const int r = 2 * t + rh;
        const float v = sm[r * 16 + 4 * ((cc >> 2) ^ ((r >> 1) & 3)) + (cc & 3)];
        if (j0 + r < p.B && col < p.cols) atomicAdd(p.dC + (size_t)(j0 + r) * p.cols + col, v);
      }
    }
  }
};

// ---- pairwise Euclidean distance sums (GDV, validate.py:23-34): acc = <a_row, b_col>,
//      d = sqrt(max(|a|^2 + |b|^2 - 2 acc, 0)); the epilogue keeps one running sum per thread, S is never stored
struct EpiDist {
  static constexpr bool kJoint = false;
  static constexpr bool kWalk = false;
  static constexpr bool kChunk16 = false;
  static constexpr int kEpiSmemBytes = 0;
  struct Params {
    const float* na;       // [rows] squared norms of the A rows
    const float* nb;       // [n_ntile * 256] squared norms of the B rows, zero padded
    int rows, cols;
    int same;              // A and B are the same set: the diagonal is exactly 0 (pairwise_distances(X) forces it)
    float* part;           // [n_split * kColQuarters][rows_padded]
    int rows_padded;
  };
  struct State { uint8_t* stage_smem; float acc; float na; };
  static __device__ __forceinline__ void init(const Params&, State&) {}
  static __device__ __forceinline__ void finish(const Params&, State&, int) {}
  static __device__ __forceinline__ void unit_begin(const Params& p, State& st, const Unit&, int row, int) {
    st.acc = 0.f;
    st.na = row < p.rows ? __ldg(p.na + row) : 0.f;
  }
  static __device__ __forceinline__ void chunk(const Params& p, State& st, const Unit&, int row, int col0, uint32_t (&v)[32]) {
    if (row >= p.rows || col0 >= p.cols) return;
    const float4* n4 = reinterpret_cast<const float4*>(p.nb + col0);
    float a0 = 0.f, a1 = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const float4 nb = __ldg(n4 + g);
      const float nn[4] = {nb.x, nb.y, nb.z, nb.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int col = col0 + 4 * g + j;
        const float d2 = fmaf(-2.f, __uint_as_float(v[4 * g + j]), st.na + nn[j]);
        const bool ok = col < p.cols && !(p.same && col == row);
        const float d = ok ? sqrtf(fmaxf(d2, 0.f)) : 0.f;
        if (j & 1) a1 += d; else a0 += d;
      }
    }
    st.acc += a0 + a1;
  }
  static __device__ __forceinline__ void unit_end(const Params& p, State& st, const Unit& un, int row, int colq) {
    p.part[((size_t)un.s * kColQuarters + colq) * p.rows_padded + row] = st.acc;
  }
};

}  // namespace mi
