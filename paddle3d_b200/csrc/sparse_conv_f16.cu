// Sparse-conv gather-GEMM on tcgen05, fp16 hi/lo split rows ("H16"), persistent + fully overlapped.
//
// Why fp16 pairs instead of tf32 pairs: the kernel is bound by bytes moved into shared memory (LDGSTS issue rate for the
// row gathers, L2->SM bandwidth for the weight slices), not by the tensor pipe.  x = hi + lo' * 2^-11 with
// hi = fp16(x), lo' = fp16((x - hi) * 2^11) carries the same 22 mantissa bits as the tf32 pair (both formats have 11
// significant bits; the power-of-two scale keeps lo' in fp16's normal range) in HALF the bytes: a split row is as large
// as the plain fp32 row, a 32-channel slice of a row is one 128-byte line holding both halves, kind::f16 MMAs run at
// twice the tf32 rate, and the weight image halves too.  Range: |x| < 65504 (flagged in `status` bit 0 otherwise);
// the tf32 kernels (sparse_conv_tc2.cu) stay available for data outside that range.
//
//   D[0, N)    += A_hi  x B_hi                      (N = Cout)
//   D[N, 2N)   += A_hi  x B_lo' + A_lo' x B_hi      (both scaled by 2^11)         out = D[0,N) + D[N,2N) * 2^-11
//   -> per 16-channel k-step: one MMA A_hi x [B_hi | B_lo'] (N' = 2N) and one MMA A_lo' x B_hi accumulating into the
//      upper half; 2N TMEM columns per tile, double buffered (<= 512 columns at Cout = 128).
//
// Row layout H16 of a C-channel row (4*C bytes): groups of KC = min(C, 32) channels, each [hi KC halfs | lo' KC halfs].
// Shared-memory operand "sub-tile": 128 rows x 128 bytes, SWIZZLE_128B K-major (64 fp16 = 4 k-steps of 16):
//   C >= 32: one (tap, 32-channel group): k-steps 0,1 = hi, 2,3 = lo'  -> one 128-byte line per gathered row
//   C == 16: two taps: k-steps 0,1 = hi, lo' of tap a; 2,3 = hi, lo' of tap b -> two 64-byte half lines per row
// A pipeline stage = NSUB sub-tiles (32 KB of rows for Cout <= 64) + their weight blocks: one full/empty mbarrier
// round trip feeds 4 * NSUB MMAs.
//
// CTA = 1 per SM, persistent over work items (tile of 128 output rows, tap split); 11 warps:
//   0-3  producers   cp.async row gathers (zero-fill for missing neighbours), run up to STAGES stages ahead
//   4-7  epilogue    tcgen05.ld -> (+ split-K fix-up) -> BN / bias / residual / ReLU -> fp32 rows and / or H16 rows;
//                    overlaps the next item's main loop (double-buffered accumulators)
//   8    MMA issue   9  weight slices (cp.async.bulk)   10  neighbour-map prefetch (cp.async.bulk) + active-tap scan
// Split-K over taps (few tiles on the deep levels): the split count is chosen ON THE DEVICE from the row count so
// that the work items fill the grid; partial tiles go to scratch slabs and the LAST arriving CTA of a tile (ticket
// counter) sums the slabs in index order (deterministic) and runs the fused epilogue - no finalize launch.
#include <cuda.h>
#include <cuda_fp16.h>

#include "h16.cuh"
#include "tc_common.cuh"

namespace p3d {
namespace f16 {

using namespace tc;

// warp roles for NPW producer warps (NPW in {4, 8, 16}): [0, NPW) producers, [NPW, NPW + 4) epilogue (TMEM lane
// quarter = wid & 3), NPW + 4 MMA issue, NPW + 5 weight slices, NPW + 6 neighbour-map prefetch
constexpr int kSub = 128 * 128;  // bytes of one A sub-tile
constexpr int kMaxSplits = 4;
constexpr int kMaxStages = 12;

template <int CIN, int COUT, int NSUB_>
struct Cfg {
  static constexpr int KC = (CIN >= 32) ? 32 : 16;
  static constexpr int G = CIN / KC;                         // sub-tiles per tap (CIN >= 32); CIN == 16: 2 taps / sub-tile
  static constexpr int NSUB = NSUB_;                         // sub-tiles per stage
  static constexpr int B_SUB = 128 * COUT;                   // bytes of the weight blocks of one sub-tile (2 k-blocks)
  static constexpr int B_BLK = 64 * COUT;                    // one 16-channel k-block: [2 chunks][2*COUT rows][16 B]
  static constexpr int STAGE = NSUB * (kSub + B_SUB);
  // ring depth from the shared-memory budget: 227 KB - 1 KB alignment slack - 2 x 16 KB neighbour map (K <= 32) - 3 KB static
  static constexpr int BUDGET = (227 - 1 - 32 - 3) * 1024;
  static constexpr int S_RAW = BUDGET / STAGE;
  static constexpr int STAGES = S_RAW > kMaxStages ? kMaxStages : S_RAW;
  static constexpr int TMEM_COLS = (4 * COUT <= 64) ? 64 : (4 * COUT <= 128) ? 128 : (4 * COUT <= 256) ? 256 : 512;
  // kind::f16: a/b format 0 (fp16), accumulator fp32, K-major both, M = 128
  static constexpr uint32_t IDESC2 = (1u << 4) | (static_cast<uint32_t>((2 * COUT) >> 3) << 17) |
                                     (static_cast<uint32_t>(kM >> 4) << 24);
  static constexpr uint32_t IDESC1 = (1u << 4) | (static_cast<uint32_t>(COUT >> 3) << 17) |
                                     (static_cast<uint32_t>(kM >> 4) << 24);
  static_assert(CIN % 16 == 0 && COUT % 16 == 0 && COUT <= 128 && CIN <= 128, "16-channel multiples up to 128");
  static_assert(CIN == 16 || CIN % 32 == 0, "CIN = 16 or a multiple of 32");
  static_assert(STAGE % 1024 == 0, "SWIZZLE_128B tiles need 1024-byte alignment");
  static_assert(STAGES >= 3, "ring too shallow");
};

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, bool valid) {
  const uint32_t sz = valid ? 16u : 0u;  // src-size 0 => 16 bytes of zeros
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint64_t desc_sw128(uint32_t addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((addr & 0x3ffffu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= 1ull << 46;
  d |= 2ull << 61;
  return d;
}
__device__ __forceinline__ void umma_f16_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&a)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]), "=r"(a[8]),
        "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15])
      : "r"(taddr));
}
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 128;" ::: "memory"); }


// Number of tap splits for `n_tiles` row tiles on `grid` persistent CTAs: minimise waves x (taps per item + fixed cost).
__host__ __device__ inline int choose_splits(long long n_tiles, int grid, int K, int smax) {
  if (smax > K) smax = K;
  if (smax < 1) smax = 1;
  int best = 1;
  long long best_cost = -1;
  for (int s = 1; s <= smax; ++s) {
    const long long waves = (n_tiles * s + grid - 1) / grid;
    const long long cost = waves * ((K + s - 1) / s + 4 + (s > 1 ? 1 : 0));
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = s;
    }
  }
  return best;
}
// taps of split `split` (t == split mod splits), K <= 32
__device__ __forceinline__ uint32_t split_taps(int split, int splits, int K) {
  uint32_t m = 0u;
  for (int t = split; t < K; t += splits) m |= 1u << t;
  return m;
}

// Work decomposition of one launch.  stream = 0: items (tile, split), split s owns the taps t == s (mod splits), item
// w = blockIdx.x + it * gridDim.x.  stream = 1 ("stream-K"): the n_tiles * K (tile, tap) units are cut into g_eff equal
// contiguous ranges, one per CTA; a CTA's items are the tiles its range touches, each with the contiguous tap range that
// falls inside.  A tile cut by range boundaries has `pieces` partial sums (its CTAs are consecutive: piece = CTA - first
// CTA), combined through the slabs / ticket like the splits.  No wave quantisation: 309 tiles on 148 CTAs cost 56 taps
// per CTA instead of 3 x 27.  Ranges are never shorter than ceil((K - 1) / (kMaxSplits - 1)) units, so pieces <= kMaxSplits.
struct Sched {
  int stream, splits, K;
  long long n_work;          // stream = 0: n_tiles * splits
  long long total, g_eff;    // stream = 1
  long long u0, u1;          // stream = 1: this CTA's unit range
};
__device__ __forceinline__ Sched make_sched(long long n_tiles, int K, int smax, int mode, int fix_taps) {
  Sched sc;
  sc.K = K;
  sc.stream = 0;
  const int grid = static_cast<int>(gridDim.x);
  sc.splits = choose_splits(n_tiles, grid, K, smax);
  sc.n_work = n_tiles * sc.splits;
  sc.total = n_tiles * K;
  sc.g_eff = 1;
  sc.u0 = sc.u1 = 0;
  if (mode && smax >= 4 && sc.total > 0) {  // slabs for 4 pieces available
    const int u_min = (K - 1 + 2) / 3 > 1 ? (K - 1 + 2) / 3 : 1;  // ceil((K - 1) / (kMaxSplits - 1)), kMaxSplits = 4
    long long g = sc.total / u_min;
    if (g > grid) g = grid;
    if (g < 1) g = 1;
    const long long waves = (sc.n_work + grid - 1) / grid;
    const long long cost_old = waves * ((K + sc.splits - 1) / sc.splits + 4 + (sc.splits > 1 ? 1 : 0));
    const long long cost_stream = (sc.total + g - 1) / g + 4 + fix_taps;
    if (mode == 2 || cost_stream < cost_old) {
      sc.stream = 1;
      sc.g_eff = g;
      const long long c = blockIdx.x;
      if (c < g) {
        sc.u0 = c * sc.total / g;
        sc.u1 = (c + 1) * sc.total / g;
      }
    }
  }
  return sc;
}
// item `it` of this CTA: false when the CTA has no more items
__device__ __forceinline__ bool sched_item(const Sched &sc, int it, long long &tile, uint32_t &mask, int &piece, int &pieces) {
  if (!sc.stream) {
    const long long w = static_cast<long long>(blockIdx.x) + static_cast<long long>(it) * gridDim.x;
    if (w >= sc.n_work) return false;
    tile = w / sc.splits;
    piece = static_cast<int>(w - tile * sc.splits);
    pieces = sc.splits;
    mask = split_taps(piece, pieces, sc.K);
    return true;
  }
  tile = sc.u0 / sc.K + it;
  const long long start = tile * sc.K;
  if (start >= sc.u1) return false;
  const int ta = static_cast<int>((sc.u0 > start ? sc.u0 : start) - start);
  const int tb = static_cast<int>((sc.u1 < start + sc.K ? sc.u1 : start + sc.K) - start);
  mask = (tb >= 32 ? 0xffffffffu : ((1u << tb) - 1u)) & ~((1u << ta) - 1u);
  const long long cf = ((start + 1) * sc.g_eff - 1) / sc.total, cl = ((start + sc.K) * sc.g_eff - 1) / sc.total;
  piece = static_cast<int>(static_cast<long long>(blockIdx.x) - cf);
  pieces = static_cast<int>(cl - cf + 1);
  return true;
}

struct Params {
  const uint8_t *in;        // H16 rows [n_in][4 * CIN bytes]
  const int32_t *nbr;       // [n_cap][K]
  const int32_t *n_out_dev; // device row count (or null: n_cap)
  long long n_cap;
  int K;
  int smax;                 // max tap splits the workspace allows (1 = never split)
  const uint8_t *packed_w;  // [K * CIN / 16] k-blocks of 64 * COUT bytes
  const float *scale, *shift;
  const uint8_t *residual;  // H16 rows [n][4 * COUT bytes] or null
  int relu;
  float *out_f32;           // [n][COUT] or null
  uint8_t *out_h16;         // [n][4 * COUT bytes] or null
  float *slabs;             // split-K scratch [smax][tiles][COUT / 4][128] float4 (smax > 1)
  int32_t *counters;        // split-K tickets [tiles], zero on entry, left zero
  int32_t *status;          // optional: bit 0 = fp16 range overflow while producing out_h16
  const uint8_t *zero_row;  // 512 zero bytes in global memory (target of missing neighbours with flag 2)
  long long *dbg;           // debug only (p3d_debug_f16_timeline): clock64 timeline of CTA `dbg_cta`, layout below
  int dbg_cta;
  int sk_mode, sk_fix;      // stream-K: 0 off, 1 when the cost model prefers it, 2 always; cost of a fix-up in taps
  int flags;                // tuning / debug: 1 all neighbours missing, 2 missing neighbours read zero_row instead of a
                            // zero-size copy, 4 all neighbours present (pseudo-random rows); 1 and 4 give wrong results
};
// dbg layout: stage use c (< 512), 8 slots: 0 producer(warp 0) empty acquired, 1 gathers issued, 2 W empty acquired,
// 3 W issued, 4 MMA full seen, 5 MMA committed.  From dbg[4096], 8 slots per item (< 64): 0 nbr buffer free, 1 map
// landed, 3 producer item start, 4 producer item end, 5 epilogue accumulators complete, 6 epilogue done, 7 MMA item
// start.  dbg[8192 ..]: kernel entry, prologue done, producer exit, n_work, splits.

// warp roles for NPW producer warps: [0, NPW) producers, [NPW, NPW + 4) epilogue (TMEM lane quarter = wid & 3),
// NPW + 4 MMA issue, NPW + 5 weight slices, NPW + 6 neighbour-map prefetch
template <int CIN, int COUT, int NPW, int NSUB>
__global__ void __launch_bounds__((NPW + 7) * 32, 1) conv_f16_kernel(const Params p) {
  using C = Cfg<CIN, COUT, NSUB>;
  constexpr int S = C::STAGES;
  constexpr int kEpiWarp0 = NPW, kMmaWarp = NPW + 4, kWWarp = NPW + 5;
  constexpr int RPW = kM / NPW, QN = RPW / 4;  // rows per producer warp, cp.async instructions per thread and sub-tile
  static_assert(NPW == 4 || NPW == 8 || NPW == 16, "producer warps: 4, 8 or 16");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const long long n = p.n_out_dev ? min(static_cast<long long>(p.n_out_dev[0]), p.n_cap) : p.n_cap;
  const long long n_tiles = (n + kM - 1) / kM;
  const int K = p.K;
  const Sched sc = make_sched(n_tiles, K, p.smax, p.sk_mode, p.sk_fix);
  if (sc.stream ? (sc.u0 >= sc.u1) : (static_cast<long long>(blockIdx.x) >= sc.n_work)) return;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  int32_t *s_nbr = reinterpret_cast<int32_t *>(smem + S * C::STAGE);  // [2][kM * K]
  __shared__ __align__(8) unsigned long long s_bar[2 * kMaxStages + 10];
  // full[S] empty[S] | accumulators: full[2] empty[2] | neighbour map: landed (tx)[2] ready[2] free[2]
  constexpr int kF = 0, kE = kMaxStages, kTF = 2 * kMaxStages, kTE = kTF + 2, kNR = kTF + 4, kNY = kTF + 6, kNE = kTF + 8;
  __shared__ uint32_t s_tmem_base;
  __shared__ int s_last;
  __shared__ float s_scale[COUT], s_shift[COUT];

  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  if (tid < COUT) {  // static parameters: safe before griddepcontrol.wait
    s_scale[tid] = p.scale ? __ldg(p.scale + tid) : 1.0f;
    s_shift[tid] = p.shift ? __ldg(p.shift + tid) : 0.0f;
  }
  const bool dbgc = p.dbg && static_cast<int>(blockIdx.x) == p.dbg_cta;
  const bool dbgl = dbgc && lane == 0;
  if (dbgc && tid == 0) {
    p.dbg[8192] = clock64();
    p.dbg[8195] = sc.stream ? (sc.u1 - sc.u0) : sc.n_work;
    p.dbg[8196] = sc.stream ? -sc.g_eff : sc.splits;
  }
  if (tid == kMmaWarp * 32) {
    for (int s = 0; s < S; ++s) {
      mbar_init(smem_u32(&s_bar[kF + s]), NPW * 32 + 1);  // producers' cp.async completions + weight expect_tx
      mbar_init(smem_u32(&s_bar[kE + s]), 1);             // tcgen05.commit
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&s_bar[kTF + b]), 1);
      mbar_init(smem_u32(&s_bar[kTE + b]), 4);
      mbar_init(smem_u32(&s_bar[kNR + b]), 1);
      mbar_init(smem_u32(&s_bar[kNY + b]), 1);
      mbar_init(smem_u32(&s_bar[kNE + b]), NPW);
    }
    fence_mbar_init();
  }
  if (wid == kMmaWarp) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)),
                 "r"(static_cast<uint32_t>(C::TMEM_COLS))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;
  const uint32_t ring = smem_u32(smem);
  const int nbr_words = kM * K;
  if (dbgc && tid == 0) p.dbg[8193] = clock64();

  // Every role walks the same item sequence it = 0, 1, ..: w = blockIdx.x + it * gridDim.x.  The taps of an item are
  // known arithmetically (all K, or the split's residue class): a tap without any neighbour in the tile just multiplies
  // zero rows (rare: the rows of a tile are not spatially sorted), so nothing on the critical path scans the map.
  if (wid < NPW) {
    // ------------------------------------------------------------------------------------------ producers
    asm volatile("griddepcontrol.wait;" ::: "memory");  // the input rows are the previous layer's output
    int s = 0;
    uint32_t eph = 1;  // parity to wait for on empty[s] (fresh barrier: parity 1 passes)
    const int sub4 = lane >> 3, ch = lane & 7;
    const int flags = p.flags;
    int it = 0;
    int cuse = 0;
    const bool dp = dbgl && wid == 0;
    long long tile;
    uint32_t m;
    int piece, pieces;
    for (; sched_item(sc, it, tile, m, piece, pieces); ++it) {
      const int b = it & 1;
      const int rows = static_cast<int>(min(static_cast<long long>(kM), n - tile * kM));
      const int n_taps = __popc(m);
      const int n_sub = (CIN == 16) ? (n_taps + 1) / 2 : n_taps * C::G;
      mbar_wait(smem_u32(&s_bar[kNY + b]), static_cast<uint32_t>((it >> 1) & 1));
      if (dp && it < 64) p.dbg[4096 + it * 8 + 3] = clock64();
      const int32_t *nb = s_nbr + b * nbr_words;
      auto fetch = [&](int row, int t) -> int {
        int idx = row < rows ? nb[row * K + t] : -1;
        if (flags & 5) {
          if (flags & 1) idx = -1;
          if ((flags & 4) && row < rows) idx = static_cast<int>(hash32(static_cast<uint32_t>(tile * kM + row) * 27u + t) % static_cast<uint32_t>(n));
        }
        return idx;
      };
      int k = 0;  // sub-tile index inside the item
      if (CIN == 16) {
        // lanes 0-3 of a row fetch tap a's 64-byte row, lanes 4-7 tap b's
        while (m) {
          const int ta = __ffs(m) - 1;
          m &= m - 1;
          int tb = -1;
          if (m) {
            tb = __ffs(m) - 1;
            m &= m - 1;
          }
          const int t = (ch < 4) ? ta : tb;
          if ((k % NSUB) == 0) {
            mbar_wait(smem_u32(&s_bar[kE + s]), eph);
            if (dp && cuse < 512) p.dbg[cuse * 8 + 0] = clock64();
          }
          const uint32_t sb = ring + static_cast<uint32_t>(s * C::STAGE + (k % NSUB) * kSub);
          if (t >= 0) {
#pragma unroll
            for (int q = 0; q < QN; ++q) {
              const int row = wid * RPW + q * 4 + sub4;
              const int idx = fetch(row, t);
              bool ok = idx >= 0;
              const uint8_t *src = p.in + (ok ? static_cast<size_t>(idx) * 64 : 0) + (ch & 3) * 16;
              if ((flags & 2) && !ok) {
                src = p.zero_row + (ch & 3) * 16;
                ok = true;
              }
              cp_async16(sb + static_cast<uint32_t>(row * 128 + ((ch ^ (row & 7)) << 4)), src, ok);
            }
          }
          ++k;
          if ((k % NSUB) == 0 || k == n_sub) {
            cp_async_arrive_noinc(smem_u32(&s_bar[kF + s]));
            if (dp && cuse < 512) p.dbg[cuse * 8 + 1] = clock64();
            ++cuse;
            if (++s == S) {
              s = 0;
              eph ^= 1u;
            }
          }
        }
      } else {
        while (m) {
          const int t = __ffs(m) - 1;
          m &= m - 1;
          int idx[QN];
#pragma unroll
          for (int q = 0; q < QN; ++q) idx[q] = fetch(wid * RPW + q * 4 + sub4, t);
#pragma unroll 1
          for (int g = 0; g < C::G; ++g) {
            if ((k % NSUB) == 0) {
              mbar_wait(smem_u32(&s_bar[kE + s]), eph);
              if (dp && cuse < 512) p.dbg[cuse * 8 + 0] = clock64();
            }
            const uint32_t sb = ring + static_cast<uint32_t>(s * C::STAGE + (k % NSUB) * kSub);
#pragma unroll
            for (int q = 0; q < QN; ++q) {
              const int row = wid * RPW + q * 4 + sub4;
              bool ok = idx[q] >= 0;
              const uint8_t *src = p.in + (ok ? static_cast<size_t>(idx[q]) * (4 * CIN) : 0) + g * 128 + ch * 16;
              if ((flags & 2) && !ok) {
                src = p.zero_row + ch * 16;
                ok = true;
              }
              cp_async16(sb + static_cast<uint32_t>(row * 128 + ((ch ^ (row & 7)) << 4)), src, ok);
            }
            ++k;
            if ((k % NSUB) == 0 || k == n_sub) {
              cp_async_arrive_noinc(smem_u32(&s_bar[kF + s]));
              if (dp && cuse < 512) p.dbg[cuse * 8 + 1] = clock64();
              ++cuse;
              if (++s == S) {
                s = 0;
                eph ^= 1u;
              }
            }
          }
        }
      }
      __syncwarp();
      if (dp && it < 64) p.dbg[4096 + it * 8 + 4] = clock64();
      if (lane == 0) mbar_arrive(smem_u32(&s_bar[kNE + b]));  // done with this item's neighbour map
    }
    if (dp) p.dbg[8194] = clock64();
  } else if (wid < kMmaWarp) {
    // ------------------------------------------------------------------------------------------ epilogue
    asm volatile("griddepcontrol.wait;" ::: "memory");  // residual rows / output buffers belong to earlier kernels
    const int quarter = wid & 3;
    const int r = quarter * 32 + lane;
    const int etid = tid - kEpiWarp0 * 32;
    constexpr int KCO = (COUT >= 32) ? 32 : 16;   // channels per H16 group of the output / residual rows
    constexpr int NCH = COUT / 16;                 // 16-channel chunks
    const size_t tiles_cap = static_cast<size_t>((p.n_cap + kM - 1) / kM);
    bool ovf = false;
    int it = 0;
    long long tile;
    uint32_t item_mask;
    int split, splits;  // piece of the tile this item computes / number of pieces the tile is cut into
    for (; sched_item(sc, it, tile, item_mask, split, splits); ++it) {
      const int b = it & 1;
      const long long row0 = tile * kM;
      const int rows = static_cast<int>(min(static_cast<long long>(kM), n - row0));
      const bool live = r < rows;
      const size_t orow = static_cast<size_t>(row0 + r);
      // residual of the first chunk: requested BEFORE waiting for the accumulators, so its L2 round trip overlaps the
      // main loop; later chunks are requested one chunk ahead of their use
      const uint8_t *res_row = p.residual ? p.residual + orow * (4 * COUT) : nullptr;
      uint4 rq[4];  // hi 32 B, lo' 32 B of the next chunk
      auto res_load = [&](int c0) {
        const uint8_t *rp = res_row + (c0 / KCO) * (4 * KCO) + (c0 % KCO) * 2;
        rq[0] = __ldg(reinterpret_cast<const uint4 *>(rp));
        rq[1] = __ldg(reinterpret_cast<const uint4 *>(rp) + 1);
        rq[2] = __ldg(reinterpret_cast<const uint4 *>(rp + 2 * KCO));
        rq[3] = __ldg(reinterpret_cast<const uint4 *>(rp + 2 * KCO) + 1);
      };
      const bool use_res = res_row != nullptr && live;
      if (use_res && splits == 1) res_load(0);
      mbar_wait(smem_u32(&s_bar[kTF + b]), static_cast<uint32_t>((it >> 1) & 1));
      tc_fence_after();
      if (dbgl && quarter == 0 && it < 64) p.dbg[4096 + it * 8 + 5] = clock64();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(b * 2 * COUT);
      // split-K slabs: [split][tile][COUT / 4][128 rows] float4 -> a warp's accesses are 512 contiguous bytes
      float4 *slab4 = p.slabs ? reinterpret_cast<float4 *>(p.slabs) + (static_cast<size_t>(tile) * (COUT / 4)) * kM + r : nullptr;
      const size_t slab_stride4 = tiles_cap * (COUT / 4) * kM;  // float4 units between two splits
      bool finish = true;  // this CTA runs the fused epilogue of the tile
      if (splits > 1) {
        // pass 1: raw partial sums to this split's slab
        float4 *mine = slab4 + static_cast<size_t>(split) * slab_stride4;
#pragma unroll 2
        for (int c = 0; c < NCH; ++c) {
          uint32_t a[16], x[16];
          tmem_ld16(taddr + static_cast<uint32_t>(c * 16), a);
          tmem_ld16(taddr + static_cast<uint32_t>(COUT + c * 16), x);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            float4 v;
            v.x = fmaf(__uint_as_float(x[j]), kLoInv, __uint_as_float(a[j]));
            v.y = fmaf(__uint_as_float(x[j + 1]), kLoInv, __uint_as_float(a[j + 1]));
            v.z = fmaf(__uint_as_float(x[j + 2]), kLoInv, __uint_as_float(a[j + 2]));
            v.w = fmaf(__uint_as_float(x[j + 3]), kLoInv, __uint_as_float(a[j + 3]));
            __stcg(mine + static_cast<size_t>(c * 4 + j / 4) * kM, v);  // rows beyond `rows` land in the slab's padding
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&s_bar[kTE + b]));  // accumulator buffer free for item it + 2
        __threadfence();
        epi_bar();
        if (etid == 0) {
          const int old = atomicAdd(p.counters + tile, 1);
          const int last = (old == splits - 1) ? 1 : 0;
          if (last) p.counters[tile] = 0;  // all splits have arrived: leave the ticket clean for the next launch
          s_last = last;
        }
        epi_bar();
        finish = s_last != 0;
        epi_bar();  // s_last is rewritten by the next item
        if (finish) {
          __threadfence();
          if (use_res) res_load(0);
        }
      }
      if (finish) {
#pragma unroll 1
        for (int c = 0; c < NCH; ++c) {
          const int c0 = c * 16;
          float v[16];
          if (splits > 1) {
            // slabs in index order (deterministic); all loads of the chunk are in flight together
            float4 t4[kMaxSplits][4];
#pragma unroll
            for (int sp = 0; sp < kMaxSplits; ++sp)
              if (sp < splits) {
#pragma unroll
                for (int j = 0; j < 4; ++j) t4[sp][j] = __ldcg(slab4 + static_cast<size_t>(sp) * slab_stride4 + static_cast<size_t>(c * 4 + j) * kM);
              }
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = 0.f;
#pragma unroll
            for (int sp = 0; sp < kMaxSplits; ++sp)
              if (sp < splits) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  v[4 * j] += t4[sp][j].x;
                  v[4 * j + 1] += t4[sp][j].y;
                  v[4 * j + 2] += t4[sp][j].z;
                  v[4 * j + 3] += t4[sp][j].w;
                }
              }
          } else {
            uint32_t a[16], x[16];
            tmem_ld16(taddr + static_cast<uint32_t>(c0), a);
            tmem_ld16(taddr + static_cast<uint32_t>(COUT + c0), x);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = fmaf(__uint_as_float(x[j]), kLoInv, __uint_as_float(a[j]));
            if (c == NCH - 1) {  // last chunk read: release the accumulator buffer before the global stores
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(smem_u32(&s_bar[kTE + b]));
            }
          }
          float res[16];
          if (use_res) {
            const uint32_t hw[8] = {rq[0].x, rq[0].y, rq[0].z, rq[0].w, rq[1].x, rq[1].y, rq[1].z, rq[1].w};
            const uint32_t lw[8] = {rq[2].x, rq[2].y, rq[2].z, rq[2].w, rq[3].x, rq[3].y, rq[3].z, rq[3].w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const __half2 hh = *reinterpret_cast<const __half2 *>(&hw[j]);
              const __half2 ll = *reinterpret_cast<const __half2 *>(&lw[j]);
              res[2 * j] = merge_h16(__low2half(hh), __low2half(ll));
              res[2 * j + 1] = merge_h16(__high2half(hh), __high2half(ll));
            }
            if (c + 1 < NCH) res_load(c0 + 16);  // next chunk's residual in flight while this one is finished
          }
          if (live) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float o = fmaf(v[j], s_scale[c0 + j], s_shift[c0 + j]);
              if (use_res) o = o + res[j];
              if (p.relu) o = fmaxf(o, 0.f);
              v[j] = o;
            }
            if (p.out_f32) {
#pragma unroll
              for (int j = 0; j < 16; j += 4)
                *reinterpret_cast<float4 *>(p.out_f32 + orow * COUT + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            }
            if (p.out_h16) {
              uint32_t hw[8], lw[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                __half h0, l0, h1, l1;
                split_h16(v[2 * j], h0, l0, ovf);
                split_h16(v[2 * j + 1], h1, l1, ovf);
                const __half2 hh = __halves2half2(h0, h1), ll = __halves2half2(l0, l1);
                hw[j] = *reinterpret_cast<const uint32_t *>(&hh);
                lw[j] = *reinterpret_cast<const uint32_t *>(&ll);
              }
              uint8_t *op = p.out_h16 + orow * (4 * COUT) + (c0 / KCO) * (4 * KCO) + (c0 % KCO) * 2;
              reinterpret_cast<uint4 *>(op)[0] = make_uint4(hw[0], hw[1], hw[2], hw[3]);
              reinterpret_cast<uint4 *>(op)[1] = make_uint4(hw[4], hw[5], hw[6], hw[7]);
              reinterpret_cast<uint4 *>(op + 2 * KCO)[0] = make_uint4(lw[0], lw[1], lw[2], lw[3]);
              reinterpret_cast<uint4 *>(op + 2 * KCO)[1] = make_uint4(lw[4], lw[5], lw[6], lw[7]);
            }
          }
        }
      }
      if (dbgl && quarter == 0 && it < 64) p.dbg[4096 + it * 8 + 6] = clock64();
    }
    if (ovf && p.status) atomicOr(p.status, 1);
  } else if (wid == kMmaWarp) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    int s = 0;
    uint32_t fph = 0;  // parity to wait for on full[s]
    int it = 0;
    int cuse = 0;
    long long tile;
    uint32_t item_mask;
    int piece, pieces;
    for (; sched_item(sc, it, tile, item_mask, piece, pieces); ++it) {
      const int b = it & 1;
      const int n_taps = __popc(item_mask);
      const int n_sub = (CIN == 16) ? (n_taps + 1) / 2 : n_taps * C::G;
      mbar_wait(smem_u32(&s_bar[kTE + b]), static_cast<uint32_t>(((it >> 1) & 1) ^ 1));  // epilogue of item it - 2 done
      tc_fence_after();
      if (dbgl && it < 64) p.dbg[4096 + it * 8 + 7] = clock64();
      const uint32_t acc = tmem_base + static_cast<uint32_t>(b * 2 * COUT);
      for (int k = 0; k < n_sub; k += NSUB) {
        mbar_wait(smem_u32(&s_bar[kF + s]), fph);
        if (dbgl && cuse < 512) p.dbg[cuse * 8 + 4] = clock64();
        fence_proxy_async();  // cp.async (generic proxy) writes -> tensor-core (async proxy) reads
        tc_fence_after();
        const uint32_t st = ring + static_cast<uint32_t>(s * C::STAGE);
#pragma unroll
        for (int j = 0; j < NSUB; ++j) {
          if (k + j < n_sub) {
            const uint32_t a_base = st + static_cast<uint32_t>(j * kSub);
            const uint32_t b_base = st + static_cast<uint32_t>(NSUB * kSub + j * C::B_SUB);
            const bool half_only = (CIN == 16) && (k + j == n_sub - 1) && (n_taps & 1);
#pragma unroll
            for (int kb = 0; kb < 2; ++kb) {
              if (kb == 1 && half_only) continue;
              const int ks_hi = (CIN == 16) ? 2 * kb : kb, ks_lo = (CIN == 16) ? 2 * kb + 1 : 2 + kb;
              const uint64_t db = smem_desc(b_base + static_cast<uint32_t>(kb * C::B_BLK), 2 * COUT * 16, 128);
              const uint32_t first = (k | j | kb) ? 1u : 0u;
              umma_f16_elect(acc, desc_sw128(a_base + ks_hi * 32), db, C::IDESC2, first);    // A_hi x [B_hi | B_lo']
              umma_f16_elect(acc + COUT, desc_sw128(a_base + ks_lo * 32), db, C::IDESC1, 1u);  // A_lo' x B_hi
            }
          }
        }
        umma_commit_elect(smem_u32(&s_bar[kE + s]));
        if (k + NSUB >= n_sub) umma_commit_elect(smem_u32(&s_bar[kTF + b]));
        if (dbgl && cuse < 512) p.dbg[cuse * 8 + 5] = clock64();
        ++cuse;
        if (++s == S) {
          s = 0;
          fph ^= 1u;
        }
      }
    }
    tc_fence_before();
  } else if (wid == kWWarp) {
    // ------------------------------------------------------------------------------------------ weight slices (one lane)
    if (lane == 0) {
      int s = 0;
      uint32_t eph = 1;
      int cuse = 0;
      long long tile;
      uint32_t m;
      int piece, pieces;
      for (int it = 0; sched_item(sc, it, tile, m, piece, pieces); ++it) {
        const int n_taps = __popc(m);
        const int n_sub = (CIN == 16) ? (n_taps + 1) / 2 : n_taps * C::G;
        int k = 0;
        while (m) {
          const int t = __ffs(m) - 1;
          m &= m - 1;
          if (CIN == 16) {
            int tb = -1;
            if (m) {
              tb = __ffs(m) - 1;
              m &= m - 1;
            }
            if ((k % NSUB) == 0) {
              mbar_wait(smem_u32(&s_bar[kE + s]), eph);
              if (dbgc && cuse < 512) p.dbg[cuse * 8 + 2] = clock64();
              const int subs = min(NSUB, n_sub - k);
              const int blocks = min(2 * subs, n_taps - 2 * k);
              mbar_arrive_expect_tx(smem_u32(&s_bar[kF + s]), static_cast<uint32_t>(blocks * C::B_BLK));
            }
            const uint32_t bb = ring + static_cast<uint32_t>(s * C::STAGE + NSUB * kSub + (k % NSUB) * C::B_SUB);
            bulk_g2s(bb, p.packed_w + static_cast<size_t>(t) * C::B_BLK, C::B_BLK, smem_u32(&s_bar[kF + s]));
            if (tb >= 0)
              bulk_g2s(bb + C::B_BLK, p.packed_w + static_cast<size_t>(tb) * C::B_BLK, C::B_BLK, smem_u32(&s_bar[kF + s]));
            ++k;
            if ((k % NSUB) == 0 || k == n_sub) {
              if (dbgc && cuse < 512) p.dbg[cuse * 8 + 3] = clock64();
              ++cuse;
              if (++s == S) {
                s = 0;
                eph ^= 1u;
              }
            }
          } else {
            for (int g = 0; g < C::G; ++g) {
              if ((k % NSUB) == 0) {
                mbar_wait(smem_u32(&s_bar[kE + s]), eph);
                if (dbgc && cuse < 512) p.dbg[cuse * 8 + 2] = clock64();
                const int subs = min(NSUB, n_sub - k);
                mbar_arrive_expect_tx(smem_u32(&s_bar[kF + s]), static_cast<uint32_t>(subs * C::B_SUB));
              }
              const uint32_t bb = ring + static_cast<uint32_t>(s * C::STAGE + NSUB * kSub + (k % NSUB) * C::B_SUB);
              bulk_g2s(bb, p.packed_w + (static_cast<size_t>(t) * (CIN / 16) + 2 * g) * C::B_BLK, C::B_SUB,
                       smem_u32(&s_bar[kF + s]));
              ++k;
              if ((k % NSUB) == 0 || k == n_sub) {
                if (dbgc && cuse < 512) p.dbg[cuse * 8 + 3] = clock64();
                ++cuse;
                if (++s == S) {
                  s = 0;
                  eph ^= 1u;
                }
              }
            }
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------ neighbour-map prefetch
    int it = 0;
    long long tile;
    uint32_t item_mask;
    int piece, pieces;
    for (; sched_item(sc, it, tile, item_mask, piece, pieces); ++it) {
      const int b = it & 1;
      const long long row0 = tile * kM;
      int32_t *nb = s_nbr + b * nbr_words;
      mbar_wait(smem_u32(&s_bar[kNE + b]), static_cast<uint32_t>(((it >> 1) & 1) ^ 1));  // buffer free (item it - 2 done)
      if (dbgl && it < 64) p.dbg[4096 + it * 8 + 0] = clock64();
      const int avail = static_cast<int>(min(static_cast<long long>(kM), p.n_cap - row0));
      const uint32_t words = static_cast<uint32_t>(avail) * K, bulk_words = words & ~3u;
      if (lane == 0) {
        fence_proxy_async();
        mbar_arrive_expect_tx(smem_u32(&s_bar[kNR + b]), bulk_words * 4);
        if (bulk_words) bulk_g2s(smem_u32(nb), p.nbr + row0 * K, bulk_words * 4, smem_u32(&s_bar[kNR + b]));
      }
      if (bulk_words + lane < words) nb[bulk_words + lane] = __ldg(p.nbr + row0 * K + bulk_words + lane);  // <= 3 tail words
      mbar_wait(smem_u32(&s_bar[kNR + b]), static_cast<uint32_t>((it >> 1) & 1));
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(smem_u32(&s_bar[kNY + b]));  // release: map (bulk copy + tail stores) visible to the producers
        if (dbgc && it < 64) p.dbg[4096 + it * 8 + 1] = clock64();
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (wid == kMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(static_cast<uint32_t>(C::TMEM_COLS))
                 : "memory");
  }
}

__device__ __align__(128) uint4 g_zero_row[32];  // 512 zero bytes: gather target of missing neighbours (flag 2)

template <int CIN, int COUT, int NPW, int NSUB>
int launch(const Params &p, cudaStream_t st) {
  using C = Cfg<CIN, COUT, NSUB>;
  const size_t smem = static_cast<size_t>(C::STAGES) * C::STAGE + 2 * static_cast<size_t>(kM) * p.K * sizeof(int32_t) + 1024;
  if (smem > 227 * 1024) return P3D_ERR_UNSUPPORTED;
  auto kern = conv_f16_kernel<CIN, COUT, NPW, NSUB>;
  P3D_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const long long work = ((p.n_cap + kM - 1) / kM) * (p.smax > 1 ? p.smax : 1);
  const unsigned int grid = static_cast<unsigned int>(work < kNumSMs ? work : kNumSMs);
  static const bool pdl = !(getenv("P3D_PDL") && atoi(getenv("P3D_PDL")) == 0);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3((NPW + 7) * 32);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  P3D_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, p));
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

// fp32 [K][Cin][Cout] -> k-blocks [K * Cin / 16][2 chunks][2 * Cout rows (hi, then lo')][8 halfs]
__global__ void __launch_bounds__(256) pack_weights_kernel(const float *__restrict__ w, int K, int Cin, int Cout,
                                                           __half *__restrict__ packed, int32_t *status) {
  const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(K) * Cin * Cout;
  if (q >= total) return;
  const int n = static_cast<int>(q % Cout);
  const int ci = static_cast<int>((q / Cout) % Cin);
  const int t = static_cast<int>(q / (static_cast<long long>(Cout) * Cin));
  const size_t kb = static_cast<size_t>(t) * (Cin / 16) + ci / 16;
  const int c = (ci % 16) / 8, j = ci % 8;
  __half hi, lo;
  bool ovf = false;
  split_h16(w[q], hi, lo, ovf);
  const size_t base = kb * (32 * static_cast<size_t>(Cout)) * 1 + 0;  // halfs per k-block = 64 * Cout / 2
  const size_t blk = kb * static_cast<size_t>(32 * Cout);
  (void)base;
  packed[blk + (static_cast<size_t>(c) * (2 * Cout) + n) * 8 + j] = hi;
  packed[blk + (static_cast<size_t>(c) * (2 * Cout) + Cout + n) * 8 + j] = lo;
  if (ovf && status) atomicOr(status, 1);
}

// rows [n, C] fp32 <-> H16 rows
__global__ void __launch_bounds__(256) rows_to_h16_kernel(const float *__restrict__ x, const int32_t *__restrict__ n_dev,
                                                          long long n_cap, int C, __half *__restrict__ out, int32_t *status) {
  const long long n = n_dev ? min(static_cast<long long>(n_dev[0]), n_cap) : n_cap;
  const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= n * C) return;
  const long long r = q / C;
  const int c = static_cast<int>(q - r * C);
  const int KC = C >= 32 ? 32 : 16;
  __half hi, lo;
  bool ovf = false;
  split_h16(x[q], hi, lo, ovf);
  __half *row = out + r * 2 * C + (c / KC) * (2 * KC);
  row[c % KC] = hi;
  row[KC + c % KC] = lo;
  if (ovf && status) atomicOr(status, 1);
}
__global__ void __launch_bounds__(256) rows_from_h16_kernel(const __half *__restrict__ xs, const int32_t *__restrict__ n_dev,
                                                            long long n_cap, int C, float *__restrict__ out) {
  const long long n = n_dev ? min(static_cast<long long>(n_dev[0]), n_cap) : n_cap;
  const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= n * C) return;
  const long long r = q / C;
  const int c = static_cast<int>(q - r * C);
  const int KC = C >= 32 ? 32 : 16;
  const __half *row = xs + r * 2 * C + (c / KC) * (2 * KC);
  out[q] = merge_h16(row[c % KC], row[KC + c % KC]);
}

}  // namespace f16
}  // namespace p3d

using namespace p3d;

// Debug aid (not in the public header): the next p3d_sparse_conv_f16 launches write the clock64 timeline of CTA `cta`
// into dbg (>= 8200 int64 words, device memory); dbg == NULL switches it off.  tools/f16_probe.py reads it.
static long long *g_dbg_buf = nullptr;
static int g_dbg_cta = 0;
extern "C" int p3d_debug_f16_timeline(long long *dbg, int cta) {
  g_dbg_buf = dbg;
  g_dbg_cta = cta;
  return 0;
}

extern "C" size_t p3d_sparse_conv_f16_packed_weight_bytes(int K, int Cin, int Cout) {
  if (K < 1 || K > 32 || Cin < 16 || Cout < 16 || Cin > 128 || Cout > 128 || Cout % 16 || (Cin != 16 && Cin % 32)) return 0;
  return align_up(static_cast<size_t>(K) * Cin * Cout * 4);
}

extern "C" int p3d_sparse_conv_f16_pack_weights(const float *weight, int K, int Cin, int Cout, void *packed,
                                                int32_t *status_dev, p3d_stream_t stream) {
  if (!weight || !packed || K < 1) return P3D_ERR_INVALID_ARG;
  if (!p3d_sparse_conv_f16_packed_weight_bytes(K, Cin, Cout)) return P3D_ERR_UNSUPPORTED;
  const long long total = static_cast<long long>(K) * Cin * Cout;
  f16::pack_weights_kernel<<<div_up(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      weight, K, Cin, Cout, static_cast<__half *>(packed), status_dev);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

// dense layers (csrc/dense_conv_f16.cu): the same k-block image for one N tile, W[tap][Cin][n_tile], any Cin % 32 == 0
extern "C" int p3d_dense_conv2d_f16_pack_weights(const float *weight_tci, int taps, int Cin, int n_tile, void *packed,
                                                 int32_t *status_dev, p3d_stream_t stream) {
  if (!weight_tci || !packed || taps < 1 || Cin < 32 || Cin % 32 || (n_tile != 16 && n_tile != 32 && n_tile != 64 && n_tile != 128))
    return P3D_ERR_INVALID_ARG;
  const long long total = static_cast<long long>(taps) * Cin * n_tile;
  f16::pack_weights_kernel<<<div_up(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      weight_tci, taps, Cin, n_tile, static_cast<__half *>(packed), status_dev);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

extern "C" int p3d_rows_convert_h16(const void *src, int to_h16, const int32_t *n_dev, int64_t n_cap, int C, void *dst,
                                    int32_t *status_dev, p3d_stream_t stream) {
  if (n_cap < 0 || C < 16 || (C != 16 && C % 32) || (n_cap && (!src || !dst))) return P3D_ERR_INVALID_ARG;
  if (n_cap == 0) return P3D_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (to_h16)
    f16::rows_to_h16_kernel<<<div_up(n_cap * C, 256), 256, 0, st>>>(static_cast<const float *>(src), n_dev, n_cap, C,
                                                                    static_cast<__half *>(dst), status_dev);
  else
    f16::rows_from_h16_kernel<<<div_up(n_cap * C, 256), 256, 0, st>>>(static_cast<const __half *>(src), n_dev, n_cap, C,
                                                                      static_cast<float *>(dst));
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

// workspace = [tickets: one int32 per 128-row tile][slabs: max_splits x n_out_cap x Cout fp32]; 0 for max_splits <= 1
extern "C" size_t p3d_sparse_conv_f16_workspace_bytes(int64_t n_out_cap, int Cout, int max_splits) {
  if (n_out_cap <= 0 || Cout < 16 || max_splits <= 1) return 0;
  if (max_splits > f16::kMaxSplits) max_splits = f16::kMaxSplits;
  const size_t tiles = static_cast<size_t>((n_out_cap + tc::kM - 1) / tc::kM);
  return align_up(tiles * sizeof(int32_t)) + align_up(static_cast<size_t>(max_splits) * tiles * tc::kM * Cout * sizeof(float));
}

extern "C" int p3d_sparse_conv_f16(const void *in_h16, const int32_t *nbr, const int32_t *n_out_dev, int64_t n_out_cap,
                                   int K, int Cin, int Cout, const void *packed_weight, const float *scale,
                                   const float *shift, const void *residual_h16, int relu, float *out_f32, void *out_h16,
                                   void *workspace, size_t workspace_bytes, int max_splits, int32_t *status_dev,
                                   p3d_stream_t stream) {
  if (n_out_cap < 0 || K < 1 || K > 32 || !packed_weight || (!out_f32 && !out_h16) || (n_out_cap && (!in_h16 || !nbr)))
    return P3D_ERR_INVALID_ARG;
  if (n_out_cap == 0) return P3D_OK;
  if ((reinterpret_cast<uintptr_t>(in_h16) & 15) || (reinterpret_cast<uintptr_t>(out_f32) & 15) ||
      (reinterpret_cast<uintptr_t>(out_h16) & 15) || (reinterpret_cast<uintptr_t>(packed_weight) & 15) ||
      (reinterpret_cast<uintptr_t>(residual_h16) & 15) || (reinterpret_cast<uintptr_t>(workspace) & 15) ||
      (reinterpret_cast<uintptr_t>(nbr) & 15))
    return P3D_ERR_INVALID_ARG;
  f16::Params p;
  p.in = static_cast<const uint8_t *>(in_h16);
  p.nbr = nbr;
  p.n_out_dev = n_out_dev;
  p.n_cap = n_out_cap;
  p.K = K;
  p.packed_w = static_cast<const uint8_t *>(packed_weight);
  p.scale = scale;
  p.shift = shift;
  p.residual = static_cast<const uint8_t *>(residual_h16);
  p.relu = relu;
  p.out_f32 = out_f32;
  p.out_h16 = static_cast<uint8_t *>(out_h16);
  p.status = status_dev;
  p.dbg = g_dbg_buf;
  p.dbg_cta = g_dbg_cta;
  static const int dflags = getenv("P3D_F16_FLAGS") ? atoi(getenv("P3D_F16_FLAGS")) : 0;  // tuning / debug, see Params::flags
  p.flags = dflags;
  {
    void *z = nullptr;
    P3D_CUDA_CHECK(cudaGetSymbolAddress(&z, f16::g_zero_row));
    p.zero_row = static_cast<const uint8_t *>(z);
  }
  // split-K is available up to the number of slabs the workspace holds
  int smax = max_splits;
  if (smax > f16::kMaxSplits) smax = f16::kMaxSplits;
  if (smax > K) smax = K;
  const size_t tiles = static_cast<size_t>((n_out_cap + tc::kM - 1) / tc::kM);
  const size_t tick = align_up(tiles * sizeof(int32_t));
  const size_t slab = tiles * tc::kM * static_cast<size_t>(Cout) * sizeof(float);  // whole tiles: [tile][Cout / 4][128] float4
  if (!workspace || workspace_bytes < tick + 2 * slab) smax = 1;
  if (smax > 1) {
    const size_t fit = (workspace_bytes - tick) / slab;
    if (static_cast<size_t>(smax) > fit) smax = static_cast<int>(fit);
  }
  p.smax = smax < 1 ? 1 : smax;
  // stream-K (contiguous (tile, tap) ranges per CTA instead of whole tiles) when the device-side cost model prefers it:
  // P3D_F16_STREAMK = 0 off / 1 auto (default) / 2 always; P3D_F16_SKFIX = cost of a tile's fix-up in taps (default 6)
  static const int sk_env = getenv("P3D_F16_STREAMK") ? atoi(getenv("P3D_F16_STREAMK")) : 1;
  static const int skfix_env = getenv("P3D_F16_SKFIX") ? atoi(getenv("P3D_F16_SKFIX")) : 6;
  p.sk_mode = sk_env;
  p.sk_fix = skfix_env;
  p.counters = p.smax > 1 ? static_cast<int32_t *>(workspace) : nullptr;
  p.slabs = p.smax > 1 ? reinterpret_cast<float *>(static_cast<char *>(workspace) + tick) : nullptr;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // tuning hooks: producer warps per CTA (P3D_F16_NPW = 4 / 8 / 16, default 8) and sub-tiles per pipeline stage
  // (P3D_F16_NSUB = 1 / 2; default: 2 for Cin <= 32 - 4 resp. 2 taps per stage -, 1 above; Cout = 128 always 1).
  // Measured on the C3 frame (profiles/r02_f16_sweep.md): 8 warps beat 4 by 5 % and 16 (register spills) by 14 %.
  static const int npw_env = getenv("P3D_F16_NPW") ? atoi(getenv("P3D_F16_NPW")) : 0;
  // 16 producer warps for the 16-channel layers (64-byte row gathers are the most LSU-bound: 41 vs 45 us per level-0
  // layer, profiles/r02_f16_sweep.md), 8 elsewhere
  const int npw = npw_env ? npw_env : (Cin == 16 ? 16 : 8);
  static const int nsub_env = getenv("P3D_F16_NSUB") ? atoi(getenv("P3D_F16_NSUB")) : 0;
  const int nsub = nsub_env ? nsub_env : (Cin <= 32 ? 2 : 1);
#define P3D_F16_NPW(CI, CO, NS)                                        \
  {                                                                    \
    if (npw == 4) return f16::launch<CI, CO, 4, NS>(p, st);            \
    if (npw == 16) return f16::launch<CI, CO, 16, NS>(p, st);          \
    return f16::launch<CI, CO, 8, NS>(p, st);                          \
  }
#define P3D_F16_CASE(CI, CO)                                           \
  if (Cin == CI && Cout == CO) {                                       \
    if (nsub == 2 && CO <= 64) P3D_F16_NPW(CI, CO, (CO <= 64 ? 2 : 1)) \
    P3D_F16_NPW(CI, CO, 1)                                             \
  }
  P3D_F16_CASE(16, 16)
  P3D_F16_CASE(16, 32)
  P3D_F16_CASE(32, 32)
  P3D_F16_CASE(32, 64)
  P3D_F16_CASE(64, 64)
  P3D_F16_CASE(64, 128)
  P3D_F16_CASE(128, 128)
#undef P3D_F16_CASE
#undef P3D_F16_NPW
  return P3D_ERR_UNSUPPORTED;
}
