// Dense 2-D convolution on tcgen05 with fp16 (hi, lo') pair operands for the RPN / neck / CenterHead row (SURVEY.md §8f-1;
// reference: backbones/second_backbone.py:72-120, necks/second_fpn.py:99-160, detection/centerpoint/center_head.py:43-220).
//
// Images travel between layers as "pixel H16 rows": NHWC, each pixel's C channels as groups of 32 channels
// [hi 32 halfs | lo' 32 halfs] (128 bytes per group; x = hi + lo' * 2^-11, the sparse layers' row format with row = pixel).
// One (32-channel group) x (pixel box) TMA load therefore lands in shared memory as a SWIZZLE_128B K-major operand tile
// whose k-steps 0,1 are the hi halves and 2,3 the lo' halves; the three partial products run as
//   D[0, N) += A_hi x B_hi          D[N, 2N) += A_hi x B_lo' + A_lo' x B_hi        out = D[0, N) + D[N, 2N) * 2^-11
// with one MMA A_hi x [B_hi | B_lo'] (N' = 2N) and one MMA A_lo' x B_hi per 16-channel k-step (kind::f16).
//
// The tf32 kernel this replaces (dense_conv_tc.cu) ran at the L2 -> SM bandwidth limit (measured 12.5 TB/s aggregate on the
// 256 -> 128 layer): every 3x3 tap re-loaded its shifted 128-pixel window and the weights of the use.  Here
//   * HALO mode (3x3, stride 1, pad 1 - 94 % of the flops): the haloed tile (10 x 18 pixels for an 8 x 16 output tile, or
//     10 x 34 for 8 x 32 = two M tiles) of a 32-channel group is loaded ONCE; the A operand of tap (dy, dx) is the same
//     shared-memory tile read through a descriptor whose start address is shifted by (dy * 10 + dx) rows and whose 8-row
//     group stride (SBO) is one haloed image row (1280 bytes): 6.3x less activation traffic.  The swizzle is a function of
//     the absolute shared-memory address bits, so TMA's writes and the shifted UMMA reads agree (descriptor base_offset 0;
//     verified on the B200 for both row pitches, tests/test_gpu_dense.py).
//   * TAP mode (1x1, stride 2, transposed k = s): one TMA box per (tap, group), as before, half the bytes.
//   * MT = 2: two M tiles (8 x 32 pixels) share every weight block: half the weight traffic per flop.
//
//   work item   (batch, pixel tile, N tile[, tap of a k = s transposed conv]), N tile fastest
//   warps 0-3   epilogue (TMEM lane quarter = warp)   4  MMA issue   5  activation TMA   6  weight blocks (cp.async.bulk)
#include <cuda.h>
#include <cuda_fp16.h>

#include "h16.cuh"
#include "p3d_b200.h"
#include "tc_common.cuh"

namespace p3d {
namespace dcf {

using namespace tc;

constexpr int kTW = 8, kTH = 16;        // output tile of one M = 128 UMMA: 8 x 16 pixels
constexpr int kThreadsD = 7 * 32;
constexpr int kMaxB = 12;               // weight ring depth limit

struct Params {
  int B, H, W, Cin;           // input image (pixel H16 rows [B*H*W][4 * Cin bytes])
  int taps, kw, stride, pad;  // conv geometry (taps = kh * kw); transposed conv: taps = up * up
  int up;                     // 1 = convolution; > 1 = transposed conv with kernel = stride = up
  int oH, oW;                 // extent of the tiled grid (conv: output image; transposed: input image)
  int tiles_x, tiles_y, n_ntiles;
  int cout;                   // valid output channels (N tiles are zero-padded above it)
  int out_H, out_W;           // output image
  int out_C, out_c0;          // H16 output: channels per row and first channel written by this layer
  int relu;
  const uint8_t *packed_w;    // [n_ntiles][taps][Cin / 16] k-blocks of 64 * N bytes
  const float *scale, *shift;
  uint8_t *out_h16;           // or null
  float *out_nchw;            // fp32 planes [B, cout, out_H, out_W] or null
  int32_t *status;            // bit 0: fp16 range overflow while writing out_h16
  // grouped mode (the 36 output convs of the CenterHead as ONE launch): N tile nt reads input channels
  // [nt * Cin, (nt + 1) * Cin) of an image with in_C channels, uses weight tile nt, and writes its first grp_cnt[nt]
  // columns to the fp32 planes grp_plane0[nt] .. of out_nchw ([B, cout planes, out_H, out_W]); shift is [n_ntiles][N]
  int grouped, in_C;
  const int32_t *grp_plane0, *grp_cnt;
  int base_offset_mode;       // 0 (default, measured correct): base_offset field zero; 1: address bits 7-9 (wrong results)
  int w_bytes;                // weight-stationary kernel: bytes of one N tile's weight image (taps * Cin / 16 k-blocks)
};

// PITCH: pixels per row of the haloed tile in shared memory: 10 (tight: 8 + 2) or 16 (8-row groups stay 1024-byte aligned)
// WS ("weight-stationary", HALO only): the whole weight image of an N tile (taps * Cin / 16 k-blocks, <= 144 KB) stays in
// shared memory while the CTA walks a contiguous range of pixel tiles of that N tile; only the haloed activation tiles
// stream.  For layers with few input and many output channels (the 64 -> 36 x 64 ConvModules of the CenterHead) this
// replaces 43 B/clk of weight ingest per SM - the L2 -> SM limit - by 13 B/clk of activations.
template <int N, int MT, bool HALO, int PITCH, bool WS = false>
struct Cfg {
  static constexpr int A_ROWS = HALO ? PITCH * (kTH * MT + 2) : kM * MT;     // rows of 128 bytes per activation buffer
  static constexpr int A_BYTES = ((A_ROWS * 128 + 1023) / 1024) * 1024;
  static constexpr int NA = WS ? 3 : (HALO ? 2 : 3);                         // activation buffers
  static constexpr int B_BYTES = 128 * N;                                    // weight blocks of one (tap, group): 2 k-blocks
  static constexpr int B_BLK = 64 * N;
  static constexpr int BUDGET = (227 - 6) * 1024 - NA * A_BYTES;  // 227 KB - alignment slack - static (barriers, scale / shift)
  static constexpr int NB_RAW = BUDGET / B_BYTES;
  static constexpr int NB = NB_RAW > kMaxB ? kMaxB : NB_RAW;                 // weight ring depth
  static constexpr int ACC_COLS = MT * 2 * N;                                // TMEM columns of one accumulator set
  static constexpr int NBUF = (2 * ACC_COLS <= 512) ? 2 : 1;                 // double-buffered accumulators when they fit
  static constexpr int TMEM_COLS = (NBUF * ACC_COLS <= 64) ? 64 : (NBUF * ACC_COLS <= 128) ? 128 : (NBUF * ACC_COLS <= 256) ? 256 : 512;
  static constexpr uint32_t IDESC2 = (1u << 4) | (static_cast<uint32_t>((2 * N) >> 3) << 17) | (static_cast<uint32_t>(kM >> 4) << 24);
  static constexpr uint32_t IDESC1 = (1u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(kM >> 4) << 24);
  static_assert(N == 16 || N == 64 || N == 128, "N tile: 16 (grouped output convs), 64 or 128");
  static_assert(MT == 1 || MT == 2, "one or two M tiles");
  static_assert(WS || NB >= 4, "weight ring too shallow");
  static_assert(!WS || (HALO && MT == 1), "weight-stationary: haloed 3x3 tiles, one M tile");
  static_assert(ACC_COLS <= 512, "accumulators exceed TMEM");
};

// SWIZZLE_128B K-major descriptor with an explicit 8-row-group stride and the base offset of a start address that is not
// 1024-byte aligned (bits 7-9 of the address: the row phase of the swizzle pattern)
__device__ __forceinline__ uint64_t desc_sw128_at(uint32_t addr, uint32_t sbo_bytes, int bo_mode) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((addr & 0x3ffffu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= 1ull << 46;
  if (bo_mode) d |= static_cast<uint64_t>((addr >> 7) & 7u) << 49;
  d |= 2ull << 61;
  return d;
}
__device__ __forceinline__ void mma_f16_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void commit_elect(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_tile4d(uint32_t dst, const CUtensorMap *map, int c, int x, int y, int b, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cta.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::
          "r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c), "r"(x), "r"(y), "r"(b), "r"(bar)
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
struct Item {
  int nt, tap0, tx0, ty0, b;
};
template <bool WS = false>
__device__ __forceinline__ Item decode(long long w, const Params &p, int th) {
  Item it;
  long long q = w;
  if (WS) {  // N tile slowest: a CTA's contiguous item range stays on one N tile
    const long long pix = static_cast<long long>(p.B) * p.tiles_y * p.tiles_x;
    it.nt = static_cast<int>(q / pix);
    q -= it.nt * pix;
  } else {
    it.nt = static_cast<int>(q % p.n_ntiles);
    q /= p.n_ntiles;
  }
  it.tap0 = 0;
  if (p.up > 1) {
    const int up2 = p.up * p.up;
    it.tap0 = static_cast<int>(q % up2);
    q /= up2;
  }
  it.tx0 = static_cast<int>(q % p.tiles_x) * kTW;
  q /= p.tiles_x;
  it.ty0 = static_cast<int>(q % p.tiles_y) * th;
  it.b = static_cast<int>(q / p.tiles_y);
  return it;
}

template <int N, int MT, bool HALO, int PITCH, bool WS = false>
__global__ void __launch_bounds__(kThreadsD, 1)
    dense_conv_f16_kernel(const __grid_constant__ CUtensorMap in_map, const Params p) {
  using C = Cfg<N, MT, HALO, PITCH, WS>;
  constexpr int TH = kTH * MT;  // output tile height
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int up2 = p.up * p.up;
  const long long n_total = static_cast<long long>(p.B) * p.tiles_y * p.tiles_x * p.n_ntiles * (p.up > 1 ? up2 : 1);
  if (static_cast<long long>(blockIdx.x) >= n_total) return;
  // item sequence of this CTA: round robin (N tile fastest), or for WS a contiguous range (N tile slowest)
  const long long w_first = WS ? (static_cast<long long>(blockIdx.x) * n_total) / gridDim.x : blockIdx.x;
  const long long n_work = WS ? (static_cast<long long>(blockIdx.x + 1) * n_total) / gridDim.x : n_total;
  const long long w_step = WS ? 1 : gridDim.x;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) unsigned long long s_bar[2 * 3 + 2 * kMaxB + 4 + 2];
  // activation buffers: full[NA] empty[NA] | weight ring: full[NB] empty[NB] | accumulators: full[2] empty[2] |
  // weight-stationary image: landed, free
  constexpr int kAF = 0, kAE = 3, kBF = 6, kBE = 6 + kMaxB, kTF = 6 + 2 * kMaxB, kTE = kTF + 2, kWF = kTE + 2, kWE = kWF + 1;
  __shared__ uint32_t s_tmem_base;
  __shared__ float s_scale[2][N], s_shift[2][N];  // per accumulator buffer: the item's N-tile slice

  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  if (tid == 4 * 32) {
    for (int s = 0; s < C::NA; ++s) {
      mbar_init(smem_u32(&s_bar[kAF + s]), 1);
      mbar_init(smem_u32(&s_bar[kAE + s]), 1);
    }
    for (int s = 0; s < (WS ? 0 : C::NB); ++s) {
      mbar_init(smem_u32(&s_bar[kBF + s]), 1);
      mbar_init(smem_u32(&s_bar[kBE + s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&s_bar[kTF + b]), 1);
      mbar_init(smem_u32(&s_bar[kTE + b]), 4);
    }
    mbar_init(smem_u32(&s_bar[kWF]), 1);
    mbar_init(smem_u32(&s_bar[kWE]), 1);
    fence_mbar_init();
  }
  if (wid == 4) {
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
  const uint32_t a_ring = smem_u32(smem);
  const uint32_t b_ring = a_ring + C::NA * C::A_BYTES;
  const int G = p.Cin / 32;
  // A-units per item: HALO: one per group (serves all taps); TAP: one per (tap, group)
  const int taps_item = p.up > 1 ? 1 : p.taps;

  if (wid < 4) {
    // ------------------------------------------------------------------------------------------ epilogue
    asm volatile("griddepcontrol.wait;" ::: "memory");
    bool ovf = false;
    int it = 0;
    for (long long w = w_first; w < n_work; w += w_step, ++it) {
      const int buf = (C::NBUF == 2) ? (it & 1) : 0;
      const int use = (C::NBUF == 2) ? (it >> 1) : it;
      const Item im = decode<WS>(w, p, TH);
      // this item's per-channel epilogue constants (one thread per channel of the N tile)
      if (tid < N) {
        const int ch = im.nt * N + tid;
        const bool okc = p.grouped ? true : ch < p.cout;
        s_scale[buf][tid] = (p.scale && okc) ? __ldg(p.scale + ch) : 1.0f;
        s_shift[buf][tid] = (p.shift && okc) ? __ldg(p.shift + ch) : 0.0f;
      }
      const int g_cnt = p.grouped ? __ldg(p.grp_cnt + im.nt) : 0, g_p0 = p.grouped ? __ldg(p.grp_plane0 + im.nt) : 0;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      mbar_wait(smem_u32(&s_bar[kTF + buf]), static_cast<uint32_t>(use & 1));
      tc_fence_after();
      const int m = tid;  // TMEM lane = pixel of the M tile
      const int py = m / kTW, px = m % kTW;
#pragma unroll 1
      for (int mt = 0; mt < MT; ++mt) {
        const int iy = im.ty0 + mt * kTH + py, ix = im.tx0 + px;
        const bool live = iy < p.oH && ix < p.oW;
        const int Y = iy * p.up + (p.up > 1 ? im.tap0 / p.up : 0), X = ix * p.up + (p.up > 1 ? im.tap0 % p.up : 0);
        const size_t opix = (static_cast<size_t>(im.b) * p.out_H + Y) * p.out_W + X;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(wid * 32) << 16) + static_cast<uint32_t>(buf * C::ACC_COLS + mt * 2 * N);
#pragma unroll 1
        for (int c0 = 0; c0 < N; c0 += 16) {
          uint32_t a[16], x[16];
          tmem_ld16(taddr + static_cast<uint32_t>(c0), a);
          tmem_ld16(taddr + static_cast<uint32_t>(N + c0), x);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (mt == MT - 1 && c0 + 16 >= N) {  // last read of the accumulators: hand the buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&s_bar[kTE + buf]));
          }
          const int ch0 = im.nt * N + c0;  // first output channel of this chunk
          if (live && (p.grouped ? c0 < g_cnt : ch0 < p.cout)) {
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float o = fmaf(__uint_as_float(x[j]), kLoInv, __uint_as_float(a[j]));
              o = fmaf(o, s_scale[buf][c0 + j], s_shift[buf][c0 + j]);
              if (p.relu) o = fmaxf(o, 0.f);
              v[j] = o;
            }
            if (p.out_h16) {  // channel counts of H16 layers are multiples of 16: whole chunks
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
              const int ch = p.out_c0 + ch0;
              uint8_t *op = p.out_h16 + opix * (4 * static_cast<size_t>(p.out_C)) + (ch / 32) * 128 + (ch % 32) * 2;
              reinterpret_cast<uint4 *>(op)[0] = make_uint4(hw[0], hw[1], hw[2], hw[3]);
              reinterpret_cast<uint4 *>(op)[1] = make_uint4(hw[4], hw[5], hw[6], hw[7]);
              reinterpret_cast<uint4 *>(op + 64)[0] = make_uint4(lw[0], lw[1], lw[2], lw[3]);
              reinterpret_cast<uint4 *>(op + 64)[1] = make_uint4(lw[4], lw[5], lw[6], lw[7]);
            }
            if (p.out_nchw) {
              if (p.grouped) {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  if (c0 + j < g_cnt)
                    p.out_nchw[((static_cast<size_t>(im.b) * p.cout + g_p0 + c0 + j) * p.out_H + Y) * p.out_W + X] = v[j];
              } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  if (ch0 + j < p.cout)
                    p.out_nchw[((static_cast<size_t>(im.b) * p.cout + ch0 + j) * p.out_H + Y) * p.out_W + X] = v[j];
              }
            }
          }
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");  // s_scale / s_shift of this buffer are rewritten two items later
    }
    if (ovf && p.status) atomicOr(p.status, 1);
  } else if (wid == 4) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    int sa = 0, sb = 0;
    uint32_t pa = 0, pb = 0;  // parities to wait for on a_full[sa] / b_full[sb]
    int it = 0;
    int cur_nt = -1;
    uint32_t pw = 0;
    for (long long w = w_first; w < n_work; w += w_step, ++it) {
      const int buf = (C::NBUF == 2) ? (it & 1) : 0;
      const int use = (C::NBUF == 2) ? (it >> 1) : it;
      mbar_wait(smem_u32(&s_bar[kTE + buf]), static_cast<uint32_t>((use & 1) ^ 1));  // epilogue of the previous use done
      tc_fence_after();
      int nt_next = -1;
      if (WS) {
        const int nt = decode<WS>(w, p, TH).nt;
        if (nt != cur_nt) {  // first item of a run on this N tile: its weight image has to have landed
          mbar_wait(smem_u32(&s_bar[kWF]), pw);
          pw ^= 1u;
          tc_fence_after();
          cur_nt = nt;
        }
        nt_next = (w + w_step < n_work) ? decode<WS>(w + w_step, p, TH).nt : -1;
      }
      const uint32_t acc = tmem_base + static_cast<uint32_t>(buf * C::ACC_COLS);
      const int n_a = HALO ? G : taps_item * G;
      for (int ua = 0; ua < n_a; ++ua) {
        mbar_wait(smem_u32(&s_bar[kAF + sa]), pa);
        tc_fence_after();
        const uint32_t a_base = a_ring + static_cast<uint32_t>(sa * C::A_BYTES);
        const int n_t = HALO ? 9 : 1;
        for (int t = 0; t < n_t; ++t) {
          if (!WS) {
            mbar_wait(smem_u32(&s_bar[kBF + sb]), pb);
            tc_fence_after();
          }
          const uint32_t b_base = WS ? b_ring + static_cast<uint32_t>((t * (p.Cin / 16) + 2 * ua) * C::B_BLK)
                                     : b_ring + static_cast<uint32_t>(sb * C::B_BYTES);
#pragma unroll
          for (int kb = 0; kb < 2; ++kb) {
            const uint64_t db = smem_desc(b_base + static_cast<uint32_t>(kb * C::B_BLK), 2 * N * 16, 128);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
              uint32_t a0;
              uint32_t sbo;
              if (HALO) {
                a0 = a_base + static_cast<uint32_t>(((mt * kTH + t / 3) * PITCH + t % 3) * 128);
                sbo = PITCH * 128;
              } else {
                a0 = a_base + static_cast<uint32_t>(mt * kM * 128);
                sbo = 1024;
              }
              const uint32_t first = (ua | t | kb) ? 1u : 0u;
              mma_f16_elect(acc + mt * 2 * N, desc_sw128_at(a0 + kb * 32, sbo, p.base_offset_mode), db, C::IDESC2, first);         // A_hi x [B_hi | B_lo']
              mma_f16_elect(acc + mt * 2 * N + N, desc_sw128_at(a0 + (2 + kb) * 32, sbo, p.base_offset_mode), db, C::IDESC1, 1u);  // A_lo' x B_hi
            }
          }
          if (!WS) {
            commit_elect(smem_u32(&s_bar[kBE + sb]));
            if (++sb == C::NB) {
              sb = 0;
              pb ^= 1u;
            }
          }
        }
        commit_elect(smem_u32(&s_bar[kAE + sa]));
        if (ua == n_a - 1) {
          commit_elect(smem_u32(&s_bar[kTF + buf]));
          if (WS && nt_next != cur_nt) commit_elect(smem_u32(&s_bar[kWE]));  // last MMAs of this N tile: image may be replaced
        }
        if (++sa == C::NA) {
          sa = 0;
          pa ^= 1u;
        }
      }
    }
    tc_fence_before();
  } else if (wid == 5) {
    // ------------------------------------------------------------------------------------------ activation TMA (one lane)
    if (lane == 0) {
      asm volatile("griddepcontrol.wait;" ::: "memory");  // the input image is the previous layer's output
      int sa = 0;
      uint32_t pe = 1;
      for (long long w = w_first; w < n_work; w += w_step) {
        const Item im = decode<WS>(w, p, TH);
        const int cg0 = p.grouped ? im.nt * G : 0;  // first 32-channel group of this item's input channels
        if (HALO) {
          for (int g = 0; g < G; ++g) {
            mbar_wait(smem_u32(&s_bar[kAE + sa]), pe);
            const uint32_t bar = smem_u32(&s_bar[kAF + sa]);
            mbar_arrive_expect_tx(bar, static_cast<uint32_t>(C::A_ROWS * 128));
            tma_tile4d(a_ring + static_cast<uint32_t>(sa * C::A_BYTES), &in_map, (cg0 + g) * 64, im.tx0 - 1, im.ty0 - 1, im.b, bar);
            if (++sa == C::NA) {
              sa = 0;
              pe ^= 1u;
            }
          }
        } else {
          const int t_begin = p.up > 1 ? im.tap0 : 0, t_end = p.up > 1 ? im.tap0 + 1 : p.taps;
          for (int t = t_begin; t < t_end; ++t) {
            const int dy = p.up > 1 ? 0 : t / p.kw, dx = p.up > 1 ? 0 : t % p.kw;
            const int x = im.tx0 * p.stride - p.pad + dx, y = im.ty0 * p.stride - p.pad + dy;  // may be negative: zero fill
            for (int g = 0; g < G; ++g) {
              mbar_wait(smem_u32(&s_bar[kAE + sa]), pe);
              const uint32_t bar = smem_u32(&s_bar[kAF + sa]);
              mbar_arrive_expect_tx(bar, static_cast<uint32_t>(C::A_ROWS * 128));
              tma_tile4d(a_ring + static_cast<uint32_t>(sa * C::A_BYTES), &in_map, (cg0 + g) * 64, x, y, im.b, bar);
              if (++sa == C::NA) {
                sa = 0;
                pe ^= 1u;
              }
            }
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------ weight blocks (one lane)
    if (lane == 0 && WS) {
      int cur_nt = -1;
      uint32_t pe = 1;
      for (long long w = w_first; w < n_work; w += w_step) {
        const int nt = decode<WS>(w, p, TH).nt;
        if (nt == cur_nt) continue;
        cur_nt = nt;
        mbar_wait(smem_u32(&s_bar[kWE]), pe);  // the MMAs reading the previous image have completed
        pe ^= 1u;
        const uint32_t bar = smem_u32(&s_bar[kWF]);
        mbar_arrive_expect_tx(bar, static_cast<uint32_t>(p.w_bytes));
        const uint8_t *w_tile = p.packed_w + static_cast<size_t>(nt) * p.w_bytes;
        for (int off = 0; off < p.w_bytes; off += 16384) {
          const int bytes = p.w_bytes - off < 16384 ? p.w_bytes - off : 16384;
          bulk_g2s(b_ring + static_cast<uint32_t>(off), w_tile + off, static_cast<uint32_t>(bytes), bar);
        }
      }
    } else if (lane == 0) {
      int sb = 0;
      uint32_t pe = 1;
      for (long long w = w_first; w < n_work; w += w_step) {
        const Item im = decode<WS>(w, p, TH);
        const uint8_t *w_tile = p.packed_w + static_cast<size_t>(im.nt) * p.taps * (p.Cin / 16) * C::B_BLK;
        // same (A-unit, tap) order as the MMA warp: HALO: group-major, taps inside; TAP: tap-major, groups inside
        const int t_begin = p.up > 1 ? im.tap0 : 0, t_end = p.up > 1 ? im.tap0 + 1 : p.taps;
        const int outer = HALO ? G : (t_end - t_begin), inner = HALO ? 9 : G;
        for (int o = 0; o < outer; ++o)
          for (int i = 0; i < inner; ++i) {
            const int t = HALO ? i : t_begin + o, g = HALO ? o : i;
            mbar_wait(smem_u32(&s_bar[kBE + sb]), pe);
            const uint32_t bar = smem_u32(&s_bar[kBF + sb]);
            mbar_arrive_expect_tx(bar, static_cast<uint32_t>(C::B_BYTES));
            bulk_g2s(b_ring + static_cast<uint32_t>(sb * C::B_BYTES),
                     w_tile + (static_cast<size_t>(t) * (p.Cin / 16) + 2 * g) * C::B_BLK, static_cast<uint32_t>(C::B_BYTES), bar);
            if (++sb == C::NB) {
              sb = 0;
              pe ^= 1u;
            }
          }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (wid == 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(static_cast<uint32_t>(C::TMEM_COLS))
                 : "memory");
  }
}

// fp32 NCHW image -> pixel H16 rows (32 x 32 tile transpose through shared memory)
__global__ void __launch_bounds__(256) nchw_to_pixel_h16_kernel(const float *__restrict__ in, int C, long long HW,
                                                                __half *__restrict__ out, int32_t *status) {
  __shared__ float s_t[32][33];
  const int b = blockIdx.z;
  const long long p0 = static_cast<long long>(blockIdx.x) * 32;
  const int c0 = blockIdx.y * 32;  // one 32-channel H16 group
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k;
    const long long px = p0 + tx;
    s_t[k][tx] = (c < C && px < HW) ? in[(static_cast<size_t>(b) * C + c) * HW + px] : 0.f;
  }
  __syncthreads();
  bool ovf = false;
  for (int k = ty; k < 32; k += 8) {
    const long long px = p0 + k;
    if (px < HW) {
      __half h, l;
      split_h16(s_t[tx][k], h, l, ovf);
      __half *grp = out + (static_cast<size_t>(b) * HW + px) * (2 * static_cast<size_t>(C)) + static_cast<size_t>(c0) * 2;
      grp[tx] = h;
      grp[32 + tx] = l;
    }
  }
  if (ovf && status) atomicOr(status, 1);
}

// pixel H16 rows -> fp32 NCHW (tests / debugging)
__global__ void __launch_bounds__(256) pixel_h16_to_nchw_kernel(const __half *__restrict__ in, int C, long long HW,
                                                                float *__restrict__ out, long long total) {
  const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= total) return;
  const long long px = q % HW;
  const int c = static_cast<int>((q / HW) % C);
  const long long b = q / (HW * C);
  const __half *grp = in + (b * HW + px) * (2 * static_cast<long long>(C)) + (c / 32) * 64;
  out[q] = fmaf(__half2float(grp[32 + c % 32]), kLoInv, __half2float(grp[c % 32]));
}

inline int make_image_map(const void *img, int B, int H, int W, int Cin, int stride, int box_x, int box_y, CUtensorMap *map) {
  // Cin = channels per pixel of the image in memory
  using Encode = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                              const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static Encode encode = nullptr;
  if (!encode) {
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) != cudaSuccess || !fn)
      return P3D_ERR_UNSUPPORTED;
    encode = reinterpret_cast<Encode>(fn);
  }
  const cuuint64_t row = static_cast<cuuint64_t>(4) * Cin;  // bytes per pixel
  const cuuint64_t gdim[4] = {static_cast<cuuint64_t>(2 * Cin), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                              static_cast<cuuint64_t>(B)};
  const cuuint64_t gstride[3] = {row, row * W, row * W * H};
  // with an element stride s the box extent is s x the number of elements loaded (cuda.h, cuTensorMapEncodeTiled)
  const cuuint32_t box[4] = {64u, static_cast<cuuint32_t>(box_x * stride), static_cast<cuuint32_t>(box_y * stride), 1u};
  const cuuint32_t estride[4] = {1u, static_cast<cuuint32_t>(stride), static_cast<cuuint32_t>(stride), 1u};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void *>(img), gdim, gstride, box, estride,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? P3D_OK : P3D_ERR_INVALID_ARG;
}

template <int N, int MT, bool HALO, int PITCH, bool WS = false>
int launch(const CUtensorMap &map, const Params &p, cudaStream_t st) {
  using C = Cfg<N, MT, HALO, PITCH, WS>;
  const size_t smem = static_cast<size_t>(C::NA) * C::A_BYTES +
                      (WS ? static_cast<size_t>(p.w_bytes) : static_cast<size_t>(C::NB) * C::B_BYTES) + 1024;
  if (smem > static_cast<size_t>(227 - 6) * 1024) return P3D_ERR_UNSUPPORTED;
  auto kern = dense_conv_f16_kernel<N, MT, HALO, PITCH, WS>;
  P3D_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const long long work = static_cast<long long>(p.B) * p.tiles_y * p.tiles_x * p.n_ntiles * (p.up > 1 ? p.up * p.up : 1);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned int>(work < kNumSMs ? work : kNumSMs));
  cfg.blockDim = dim3(kThreadsD);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  P3D_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, map, p));
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// CenterHead output convs with the 9 taps in the N dimension ("tap-as-N", center_head.py:80-117 SeparateHead finals).
//
// A 3x3 conv with <= 3 output channels is 9 * Cin/16 k-steps of N = 16 UMMAs per 128 pixels in the generic kernel above:
// 144 tiny MMAs per item, bound by the MMA issue latency (190 us for the 36 convs of the C3 head).  Here one item is a
// 16 x 16-pixel haloed tile (256 rows = 2 M tiles) of one group's Cin channels and ONE GEMM
//     P[pixel][tap * 3 + co] = sum_c  mid[pixel][c] * W[tap][c][co]            (N = 27 -> 32, K = Cin: 4 k-steps for 64)
// = 16 MMAs; the epilogue parks P in shared memory and every output pixel of the 14 x 14 interior adds its 9 shifted
// entries  out[y][x][co] = bias + sum_tap P[(y + dy) * 16 + x + dx][tap * 3 + co].  The kernel is then bound by reading
// the intermediate image once (x 1.31 halo overhead, mostly L2 hits).
//   warps 0-3 epilogue + tap sums   4 MMA issue   5 activation TMA   6 weight blocks
namespace out9 {
constexpr int kHT = 16, kOT = 14;                 // haloed / output tile side
constexpr int kRows = kHT * kHT;                  // 256 rows of 128 bytes per 32-channel group
constexpr int kABytes = kRows * 128;              // 32 KB
constexpr int kN = 32, kStride = 29;              // GEMM N, fp32 row stride of P in shared memory
constexpr int kWBlk = 64 * kN;                    // bytes of one 16-channel weight k-block ([2 chunks][2N rows][8 halfs])
constexpr int kPBytes = kRows * kStride * 4;
constexpr int kMaxNA = 5, kNW = 3;
constexpr uint32_t IDESC2 = (1u << 4) | (static_cast<uint32_t>((2 * kN) >> 3) << 17) | (static_cast<uint32_t>(kM >> 4) << 24);
constexpr uint32_t IDESC1 = (1u << 4) | (static_cast<uint32_t>(kN >> 3) << 17) | (static_cast<uint32_t>(kM >> 4) << 24);

struct Params {
  int B, H, W, G;              // image, 32-channel groups per conv group (Cin / 32)
  int tiles_x, tiles_y, groups, planes, NA;
  const uint8_t *packed_w;     // [groups][Cin / 16] k-blocks of W2[c][tap * 3 + co] (kWBlk bytes each)
  const float *bias;           // [groups][4]
  const int32_t *cin0;         // [groups] first input channel of the group's slice (multiple of 32) or null: g * Cin
  const int32_t *plane0, *cnt; // [groups]
  float *out;                  // [B, planes, H, W]
};

__global__ void __launch_bounds__(kThreadsD, 1) head_out9_kernel(const __grid_constant__ CUtensorMap in_map, const Params p) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const long long n_work = static_cast<long long>(p.B) * p.tiles_y * p.tiles_x * p.groups;
  if (static_cast<long long>(blockIdx.x) >= n_work) return;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) unsigned long long s_bar[2 * kMaxNA + 2 * kNW + 4];
  constexpr int kAF = 0, kAE = kMaxNA, kWF = 2 * kMaxNA, kWE = kWF + kNW, kTF = kWE + kNW, kTE = kTF + 2;
  __shared__ uint32_t s_tmem_base;
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  const int NA = p.NA, G = p.G;
  const uint32_t w_slot = static_cast<uint32_t>(2 * G * kWBlk);
  if (tid == 4 * 32) {
    for (int s = 0; s < kMaxNA; ++s) {
      mbar_init(smem_u32(&s_bar[kAF + s]), 1);
      mbar_init(smem_u32(&s_bar[kAE + s]), 1);
    }
    for (int s = 0; s < kNW; ++s) {
      mbar_init(smem_u32(&s_bar[kWF + s]), 1);
      mbar_init(smem_u32(&s_bar[kWE + s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&s_bar[kTF + b]), 1);
      mbar_init(smem_u32(&s_bar[kTE + b]), 4);
    }
    fence_mbar_init();
  }
  if (wid == 4) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem_base)), "r"(256u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;
  const uint32_t a_ring = smem_u32(smem);
  const uint32_t w_ring = a_ring + static_cast<uint32_t>(NA * kABytes);
  float *s_p = reinterpret_cast<float *>(smem + static_cast<size_t>(NA) * kABytes + static_cast<size_t>(kNW) * w_slot);

  auto decode = [&](long long w, int &g, int &tx0, int &ty0, int &b) {
    g = static_cast<int>(w % p.groups);
    long long q = w / p.groups;
    tx0 = static_cast<int>(q % p.tiles_x) * kOT;
    q /= p.tiles_x;
    ty0 = static_cast<int>(q % p.tiles_y) * kOT;
    b = static_cast<int>(q / p.tiles_y);
  };

  if (wid < 4) {
    // ------------------------------------------------------------------------------------------ epilogue + tap sums
    asm volatile("griddepcontrol.wait;" ::: "memory");
    int it = 0;
    for (long long w = blockIdx.x; w < n_work; w += gridDim.x, ++it) {
      const int buf = it & 1, use = it >> 1;
      int g, tx0, ty0, b;
      decode(w, g, tx0, ty0, b);
      const int cnt = __ldg(p.cnt + g), p0 = __ldg(p.plane0 + g);
      const float4 bias = __ldg(reinterpret_cast<const float4 *>(p.bias) + g);
      mbar_wait(smem_u32(&s_bar[kTF + buf]), static_cast<uint32_t>(use & 1));
      tc_fence_after();
#pragma unroll 1
      for (int mt = 0; mt < 2; ++mt) {
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(wid * 32) << 16) + static_cast<uint32_t>(buf * 128 + mt * 64);
        uint32_t a0[16], a1[16], x0[16], x1[16];
        tmem_ld16(taddr, a0);
        tmem_ld16(taddr + 16, a1);
        tmem_ld16(taddr + 32, x0);
        tmem_ld16(taddr + 48, x1);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (mt == 1) {  // accumulators read: hand the buffer back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(&s_bar[kTE + buf]));
        }
        float *row = s_p + (mt * 128 + tid) * kStride;
#pragma unroll
        for (int j = 0; j < 16; ++j) row[j] = fmaf(__uint_as_float(x0[j]), kLoInv, __uint_as_float(a0[j]));
#pragma unroll
        for (int j = 0; j < 11; ++j) row[16 + j] = fmaf(__uint_as_float(x1[j]), kLoInv, __uint_as_float(a1[j]));
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      for (int o = tid; o < kOT * kOT; o += 128) {
        const int oy = o / kOT, ox = o - oy * kOT;
        const int Y = ty0 + oy, X = tx0 + ox;
        if (Y < p.H && X < p.W) {
          float s0 = bias.x, s1 = bias.y, s2 = bias.z;
#pragma unroll
          for (int t = 0; t < 9; ++t) {
            const float *e = s_p + ((oy + t / 3) * kHT + ox + t % 3) * kStride + t * 3;
            s0 += e[0];
            s1 += e[1];
            s2 += e[2];
          }
          float *op = p.out + ((static_cast<size_t>(b) * p.planes + p0) * p.H + Y) * p.W + X;
          const size_t plane = static_cast<size_t>(p.H) * p.W;
          op[0] = s0;
          if (cnt > 1) op[plane] = s1;
          if (cnt > 2) op[2 * plane] = s2;
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");  // P is rewritten by the next item
    }
  } else if (wid == 4) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    int sa = 0, sw = 0;
    uint32_t pa = 0, pw = 0;
    int it = 0;
    for (long long w = blockIdx.x; w < n_work; w += gridDim.x, ++it) {
      const int buf = it & 1, use = it >> 1;
      mbar_wait(smem_u32(&s_bar[kTE + buf]), static_cast<uint32_t>((use & 1) ^ 1));
      mbar_wait(smem_u32(&s_bar[kWF + sw]), pw);
      tc_fence_after();
      const uint32_t acc = tmem_base + static_cast<uint32_t>(buf * 128);
      const uint32_t w_base = w_ring + static_cast<uint32_t>(sw) * w_slot;
      for (int g = 0; g < G; ++g) {
        mbar_wait(smem_u32(&s_bar[kAF + sa]), pa);
        tc_fence_after();
        const uint32_t a_base = a_ring + static_cast<uint32_t>(sa * kABytes);
#pragma unroll
        for (int kb = 0; kb < 2; ++kb) {
          const uint64_t db = smem_desc(w_base + static_cast<uint32_t>((g * 2 + kb) * kWBlk), 2 * kN * 16, 128);
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
            const uint32_t a0 = a_base + static_cast<uint32_t>(mt * kM * 128);
            mma_f16_elect(acc + mt * 64, desc_sw128_at(a0 + kb * 32, 1024, 0), db, IDESC2, (g | kb) ? 1u : 0u);
            mma_f16_elect(acc + mt * 64 + kN, desc_sw128_at(a0 + (2 + kb) * 32, 1024, 0), db, IDESC1, 1u);
          }
        }
        commit_elect(smem_u32(&s_bar[kAE + sa]));
        if (++sa == NA) {
          sa = 0;
          pa ^= 1u;
        }
      }
      commit_elect(smem_u32(&s_bar[kWE + sw]));
      commit_elect(smem_u32(&s_bar[kTF + buf]));
      if (++sw == kNW) {
        sw = 0;
        pw ^= 1u;
      }
    }
    tc_fence_before();
  } else if (wid == 5) {
    // ------------------------------------------------------------------------------------------ activation TMA (one lane)
    if (lane == 0) {
      asm volatile("griddepcontrol.wait;" ::: "memory");
      int sa = 0;
      uint32_t pe = 1;
      for (long long w = blockIdx.x; w < n_work; w += gridDim.x) {
        int g, tx0, ty0, b;
        decode(w, g, tx0, ty0, b);
        const int cg0 = (p.cin0 ? __ldg(p.cin0 + g) : g * G * 32) / 32;
        for (int k = 0; k < G; ++k) {
          mbar_wait(smem_u32(&s_bar[kAE + sa]), pe);
          const uint32_t bar = smem_u32(&s_bar[kAF + sa]);
          mbar_arrive_expect_tx(bar, static_cast<uint32_t>(kABytes));
          tma_tile4d(a_ring + static_cast<uint32_t>(sa * kABytes), &in_map, (cg0 + k) * 64, tx0 - 1, ty0 - 1, b, bar);
          if (++sa == NA) {
            sa = 0;
            pe ^= 1u;
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------ weights (one lane)
    if (lane == 0) {
      int sw = 0;
      uint32_t pe = 1;
      for (long long w = blockIdx.x; w < n_work; w += gridDim.x) {
        const int g = static_cast<int>(w % p.groups);
        mbar_wait(smem_u32(&s_bar[kWE + sw]), pe);
        const uint32_t bar = smem_u32(&s_bar[kWF + sw]);
        mbar_arrive_expect_tx(bar, w_slot);
        bulk_g2s(w_ring + static_cast<uint32_t>(sw) * w_slot, p.packed_w + static_cast<size_t>(g) * w_slot, w_slot, bar);
        if (++sw == kNW) {
          sw = 0;
          pe ^= 1u;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (wid == 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u) : "memory");
  }
}
}  // namespace out9

}  // namespace dcf
}  // namespace p3d

using namespace p3d;

extern "C" int p3d_nchw_to_pixel_h16(const float *in, int B, int C, int H, int W, void *out_h16, int32_t *status_dev,
                                     p3d_stream_t stream) {
  if (!in || !out_h16 || B < 1 || C < 32 || C % 32 || H < 1 || W < 1) return P3D_ERR_INVALID_ARG;
  const long long hw = static_cast<long long>(H) * W;
  dim3 grid(static_cast<unsigned int>((hw + 31) / 32), static_cast<unsigned int>(C / 32), B);
  dcf::nchw_to_pixel_h16_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(in, C, hw, static_cast<__half *>(out_h16),
                                                                                      status_dev);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

extern "C" int p3d_pixel_h16_to_nchw(const void *in_h16, int B, int C, int H, int W, float *out, p3d_stream_t stream) {
  if (!in_h16 || !out || B < 1 || C < 32 || C % 32 || H < 1 || W < 1) return P3D_ERR_INVALID_ARG;
  const long long hw = static_cast<long long>(H) * W, total = hw * C * B;
  dcf::pixel_h16_to_nchw_kernel<<<div_up(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __half *>(in_h16), C, hw, out, total);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

// packed weights: per N tile the image p3d_sparse_conv_f16_pack_weights makes of W[tap][Cin][n_tile] (zero-padded columns)
extern "C" size_t p3d_dense_conv2d_f16_packed_weight_bytes(int taps, int Cin, int Cout, int n_tile) {
  if (taps < 1 || Cin < 32 || Cin % 32 || Cout < 1 || (n_tile != 16 && n_tile != 32 && n_tile != 64 && n_tile != 128)) return 0;
  const size_t tiles = static_cast<size_t>((Cout + n_tile - 1) / n_tile);
  return align_up(tiles * taps * Cin * static_cast<size_t>(n_tile) * 4);
}

// mode: 0 auto (HALO for 3x3 stride 1 pad 1 convolutions - weight-stationary when it applies -, TAP otherwise), 1 force TAP,
// 2 force the weight-stationary kernel (P3D_ERR_UNSUPPORTED when it does not apply); m_tiles: 0 auto, 1 or 2
static int dense_conv_f16(const void *in_h16, int B, int H, int W, int Cin, const void *packed_weight, int Cout, int n_tile,
                          int kh, int kw, int stride, int pad, int up, const float *scale, const float *shift, int relu,
                          void *out_h16, int out_C, int out_c0, float *out_nchw, int mode, int m_tiles, int32_t *status_dev,
                          p3d_stream_t stream, int groups, int in_C, const int32_t *grp_plane0, const int32_t *grp_cnt) {
  if (!in_h16 || !packed_weight || (!out_h16 && !out_nchw) || B < 1 || H < 1 || W < 1 || Cout < 1) return P3D_ERR_INVALID_ARG;
  if (Cin < 32 || Cin % 32 || (n_tile != 64 && n_tile != 128 && !(groups && n_tile == 16))) return P3D_ERR_UNSUPPORTED;
  if (up < 1 || (up > 1 && (kh != up || kw != up || stride != up || pad != 0))) return P3D_ERR_UNSUPPORTED;
  if (up == 1 && (kh < 1 || kw < 1 || kh * kw > 32 || stride < 1 || stride > 2 || pad < 0)) return P3D_ERR_UNSUPPORTED;
  if (out_h16 && (Cout % 16 || out_C % 32 || out_c0 % 16 || out_c0 + Cout > out_C)) return P3D_ERR_INVALID_ARG;
  if ((reinterpret_cast<uintptr_t>(in_h16) & 15) || (reinterpret_cast<uintptr_t>(packed_weight) & 15) ||
      (reinterpret_cast<uintptr_t>(out_h16) & 15))
    return P3D_ERR_INVALID_ARG;
  dcf::Params p;
  p.B = B;
  p.H = H;
  p.W = W;
  p.Cin = Cin;
  p.taps = kh * kw;
  p.kw = kw;
  p.up = up;
  p.stride = up > 1 ? 1 : stride;
  p.pad = up > 1 ? 0 : pad;
  p.oH = up > 1 ? H : (H + 2 * pad - kh) / stride + 1;
  p.oW = up > 1 ? W : (W + 2 * pad - kw) / stride + 1;
  if (p.oH < 1 || p.oW < 1) return P3D_ERR_INVALID_ARG;
  p.out_H = up > 1 ? H * up : p.oH;
  p.out_W = up > 1 ? W * up : p.oW;
  p.n_ntiles = groups ? groups : (Cout + n_tile - 1) / n_tile;
  p.cout = Cout;
  p.grouped = groups ? 1 : 0;
  p.in_C = groups ? in_C : Cin;
  p.grp_plane0 = grp_plane0;
  p.grp_cnt = grp_cnt;
  p.out_C = out_C;
  p.out_c0 = out_c0;
  p.relu = relu;
  p.packed_w = static_cast<const uint8_t *>(packed_weight);
  p.scale = scale;
  p.shift = shift;
  p.out_h16 = static_cast<uint8_t *>(out_h16);
  p.out_nchw = out_nchw;
  p.status = status_dev;
  static const int env_mode = getenv("P3D_DENSE_MODE") ? atoi(getenv("P3D_DENSE_MODE")) : -1;  // tuning hooks
  static const int env_mt = getenv("P3D_DENSE_MT") ? atoi(getenv("P3D_DENSE_MT")) : -1;
  static const int env_pitch = getenv("P3D_DENSE_PITCH") ? atoi(getenv("P3D_DENSE_PITCH")) : 10;
  // measured on the B200 (profiles/r02_dense_halo_probe.md): shifted tiles read correctly with base_offset = 0 (the swizzle
  // is a function of the absolute shared-memory address) and wrongly with base_offset = address bits 7-9
  static const int env_bo = getenv("P3D_DENSE_BO") ? atoi(getenv("P3D_DENSE_BO")) : 0;
  p.base_offset_mode = env_bo;
  const int pitch = env_pitch == 16 ? 16 : 10;
  if (env_mode >= 0) mode = env_mode;
  if (env_mt >= 0) m_tiles = env_mt;
  const bool halo = (mode == 0 || mode == 2) && up == 1 && kh == 3 && kw == 3 && stride == 1 && pad == 1;
  // two M tiles per item (half the weight traffic per flop) when that still leaves every SM an item
  int mt = m_tiles;
  if (mt != 1 && mt != 2) {
    const long long tx = (p.oW + dcf::kTW - 1) / dcf::kTW, ty2 = (p.oH + 2 * dcf::kTH - 1) / (2 * dcf::kTH);
    const long long items2 = static_cast<long long>(B) * tx * ty2 * p.n_ntiles * (up > 1 ? up * up : 1);
    // measured (profiles/r02_dense_bench.jsonl): two M tiles pay off for the narrow N = 64 layers (weights are a small
    // share, the second tile amortises the per-item prologue); N = 128 is faster with one tile and double-buffered
    // accumulators (the epilogue overlaps the next item)
    mt = (n_tile <= 64 && items2 >= (kNumSMs * 9) / 10) ? 2 : 1;
  }
  // weight-stationary variant: haloed 3x3, N tile 64, the N tile's weight image + 3 activation tiles fit in shared memory,
  // and every CTA has enough pixel tiles per weight image to amortise loading it (mode 2 forces it, P3D_DENSE_WS=0 disables)
  // Measured on the CenterHead's 64 -> 2304 layer (profiles/r02_dense_ws.md): 248 us against 236 us for the streaming
  // N = 128 kernel - the layer is bound by the shared-memory reads of the MMA operands (N = 64 needs 128-192 B/clk), not by
  // the weight ingest, so the variant is OFF unless asked for (mode 2 or P3D_DENSE_WS=1).
  static const int env_ws = getenv("P3D_DENSE_WS") ? atoi(getenv("P3D_DENSE_WS")) : 0;
  p.w_bytes = p.taps * (Cin / 16) * 64 * n_tile;
  bool ws = false;
  if (halo && n_tile == 64 && !groups && pitch == 10 && (env_ws || mode == 2)) {
    const size_t need = 3 * static_cast<size_t>(dcf::Cfg<64, 1, true, 10, true>::A_BYTES) + p.w_bytes + 1024;
    const long long pix = static_cast<long long>(B) * ((p.oW + dcf::kTW - 1) / dcf::kTW) * ((p.oH + dcf::kTH - 1) / dcf::kTH);
    const long long items = pix * p.n_ntiles;
    ws = need <= static_cast<size_t>(227 - 6) * 1024 && (mode == 2 || items >= 8ll * kNumSMs);
  }
  if (mode == 2 && !ws) return P3D_ERR_UNSUPPORTED;
  if (ws) mt = 1;
  p.tiles_x = (p.oW + dcf::kTW - 1) / dcf::kTW;
  p.tiles_y = (p.oH + dcf::kTH * mt - 1) / (dcf::kTH * mt);
  CUtensorMap map;
  const int bx = halo ? pitch : dcf::kTW, by = halo ? dcf::kTH * mt + 2 : dcf::kTH * mt;
  const int rc = dcf::make_image_map(in_h16, B, H, W, p.in_C, p.stride, bx, by, &map);
  if (rc != P3D_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (ws) return dcf::launch<64, 1, true, 10, true>(map, p, st);
#define P3D_DCF(NT, M)                                                                          \
  if (n_tile == NT && mt == M) {                                                                \
    if (!halo) return dcf::launch<NT, M, false, 10>(map, p, st);                                \
    if (pitch == 16) return dcf::launch<NT, M, true, 16>(map, p, st);                           \
    return dcf::launch<NT, M, true, 10>(map, p, st);                                            \
  }
  P3D_DCF(16, 1)
  P3D_DCF(16, 2)
  P3D_DCF(64, 1)
  P3D_DCF(64, 2)
  P3D_DCF(128, 1)
  P3D_DCF(128, 2)
#undef P3D_DCF
  return P3D_ERR_UNSUPPORTED;
}

extern "C" int p3d_dense_conv2d_f16(const void *in_h16, int B, int H, int W, int Cin, const void *packed_weight, int Cout,
                                    int n_tile, int kh, int kw, int stride, int pad, int up, const float *scale,
                                    const float *shift, int relu, void *out_h16, int out_C, int out_c0, float *out_nchw,
                                    int mode, int m_tiles, int32_t *status_dev, p3d_stream_t stream) {
  return dense_conv_f16(in_h16, B, H, W, Cin, packed_weight, Cout, n_tile, kh, kw, stride, pad, up, scale, shift, relu, out_h16,
                        out_C, out_c0, out_nchw, mode, m_tiles, status_dev, stream, 0, 0, nullptr, nullptr);
}

// Grouped 3x3 / stride 1 / pad 1 output convs (CenterHead SeparateHead finals, center_head.py:80-117) on the tensor cores:
// group g convolves input channels [g * Cin, (g + 1) * Cin) of the in_C-channel image with its own W[9][Cin][16]
// (columns >= cnt[g] zero) and writes cnt[g] fp32 planes from plane0[g] of out_nchw [B, planes, H, W].
// packed_weight: `groups` weight tiles of p3d_dense_conv2d_f16_pack_weights(taps 9, Cin, n_tile 16); bias [groups][16].
extern "C" int p3d_grouped_head_conv_f16(const void *in_h16, int B, int H, int W, int in_C, int Cin, int groups,
                                         const void *packed_weight, const float *bias, const int32_t *plane0_dev,
                                         const int32_t *cnt_dev, int planes, float *out_nchw, int32_t *status_dev,
                                         p3d_stream_t stream) {
  if (!plane0_dev || !cnt_dev || groups < 1 || groups * Cin > in_C || in_C % 32 || planes < 1) return P3D_ERR_INVALID_ARG;
  return dense_conv_f16(in_h16, B, H, W, Cin, packed_weight, planes, 16, 3, 3, 1, 1, 1, nullptr, bias, 0, nullptr, 32, 0, out_nchw,
                        0, 0, status_dev, stream, groups, in_C, plane0_dev, cnt_dev);
}

// Output convs of the CenterHead, 9 taps in the GEMM's N dimension (dcf::out9 above): group g convolves input channels
// [cin0[g], cin0[g] + Cin) (cin0 null: g * Cin) of the in_C-channel pixel fp16-pair image with its own 3x3 weights and
// writes cnt[g] <= 3 fp32 planes from plane0[g] of out_nchw [B, planes, H, W].  packed_weight: per group the image
// p3d_dense_conv2d_f16_pack_weights(taps 1, Cin, n_tile 32) makes of W2[c][tap * 3 + co]; bias [groups][4].
extern "C" int p3d_head_out_conv_f16(const void *in_h16, int B, int H, int W, int in_C, int Cin, int groups,
                                     const void *packed_weight, const float *bias, const int32_t *cin0_dev,
                                     const int32_t *plane0_dev, const int32_t *cnt_dev, int planes, float *out_nchw,
                                     p3d_stream_t stream) {
  if (!in_h16 || !packed_weight || !bias || !plane0_dev || !cnt_dev || !out_nchw || B < 1 || H < 1 || W < 1 || groups < 1 ||
      planes < 1 || in_C % 32 || Cin > in_C)
    return P3D_ERR_INVALID_ARG;
  if (Cin != 32 && Cin != 64 && Cin != 128) return P3D_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(in_h16) & 15) || (reinterpret_cast<uintptr_t>(packed_weight) & 15) ||
      (reinterpret_cast<uintptr_t>(bias) & 15))
    return P3D_ERR_INVALID_ARG;
  namespace o9 = dcf::out9;
  o9::Params p;
  p.B = B;
  p.H = H;
  p.W = W;
  p.G = Cin / 32;
  p.tiles_x = (W + o9::kOT - 1) / o9::kOT;
  p.tiles_y = (H + o9::kOT - 1) / o9::kOT;
  p.groups = groups;
  p.planes = planes;
  p.NA = p.G <= 2 ? 5 : 4;
  p.packed_w = static_cast<const uint8_t *>(packed_weight);
  p.bias = bias;
  p.cin0 = cin0_dev;
  p.plane0 = plane0_dev;
  p.cnt = cnt_dev;
  p.out = out_nchw;
  CUtensorMap map;
  const int rc = dcf::make_image_map(in_h16, B, H, W, in_C, 1, o9::kHT, o9::kHT, &map);
  if (rc != P3D_OK) return rc;
  const size_t smem = static_cast<size_t>(p.NA) * o9::kABytes + static_cast<size_t>(o9::kNW) * 2 * p.G * o9::kWBlk + o9::kPBytes + 1024;
  auto kern = o9::head_out9_kernel;
  P3D_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const long long work = static_cast<long long>(B) * p.tiles_y * p.tiles_x * groups;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned int>(work < kNumSMs ? work : kNumSMs));
  cfg.blockDim = dim3(dcf::kThreadsD);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  P3D_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, map, p));
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}
