// Sparse-conv gather-GEMM for the NARROW layers (Cin, Cout <= 32) on fp16 hi/lo' pair rows: register gather + warp MMA.
//
// Why a second kernel next to sparse_conv_f16.cu (tcgen05): on the 16- and 32-channel levels the tcgen05 pipeline is
// bound by what it costs to stage a gathered row in shared memory, not by the tensor pipe (profiles/r02_f16_sweep.md:
// a missing neighbour costs a full cp.async slot, 55 % of the slots are missing neighbours, one full/empty mbarrier
// round trip per 2-4 taps) - a level-0 layer takes 44 us for 0.38 GFLOP.  Here nothing is staged:
//
//   * the product is computed TRANSPOSED, out^T[cout][row] = W^T[cout][k] x X^T[k][row] with mma.sync.m16n8k16: the
//     weights are the A operand (16 output channels x 16 k), 8 gathered rows are the B operand.  A lane's B fragment
//     (k-slots 2t, 2t+1, 2t+8, 2t+9 of column g) then belongs to ONE row, and with the k dimension permuted so that these
//     four slots are 4 contiguous channels it is one vector load (8 B for Cin = 16, 16 B = two k-steps for Cin = 32) per
//     row half, straight from L2 into the registers the MMA reads - no shared-memory staging, no shuffles, no moves;
//     a missing neighbour is a predicated-off load (no request, no bytes);
//   * the weight image is packed with the same permutation, in A-fragment order, and sits in shared memory for the
//     whole kernel (27-110 KB): one conflict-free LDS.128 per fragment;
//   * a warp owns 16 output rows (two 8-row B tiles); loads run D taps ahead of the MMAs in a register ring of
//     compile-time slots ("groups" of up to D taps of one tile) that prefetches across tile boundaries; the neighbour
//     indices of the next tile are staged with cp.async while the current one is computed;
//   * work is cut stream-K style: the (tile, tap) units are divided into one equal contiguous range per warp of the grid
//     (no wave quantisation: 2471 tiles on 2368 warps would otherwise take two rounds); a tile cut by a range boundary
//     is summed by the LAST warp to finish it (ticket), pieces in warp order -> deterministic;
//   * products exactly as the tcgen05 kernel: acc_m += hi x hi, acc_l += hi x lo' + lo' x hi (fp32 accumulators),
//     out = acc_m + acc_l * 2^-11, then the same fused BN / bias / residual / ReLU epilogue (transposed back through a
//     per-warp shared-memory tile so that rows are read and written 16 bytes at a time) and the same H16 / fp32 outputs:
//     a drop-in for p3d_sparse_conv_f16 on these shapes.
//
// The tcgen05 pipe is irrelevant at these widths (N = 16/32): the bounds are the L2 gather (pairs x 4 Cin bytes), the
// issue slots of the gather loop and, for 32 -> 32, the legacy HMMA rate - see DESIGN.md section 3 / 6.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "h16.cuh"

namespace p3d {
namespace wm {

constexpr int kWarps = 16;  // warps per CTA of every instantiation, one CTA per SM

struct Params {
  const uint8_t *in;         // H16 rows [n_in][4 * CIN bytes]
  const int32_t *nbr;        // [n_cap][K]
  const int32_t *n_out_dev;  // device row count (or null: n_cap)
  long long n_cap;
  int K;
  const uint4 *packed_w;     // [K][CIN / 16][COUT / 16][2: hi, lo'][32 lanes] x (a0, a1, a2, a3)
  const float *scale, *shift;
  const uint8_t *residual;   // H16 rows [n][4 * COUT bytes] or null
  int relu;
  float *out_f32;            // [n][COUT] or null
  uint8_t *out_h16;          // [n][4 * COUT bytes] or null
  int32_t *status;           // bit 0: fp16 range overflow while producing out_h16
  float *slabs;              // stream-K partial tiles [warps of the grid][2][COUT / 2][32 lanes]
  int32_t *tickets;          // [tiles] arrival counters of split tiles, zero on entry, left zero
};

__device__ __forceinline__ void mma16816(float (&c)[4], const uint4 &a, uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b0), "r"(b1));
}


// B-fragment words of one (tile, tap) unit for the two rows (g, g + 8) a lane serves: [row][half: hi, lo'][CIN / 8 words];
// words 2s, 2s + 1 are (b0, b1) of k-step s
template <int CIN>
struct Frag {
  static constexpr int W = CIN / 8;  // 32-bit words per row half: 2 (8 B) or 4 (16 B)
  uint32_t w[2][2][W];
};

// predicated vector loads with zero fill (a missing neighbour issues no request)
__device__ __forceinline__ void ldg8_or_zero(uint32_t &x, uint32_t &y, const uint8_t *addr, int idx) {
  asm("{\n\t.reg .pred p;\n\t"
      "setp.ge.s32 p, %3, 0;\n\t"
      "mov.b32 %0, 0;\n\tmov.b32 %1, 0;\n\t"
      "@p ld.global.nc.v2.u32 {%0, %1}, [%2];\n\t}"
      : "=r"(x), "=r"(y)
      : "l"(addr), "r"(idx));
}
__device__ __forceinline__ void ldg16_or_zero(uint32_t &x, uint32_t &y, uint32_t &z, uint32_t &w, const uint8_t *addr, int idx) {
  asm("{\n\t.reg .pred p;\n\t"
      "setp.ge.s32 p, %5, 0;\n\t"
      "mov.b32 %0, 0;\n\tmov.b32 %1, 0;\n\tmov.b32 %2, 0;\n\tmov.b32 %3, 0;\n\t"
      "@p ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];\n\t}"
      : "=r"(x), "=r"(y), "=r"(z), "=r"(w)
      : "l"(addr), "r"(idx));
}

// in_t = rows + this lane's byte offset inside a row half; idx0 / idx1 = this lane's two index rows in shared memory
template <int CIN>
__device__ __forceinline__ void load_frag(Frag<CIN> &f, const uint8_t *in_t, const int32_t *idx0, const int32_t *idx1, int tap) {
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int idx = r ? idx1[tap] : idx0[tap];
    const uint8_t *src = in_t + static_cast<size_t>(static_cast<uint32_t>(idx)) * (4 * CIN);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (CIN == 16)
        ldg8_or_zero(f.w[r][h][0], f.w[r][h][1], src + h * 32, idx);
      else
        ldg16_or_zero(f.w[r][h][0], f.w[r][h][1], f.w[r][h][2], f.w[r][h][3], src + h * 64, idx);
    }
  }
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
// ticket of a split tile: acq_rel at gpu scope - with the __syncwarp() on either side it publishes the whole warp's
// partial sums and orders the finisher's reads behind the other pieces (PTX release / acquire patterns are cumulative),
// without the two full fences a __threadfence() pair costs
__device__ __forceinline__ int atom_add_acq_rel(int32_t *addr, int v) {
  int old;
  asm volatile("atom.acq_rel.gpu.global.add.s32 %0, [%1], %2;" : "=r"(old) : "l"(addr), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// A group = up to D consecutive taps of one tile: the unit of the register ring (slot d = d-th tap of the group), so the
// ring slots stay compile-time registers while the prefetch runs across tile boundaries.
struct Group {
  int tile;
  int tap0, count;
  bool valid, last;  // last group of this warp's tap range of the tile
};

template <int CIN, int COUT, int D>
__global__ void __launch_bounds__(kWarps * 32, 1) conv_wm_kernel(const Params p) {
  constexpr int KS = CIN / 16, MT = COUT / 16;
  constexpr int KCO = (COUT >= 32) ? 32 : 16;
  constexpr int SO = COUT + 4;          // row stride (floats) of the per-warp output tile: conflict-free both ways
  constexpr int NV = MT * 2 * 4;        // accumulator values per lane
  extern __shared__ __align__(16) uint8_t smem_raw[];
  uint4 *s_w = reinterpret_cast<uint4 *>(smem_raw);  // [K][KS][MT][2][32]
  const int K = p.K;
  const int w_vec = K * KS * MT * 2 * 32;
  int32_t *s_idx_all = reinterpret_cast<int32_t *>(smem_raw + static_cast<size_t>(w_vec) * 16);  // [kWarps][2][16 * K]
  float *s_out_all = reinterpret_cast<float *>(s_idx_all + kWarps * 2 * 16 * K);               // [kWarps][16][SO]
  pdl_trigger();
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  for (int i = tid; i < w_vec; i += kWarps * 32) s_w[i] = __ldg(p.packed_w + i);  // static parameters
  __shared__ __align__(16) float s_sc[COUT], s_sh[COUT];
  const int g = lane >> 2, t = lane & 3;
  if (tid < COUT) {
    s_sc[tid] = p.scale ? __ldg(p.scale + tid) : 1.0f;
    s_sh[tid] = p.shift ? __ldg(p.shift + tid) : 0.0f;
  }
  __syncthreads();
  pdl_wait();  // rows / neighbour map / residual belong to earlier kernels
  const long long n = p.n_out_dev ? min(static_cast<long long>(p.n_out_dev[0]), p.n_cap) : p.n_cap;
  const int n_tiles = static_cast<int>((n + 15) / 16);
  const int U = n_tiles * K;  // (tile, tap) units; the host guarantees < 2^31
  int W = static_cast<int>(gridDim.x) * kWarps;
  if (W > U / 8) W = U / 8 > 0 ? U / 8 : 1;  // ranges of >= 8 units
  const int w = wid * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);  // consecutive warp ids on different SMs
  if (w >= W || U == 0) return;
  const int u0 = static_cast<int>(static_cast<long long>(w) * U / W), u1 = static_cast<int>(static_cast<long long>(w + 1) * U / W);
  if (u0 >= u1) return;
  const int t_first = u0 / K, t_last = (u1 - 1) / K;
  int32_t *s_idx = s_idx_all + wid * (2 * 16 * K);
  float *s_out = s_out_all + wid * (16 * SO);
  const uint8_t *in_t;  // this lane's 8 B (Cin = 16) / 16 B (Cin = 32) inside a row half; opaque so that it stays in registers
  asm volatile("mov.u64 %0, %1;" : "=l"(in_t) : "l"(p.in + t * (CIN / 2)));

  auto stage = [&](int tile) {  // neighbour indices of `tile` -> buffer tile & 1 (asynchronous, 16 bytes per request)
    int32_t *dst = s_idx + (tile & 1) * (16 * K);
    const long long row0 = static_cast<long long>(tile) * 16;
    const int have = static_cast<int>(min(16ll, n - row0)) * K;  // valid words; the region starts 64-byte aligned
    const int32_t *src = p.nbr + row0 * K;
    const uint32_t dsts = static_cast<uint32_t>(__cvta_generic_to_shared(dst));
    for (int i = lane * 4; i < 16 * K; i += 128) {
      if (i + 4 <= have) {
        cp_async16(dsts + i * 4, src + i);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) dst[i + e] = (i + e < have) ? __ldg(src + i + e) : -1;  // rows beyond n read as "missing"
      }
    }
  };
  auto group_at = [&](int tile, int tap) {  // the group starting at (tile, tap) inside [u0, u1)
    Group gq;
    gq.tile = tile;
    gq.tap0 = tap;
    const int tb = min(u1 - tile * K, K);
    gq.valid = tile <= t_last;
    gq.count = gq.valid ? min(D, tb - tap) : 0;
    gq.last = tap + gq.count >= tb;
    return gq;
  };
  auto next_group = [&](const Group &c) {
    if (!c.last) return group_at(c.tile, c.tap0 + c.count);
    return group_at(c.tile + 1, 0);  // a later tile of the range starts at tap 0
  };

  stage(t_first);
  if (t_last > t_first) stage(t_first + 1);
  cp_async_wait_all();
  __syncwarp();
  int ready_tile = min(t_last, t_first + 1);  // highest tile whose indices are in shared memory

  // [m tile: 16 output channels][n tile: rows 0-7 / 8-15][c0..c3]; the two cross products have their own accumulators so
  // that the three MMAs of a k-step are independent
  // (only for Cout = 16: with two m tiles there are already four independent chains per accumulator kind)
  constexpr int XS = (MT == 1) ? 1 : 0;  // ax is a separate register set / an alias of al
  float am[MT][2][4], al[MT][2][4], ax_[MT][2][4];
  auto &ax = XS ? ax_ : al;
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
      for (int j = 0; j < 4; ++j) am[m][q][j] = al[m][q][j] = ax_[m][q][j] = 0.f;
  bool ovf = false;

  Group cur = group_at(t_first, u0 - t_first * K);
  Group nxt = next_group(cur);
  Frag<CIN> buf[D];
  {
    const int32_t *i0 = s_idx + (cur.tile & 1) * (16 * K) + g * K + cur.tap0;
#pragma unroll
    for (int d = 0; d < D; ++d)
      if (d < cur.count) load_frag<CIN>(buf[d], in_t, i0, i0 + 8 * K, d);
  }
  while (cur.valid) {
    if (nxt.valid && nxt.tile > ready_tile) {  // the indices of the next tile were staged one tile ago: complete them
      cp_async_wait_all();
      __syncwarp();
      ready_tile = nxt.tile;
    }
    const uint4 *wt = s_w + static_cast<size_t>(cur.tap0) * (KS * MT * 2 * 32) + lane;
    const int32_t *n0 = s_idx + (nxt.tile & 1) * (16 * K) + g * K + nxt.tap0;
#pragma unroll
    for (int d = 0; d < D; ++d) {
      if (d < cur.count) {
#pragma unroll
        for (int s = 0; s < KS; ++s) {
#pragma unroll
          for (int m = 0; m < MT; ++m) {
            const uint4 a_hi = wt[((d * KS + s) * MT + m) * 64];
            const uint4 a_lo = wt[((d * KS + s) * MT + m) * 64 + 32];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              mma16816(am[m][q], a_hi, buf[d].w[q][0][2 * s], buf[d].w[q][0][2 * s + 1]);
              mma16816(al[m][q], a_hi, buf[d].w[q][1][2 * s], buf[d].w[q][1][2 * s + 1]);
              mma16816(ax[m][q], a_lo, buf[d].w[q][0][2 * s], buf[d].w[q][0][2 * s + 1]);
            }
          }
        }
      }
      if (d < nxt.count) load_frag<CIN>(buf[d], in_t, n0, n0 + 8 * K, d);
    }
    if (cur.last) {
      // ---------------------------------------------------------------- tile finished (for this warp)
      const int tile = cur.tile;
      const long long row0 = static_cast<long long>(tile) * 16;
      const int rows = static_cast<int>(min(16ll, n - row0));
      const int start = tile * K;
      const bool split = start < u0 || start + K > u1;  // other warps hold taps of this tile
      float v[NV];
#pragma unroll
      for (int m = 0; m < MT; ++m)
#pragma unroll
        for (int q = 0; q < 2; ++q)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            v[(m * 2 + q) * 4 + j] = fmaf(XS ? al[m][q][j] + ax_[m][q][j] : al[m][q][j], kLoInv, am[m][q][j]);
            am[m][q][j] = al[m][q][j] = ax_[m][q][j] = 0.f;
          }
      bool finish = true;
      if (split) {
        // contributors of this tile: warps cf .. cl (ranges are monotone in the warp id)
        const int cf = static_cast<int>((static_cast<long long>(start + 1) * W - 1) / U);
        const int cl = static_cast<int>((static_cast<long long>(start + K) * W - 1) / U);
        // partial sums: slab[warp][0] = piece of a tile begun by an earlier warp, [1] = piece of a tile that continues
        float *mine = p.slabs + (static_cast<size_t>(w) * 2 + (u0 > start ? 0 : 1)) * (NV * 32);
#pragma unroll
        for (int j = 0; j < NV; ++j) __stcg(mine + j * 32 + lane, v[j]);
        __syncwarp();
        int last = 0;
        if (lane == 0) {
          const int old = atom_add_acq_rel(p.tickets + tile, 1);
          last = (old == cl - cf) ? 1 : 0;
          if (last) p.tickets[tile] = 0;  // all pieces have arrived: leave the ticket clean for the next launch
        }
        finish = __shfl_sync(0xffffffffu, last, 0) != 0;
        __syncwarp();  // the other lanes' slab reads are ordered behind lane 0's acquire
        if (finish) {
#pragma unroll
          for (int j = 0; j < NV; ++j) v[j] = 0.f;
          for (int x = cf; x <= cl; ++x) {  // pieces in warp order: deterministic
            const float *sl = p.slabs + (static_cast<size_t>(x) * 2 + (x == cf ? 1 : 0)) * (NV * 32);
#pragma unroll
            for (int j = 0; j < NV; ++j) v[j] += __ldcg(sl + j * 32 + lane);
          }
        }
      }
      if (finish) {
        // transpose back: the lane holds channels 16m + g (+ 8) of rows 8q + 2t (+ 1)
        __syncwarp();
#pragma unroll
        for (int m = 0; m < MT; ++m)
#pragma unroll
          for (int q = 0; q < 2; ++q)
#pragma unroll
            for (int j = 0; j < 4; ++j)
              s_out[(q * 8 + 2 * t + (j & 1)) * SO + m * 16 + g + 8 * (j >> 1)] = v[(m * 2 + q) * 4 + j];
        __syncwarp();
        // epilogue: lane = (row lane / 2, channel half lane & 1): COUT / 2 contiguous channels, 16-byte accesses
        constexpr int CH = COUT / 2;
        const int lr = lane >> 1, c0 = (lane & 1) * CH;
        if (lr < rows) {
          const size_t orow = static_cast<size_t>(row0 + lr);
          float o[CH];
#pragma unroll
          for (int j = 0; j < CH; j += 4) {
            const float4 x = *reinterpret_cast<const float4 *>(s_out + lr * SO + c0 + j);
            const float4 sc = *reinterpret_cast<const float4 *>(s_sc + c0 + j), sh = *reinterpret_cast<const float4 *>(s_sh + c0 + j);
            o[j] = fmaf(x.x, sc.x, sh.x);
            o[j + 1] = fmaf(x.y, sc.y, sh.y);
            o[j + 2] = fmaf(x.z, sc.z, sh.z);
            o[j + 3] = fmaf(x.w, sc.w, sh.w);
          }
          const size_t hoff = orow * (4 * COUT) + (c0 / KCO) * (4 * KCO) + (c0 % KCO) * 2;  // hi halfs; lo' at + 2 KCO
          if (p.residual) {
#pragma unroll
            for (int j = 0; j < CH; j += 8) {
              const uint4 rh = __ldg(reinterpret_cast<const uint4 *>(p.residual + hoff + j * 2));
              const uint4 rl = __ldg(reinterpret_cast<const uint4 *>(p.residual + hoff + 2 * KCO + j * 2));
              const uint32_t hw[4] = {rh.x, rh.y, rh.z, rh.w}, lw[4] = {rl.x, rl.y, rl.z, rl.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const __half2 hh = *reinterpret_cast<const __half2 *>(&hw[e]), ll = *reinterpret_cast<const __half2 *>(&lw[e]);
                o[j + 2 * e] += merge_h16(__low2half(hh), __low2half(ll));
                o[j + 2 * e + 1] += merge_h16(__high2half(hh), __high2half(ll));
              }
            }
          }
          if (p.relu) {
#pragma unroll
            for (int j = 0; j < CH; ++j) o[j] = fmaxf(o[j], 0.f);
          }
          if (p.out_f32) {
#pragma unroll
            for (int j = 0; j < CH; j += 4)
              *reinterpret_cast<float4 *>(p.out_f32 + orow * COUT + c0 + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
          }
          if (p.out_h16) {
#pragma unroll
            for (int j = 0; j < CH; j += 8) {
              uint32_t hw[4], lw[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                __half h0, l0, h1, l1;
                split_h16(o[j + 2 * e], h0, l0, ovf);
                split_h16(o[j + 2 * e + 1], h1, l1, ovf);
                const __half2 hh = __halves2half2(h0, h1), ll = __halves2half2(l0, l1);
                hw[e] = *reinterpret_cast<const uint32_t *>(&hh);
                lw[e] = *reinterpret_cast<const uint32_t *>(&ll);
              }
              *reinterpret_cast<uint4 *>(p.out_h16 + hoff + j * 2) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
              *reinterpret_cast<uint4 *>(p.out_h16 + hoff + 2 * KCO + j * 2) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
            }
          }
        }
      }
      // the finished tile's index buffer is free (the prefetch is already in the next tile): refill it with the tile
      // after next
      if (tile + 2 <= t_last) {
        __syncwarp();
        stage(tile + 2);
      }
    }
    cur = nxt;
    nxt = next_group(nxt);
  }
  if (ovf && p.status) atomicOr(p.status, 1);
}

// fp32 [K][Cin][Cout] -> A-fragment-order image [K][Cin / 16][Cout / 16][2: hi, lo'][32 lanes][a0, a1, a2, a3]:
// lane (g = lane / 4, t = lane % 4) of k-step s, m-tile m holds output channels 16 m + g (a0, a2) and 16 m + g + 8
// (a1, a3) and the input channels (Cin / 4) t + 4 s + {0, 1} (a0, a1) and + {2, 3} (a2, a3) - the k permutation of the
// header comment
__global__ void __launch_bounds__(256) pack_weights_wm_kernel(const float *__restrict__ w, int K, int Cin, int Cout,
                                                              uint32_t *__restrict__ packed, int32_t *status) {
  const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int KS = Cin / 16, MT = Cout / 16;
  const long long total = static_cast<long long>(K) * KS * MT * 32;
  if (q >= total) return;
  const int lane = static_cast<int>(q % 32);
  const int m = static_cast<int>((q / 32) % MT);
  const int s = static_cast<int>((q / (32 * MT)) % KS);
  const int tap = static_cast<int>(q / (32ll * MT * KS));
  const int g = lane >> 2, t = lane & 3;
  const int ch0 = (Cin / 4) * t + 4 * s;
  uint32_t hi_w[4], lo_w[4];
  bool ovf = false;
  for (int a = 0; a < 4; ++a) {  // a0: (co g, ch 0,1)  a1: (co g + 8, ch 0,1)  a2: (co g, ch 2,3)  a3: (co g + 8, ch 2,3)
    const int co = m * 16 + g + 8 * (a & 1), ch = ch0 + 2 * (a >> 1);
    __half h0, l0, h1, l1;
    split_h16(w[(static_cast<size_t>(tap) * Cin + ch) * Cout + co], h0, l0, ovf);
    split_h16(w[(static_cast<size_t>(tap) * Cin + ch + 1) * Cout + co], h1, l1, ovf);
    const __half2 hh = __halves2half2(h0, h1), ll = __halves2half2(l0, l1);
    hi_w[a] = *reinterpret_cast<const uint32_t *>(&hh);
    lo_w[a] = *reinterpret_cast<const uint32_t *>(&ll);
  }
  const size_t blk = (static_cast<size_t>(tap) * KS + s) * MT + m;  // [2][32] uint4
  uint32_t *ph = packed + ((blk * 2 + 0) * 32 + lane) * 4, *pl = packed + ((blk * 2 + 1) * 32 + lane) * 4;
  for (int a = 0; a < 4; ++a) {
    ph[a] = hi_w[a];
    pl[a] = lo_w[a];
  }
  if (ovf && status) atomicOr(status, 1);
}

template <int CIN, int COUT, int D>
int launch(const Params &p, cudaStream_t st) {
  constexpr int KS = CIN / 16, MT = COUT / 16;
  const size_t smem = static_cast<size_t>(p.K) * KS * MT * 1024 + static_cast<size_t>(kWarps) * 2 * 16 * p.K * sizeof(int32_t) +
                      static_cast<size_t>(kWarps) * 16 * (COUT + 4) * sizeof(float);
  if (smem > 227 * 1024) return P3D_ERR_UNSUPPORTED;
  auto kern = conv_wm_kernel<CIN, COUT, D>;
  P3D_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const long long blocks_needed = (p.n_cap + 16 * kWarps - 1) / (16 * kWarps);
  long long grid = kNumSMs;
  if (grid > blocks_needed) grid = blocks_needed;
  if (grid < 1) grid = 1;
  P3D_CUDA_CHECK(launch_pdl(kern, dim3(static_cast<unsigned int>(grid)), dim3(kWarps * 32), smem, st, p));
  return P3D_OK;
}

inline bool supported(int K, int Cin, int Cout) {
  if (K < 1 || K > 32) return false;
  return (Cin == 16 && (Cout == 16 || Cout == 32)) || (Cin == 32 && Cout == 32);
}

}  // namespace wm
}  // namespace p3d

using namespace p3d;

extern "C" size_t p3d_sparse_conv_wm_packed_weight_bytes(int K, int Cin, int Cout) {
  if (!wm::supported(K, Cin, Cout)) return 0;
  return align_up(static_cast<size_t>(K) * (Cin / 16) * (Cout / 16) * 1024);
}

extern "C" int p3d_sparse_conv_wm_pack_weights(const float *weight, int K, int Cin, int Cout, void *packed,
                                               int32_t *status_dev, p3d_stream_t stream) {
  if (!weight || !packed) return P3D_ERR_INVALID_ARG;
  if (!wm::supported(K, Cin, Cout)) return P3D_ERR_UNSUPPORTED;
  const long long total = static_cast<long long>(K) * (Cin / 16) * (Cout / 16) * 32;
  wm::pack_weights_wm_kernel<<<div_up(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      weight, K, Cin, Cout, static_cast<uint32_t *>(packed), status_dev);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

// workspace = [tickets: one int32 per 16-row tile, ZERO on first use (left zero)][slabs of the stream-K partial tiles]
extern "C" size_t p3d_sparse_conv_wm_workspace_bytes(int64_t n_out_cap, int Cout) {
  if (n_out_cap <= 0 || Cout < 16) return 0;
  const size_t tiles = static_cast<size_t>((n_out_cap + 15) / 16);
  return align_up(tiles * sizeof(int32_t)) +
         align_up(static_cast<size_t>(kNumSMs) * wm::kWarps * 2 * (Cout / 2) * 32 * sizeof(float));
}

extern "C" int p3d_sparse_conv_wm(const void *in_h16, const int32_t *nbr, const int32_t *n_out_dev, int64_t n_out_cap,
                                  int K, int Cin, int Cout, const void *packed_weight, const float *scale,
                                  const float *shift, const void *residual_h16, int relu, float *out_f32, void *out_h16,
                                  void *workspace, size_t workspace_bytes, int32_t *status_dev, p3d_stream_t stream) {
  if (n_out_cap < 0 || !packed_weight || (!out_f32 && !out_h16) || (n_out_cap && (!in_h16 || !nbr)))
    return P3D_ERR_INVALID_ARG;
  if (!wm::supported(K, Cin, Cout) || n_out_cap > kMaxRows) return P3D_ERR_UNSUPPORTED;  // (tile, tap) units fit 31 bits
  if (n_out_cap == 0) return P3D_OK;
  if ((reinterpret_cast<uintptr_t>(in_h16) & 15) || (reinterpret_cast<uintptr_t>(out_f32) & 15) ||
      (reinterpret_cast<uintptr_t>(out_h16) & 15) || (reinterpret_cast<uintptr_t>(packed_weight) & 15) ||
      (reinterpret_cast<uintptr_t>(residual_h16) & 15) || (reinterpret_cast<uintptr_t>(nbr) & 15) ||  // 16-byte cp.async
      (reinterpret_cast<uintptr_t>(workspace) & 15))
    return P3D_ERR_INVALID_ARG;
  if (!workspace || workspace_bytes < p3d_sparse_conv_wm_workspace_bytes(n_out_cap, Cout)) return P3D_ERR_WORKSPACE;
  wm::Params p;
  p.in = static_cast<const uint8_t *>(in_h16);
  p.nbr = nbr;
  p.n_out_dev = n_out_dev;
  p.n_cap = n_out_cap;
  p.K = K;
  p.packed_w = static_cast<const uint4 *>(packed_weight);
  p.scale = scale;
  p.shift = shift;
  p.residual = static_cast<const uint8_t *>(residual_h16);
  p.relu = relu;
  p.out_f32 = out_f32;
  p.out_h16 = static_cast<uint8_t *>(out_h16);
  p.status = status_dev;
  p.tickets = static_cast<int32_t *>(workspace);
  p.slabs = reinterpret_cast<float *>(static_cast<char *>(workspace) + align_up(static_cast<size_t>((n_out_cap + 15) / 16) * sizeof(int32_t)));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  static const int d_env = getenv("P3D_WM_D") ? atoi(getenv("P3D_WM_D")) : 0;  // tuning hook: ring depth
  if (Cin == 16 && Cout == 16) {  // measured per level-0 layer: D = 3 25.5 us, D = 5 25.0 us, D = 9 27.0 us
    if (d_env == 3) return wm::launch<16, 16, 3>(p, st);
    if (d_env == 9) return wm::launch<16, 16, 9>(p, st);
    return wm::launch<16, 16, 5>(p, st);
  }
  if (Cin == 16 && Cout == 32) {
    if (d_env == 3) return wm::launch<16, 32, 3>(p, st);
    if (d_env == 9) return wm::launch<16, 32, 7>(p, st);
    return wm::launch<16, 32, 5>(p, st);
  }
  if (Cin == 32 && Cout == 32) {  // measured: D = 3 33.4 us, D = 4 (8 bytes of spills) 35.4 us per level-1 layer
    if (d_env == 4) return wm::launch<32, 32, 4>(p, st);
    return wm::launch<32, 32, 3>(p, st);
  }
  return P3D_ERR_UNSUPPORTED;
}
