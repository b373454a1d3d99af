// Implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM), operands
// staged by TMA straight from the channels-last activation tensor: no im2col buffer ever exists.
//
// GEMM view: M = output positions, N = Cout, K = taps x Cin.  One CTA owns an output patch of
// TH x TW positions of one output frame (TH = NACC * 128/TW) and N_cta output channels; it keeps NACC
// accumulators of 128 x N_cta fp32 in TMEM (<= 512 columns) so that every weight tile staged in shared
// memory feeds NACC MMAs, and every activation slab feeds all KH row-taps:
//
//   A slab  (one per kt, kw, 64-channel block): the (TH+KH-1) x TW input window, shifted by kw, loaded by
//           ONE 5-D TMA box into a SWIZZLE_128B buffer [row][w][64 ch].  Because the slab pitch is exactly
//           TW positions (a multiple of 8 -> 1024 B), the A operand of row-tap kh / sub-tile s is the same
//           buffer at byte offset ((s*ROWS + kh) * TW) * 128: a 1024-B aligned UMMA descriptor, no copy.
//           Zero padding in H/W is TMA out-of-bounds fill; time padding is a coordinate clamp (replicate)
//           or a skipped tap (zeros).  Strided (down-sampling) convs use TMA element strides.
//   B tile  (one per tap, 64-channel block): [N_cta][64] slice of the packed weights [tap][Cout][Cin].
//
// Warp roles (256 threads): w0 A-producer, w1 B-producer, w2 MMA issuer (one elected thread), w3 TMEM
// allocator, w4-7 epilogue (TMEM -> registers -> bias/alpha/residual -> 16-bit stores, with the
// time-interleave scatter of Upsample3D folded into the store address).
//
// Replaces cuDNN behind CausalConv3d / nn.Conv3d / Conv2dWithExtraDim / Downsample3D / Upsample3D
// (reference: models/vae_models.py:198-340, models/vae_blocks3d_sd3.py:16-364); see include/cvvae_b200.h.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "ptx.cuh"

namespace cvvae {

struct ConvTcParams {
  int B, T_in, T_out, H_out, W_out, Cin, Cout;
  int KT, KH, KW, st, sh, sw, off_t, off_h, off_w, pad_t;
  int up_time, flags;
  float alpha;
  // tiling
  int TW, ROWS, NACC, TH, N_cta, KHs, n_hgroups, slab_rows;
  int tiles_w, tiles_h, n_tiles_n, cblocks, flat;
  int tiles_hg, tiles_wg;  // grid extents in tiles: a CTA pair (cta_group::2) owns two tiles adjacent in H (default) or, with
  int pair_w;              // wide slabs, in W (pair_w = 1); tiles_hg / tiles_wg = ceil(tiles / 2) along the paired axis
  int NA, NB;
  uint32_t slab_bytes, b_bytes, idesc;
  // epilogue
  const float* bias;
  const void* residual;
  void* y;
  long long ys_b, ys_t, ys_h, ys_w, ys_c;
  int yC, yT, vec_ok, bias_vec;
  int64_t* gn_stats;  // fused GroupNorm statistics of y (TMA epilogue only)
  int gn_groups, gn_cpg;
  int persist;  // persistent swap kernel: 256-position tiles, two TMEM stages, epilogue overlapped with the next tile
  int n_tiles;  // tiles of the whole launch (persistent kernel)
  // persistent kernel, stride-1 layers: ONE slab per (kt, channel block) serves all KH x KW taps.  Tiles are 8 positions
  // wide (one 8-row swizzle group per image row), the slab keeps PW >= 8 + KW - 1 positions per row, and the UMMA
  // descriptor walks the image rows with SBO = PW * 128 B from a start address shifted by (kh * PW + kw) * 128 B.
  int wide, PW;
  uint32_t slab_stride;  // bytes between slab ring slots (slab_bytes rounded up to 1024)
  int tma_epi, box_w;  // epilogue through swizzled smem + TMA store (box_w = min(TW, 32) positions per box row)
  // fused 1x1 shortcut (ResnetBlock3D nin_shortcut / conv_shortcut as extra K steps of conv2): cblocks2 64-channel blocks
  // of a second input tensor (same positions as the output) times a [Cout][Cin2] matrix, accumulated after the taps
  int Cin2, cblocks2;
  uint32_t sc_off16;  // wide slabs: descriptor offset (>> 4) of the centre tap inside the slab
  unsigned long long* trace;  // optional [trace_n][8] globaltimer stamps per CTA (diagnostics)
  int trace_n;
};

static constexpr int kThreads = 256;
static constexpr uint32_t kTmemCols = 512;

__device__ __forceinline__ void wait_bar(uint64_t* bar, uint32_t parity) { ptx::mbar_wait(bar, parity); }

struct TileCoord {
  int b, t, h0, w0, n0;
};

template <int CG>
__device__ __forceinline__ TileCoord decode_tile(const ConvTcParams& p, int rank, int tile_id = -1) {
  int id = tile_id >= 0 ? tile_id : static_cast<int>(blockIdx.x) / CG;
  TileCoord c;
  c.n0 = (id % p.n_tiles_n) * p.N_cta;
  id /= p.n_tiles_n;
  c.t = id % p.T_out;
  id /= p.T_out;
  const int cgw = p.pair_w ? CG : 1, cgh = p.pair_w ? 1 : CG;   // the two CTAs of a pair own tiles adjacent in W or in H
  c.w0 = ((id % p.tiles_wg) * cgw + (p.pair_w ? rank : 0)) * (p.flat ? p.NACC * 128 : p.TW);
  id /= p.tiles_wg;
  c.h0 = ((id % p.tiles_hg) * cgh + (p.pair_w ? 0 : rank)) * p.TH;
  c.b = id / p.tiles_hg;
  return c;
}

// Enumerate the activation-slab steps of one tile in the order every role agrees on.
// f(kt, ti, hg, kw, cb)
template <class F>
__device__ __forceinline__ void for_each_slab(const ConvTcParams& p, int t, F&& f) {
  for (int kt = 0; kt < p.KT; ++kt) {
    int ti = t * p.st + kt + p.off_t;
    if (ti < 0 || ti >= p.T_in) {
      if (p.pad_t == CVVAE_PAD_ZERO) continue;
      ti = ti < 0 ? 0 : p.T_in - 1;
    }
    for (int hg = 0; hg < p.n_hgroups; ++hg)
      for (int kw = 0; kw < p.KW; ++kw)
        for (int cb = 0; cb < p.cblocks; ++cb) f(kt, ti, hg, kw, cb);
  }
}

// Wide-slab variant: one step per (kt, channel block).  f(kt, ti, cb)
template <class F>
__device__ __forceinline__ void for_each_wslab(const ConvTcParams& p, int t, F&& f) {
  for (int kt = 0; kt < p.KT; ++kt) {
    int ti = t * p.st + kt + p.off_t;
    if (ti < 0 || ti >= p.T_in) {
      if (p.pad_t == CVVAE_PAD_ZERO) continue;
      ti = ti < 0 ? 0 : p.T_in - 1;
    }
    for (int cb = 0; cb < p.cblocks; ++cb) f(kt, ti, cb);
  }
}

// CG = 1: one CTA per tile.  CG = 2: a CTA pair (cluster of 2, cta_group::2) shares every weight tile - each
// CTA stages half of its rows, the 256 x N MMA reads both halves - which halves the weight traffic from L2 and
// the tensor core's shared-memory operand reads per FLOP (the N = 128 layers are bound by the latter).
template <int DT, int CG>
__global__ void __launch_bounds__(kThreads, 1)
    conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmR,
                   const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
                   const ConvTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = sA + static_cast<size_t>(p.NA) * p.slab_stride;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + static_cast<size_t>(p.NB) * p.b_bytes);
  uint64_t* fullA = bars;         // [8]
  uint64_t* emptyA = bars + 8;    // [8]
  uint64_t* fullB = bars + 16;    // [8]
  uint64_t* emptyB = bars + 24;   // [8]
  uint64_t* accFull = bars + 32;  // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 33);
  uint64_t* resBar = bars + 40;   // [8] one per warp: residual tile landed (TMA epilogue)
  unsigned long long* gn_bins = reinterpret_cast<unsigned long long*>(bars + 64);  // [64 groups][2] fixed-point partial sums

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool traced = p.trace != nullptr && static_cast<int>(blockIdx.x) < p.trace_n;
  unsigned long long* trc = traced ? p.trace + static_cast<size_t>(blockIdx.x) * 8 : nullptr;
  if (traced && threadIdx.x == 0) trc[0] = ptx::globaltimer_ns();
  const int rank = CG == 2 ? static_cast<int>(ptx::cluster_ctarank()) : 0;
  const TileCoord tc = decode_tile<CG>(p, rank);
  // sub-tiles that contain at least one valid output position (0 for the idle half of an odd last pair)
  int nacc_eff;
  if (p.flat) {
    int rem = p.W_out - tc.w0;
    nacc_eff = min(p.NACC, (rem + 127) / 128);
  } else {
    int rem = p.H_out - tc.h0;
    nacc_eff = max(0, min(p.NACC, (rem + p.ROWS - 1) / p.ROWS));
    if (tc.w0 >= p.W_out) nacc_eff = 0;   // idle half of an odd last pair along W
  }

  if (threadIdx.x < 128) gn_bins[threadIdx.x] = 0ull;
  if (threadIdx.x == 0) {
    for (int i = 0; i < p.NA; ++i) {
      ptx::mbar_init(&fullA[i], 1);
      ptx::mbar_init(&emptyA[i], 1);
    }
    for (int i = 0; i < p.NB; ++i) {
      ptx::mbar_init(&fullB[i], 1);
      ptx::mbar_init(&emptyB[i], 1);
    }
    ptx::mbar_init(accFull, 1);
    for (int i = 0; i < 8; ++i) ptx::mbar_init(&resBar[i], 1);
    ptx::fence_mbar_init();
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
  }
  if (warp == 3) {
    if (CG == 2) {
      ptx::tmem_alloc_cg2(tmem_slot, kTmemCols);
      ptx::tmem_relinquish_cg2();
    } else {
      ptx::tmem_alloc(tmem_slot, kTmemCols);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  __syncthreads();                    // tmem_slot / barrier init visible CTA-wide
  if (CG == 2) ptx::cluster_sync();   // the peer's barriers / TMEM exist before anyone signals them
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (traced && threadIdx.x == 0) trc[1] = ptx::globaltimer_ns();

  if (warp == 0) {
    // ------------------------------------------------------------- A producer
    // The whole warp walks the step sequence (so every operand the TMA instruction takes is provably
    // warp-uniform and lives in uniform registers); one elected lane issues.
    {
      int slot = 0;
      uint32_t phase = 0;
      const int xb = (p.flags & CVVAE_CONV_X_SHARED) ? 0 : tc.b;  // batched GEMM with one shared left operand
      auto load_slab = [&](const CUtensorMap* tm, int c0, int cw, int chh, int ti) {
        wait_bar(&emptyA[slot], phase ^ 1);
        uint8_t* dst = sA + static_cast<size_t>(slot) * p.slab_stride;
        if (ptx::elect_one()) {
          if (CG == 2) {
            if (rank == 0) ptx::mbar_expect_tx(&fullA[slot], 2u * p.slab_bytes);   // both CTAs' bytes land on the leader's barrier
            ptx::tma_load_5d_cg2(dst, tm, ptx::mapa_u32(ptx::smem_u32(&fullA[slot]), 0), c0, cw, chh, ti, xb);
          } else {
            ptx::mbar_expect_tx(&fullA[slot], p.slab_bytes);
            ptx::tma_load_5d(dst, tm, &fullA[slot], c0, cw, chh, ti, xb);
          }
        }
        __syncwarp();
        if (++slot == p.NA) {
          slot = 0;
          phase ^= 1;
        }
      };
      if (p.wide) {
        // one slab per (kt, channel block) for all KH x KW taps (8-wide tiles, see conv_tc_psw_kernel)
        for_each_wslab(p, tc.t, [&](int kt, int ti, int cb) { load_slab(&tmA, cb * 64, tc.w0 + p.off_w, tc.h0 + p.off_h, ti); });
        for (int cb2 = 0; cb2 < p.cblocks2; ++cb2) load_slab(&tmA2, cb2 * 64, tc.w0 + p.off_w, tc.h0 + p.off_h, tc.t);
      } else {
      for_each_slab(p, tc.t, [&](int kt, int ti, int hg, int kw, int cb) {
        wait_bar(&emptyA[slot], phase ^ 1);
        uint8_t* dst = sA + static_cast<size_t>(slot) * p.slab_stride;
        if (ptx::elect_one()) {
          if (p.flat) {
            ptx::mbar_expect_tx(&fullA[slot], static_cast<uint32_t>(nacc_eff) * 128u * 128u);
            for (int s = 0; s < nacc_eff; ++s)
              ptx::tma_load_5d(dst + s * 16384, &tmA, &fullA[slot], cb * 64, tc.w0 + s * 128, 0, ti, xb);
          } else if (CG == 2) {
            // both CTAs' bytes complete on the leader's barrier
            if (rank == 0) ptx::mbar_expect_tx(&fullA[slot], 2u * p.slab_bytes);
            ptx::tma_load_5d_cg2(dst, &tmA, ptx::mapa_u32(ptx::smem_u32(&fullA[slot]), 0), cb * 64,
                                 tc.w0 * p.sw + kw + p.off_w, tc.h0 * p.sh + hg * p.KHs + p.off_h, ti, xb);
          } else {
            ptx::mbar_expect_tx(&fullA[slot], p.slab_bytes);
            ptx::tma_load_5d(dst, &tmA, &fullA[slot], cb * 64, tc.w0 * p.sw + kw + p.off_w,
                             tc.h0 * p.sh + hg * p.KHs + p.off_h, ti, xb);
          }
        }
        __syncwarp();
        if (++slot == p.NA) {
          slot = 0;
          phase ^= 1;
        }
      });
      // fused 1x1 shortcut: the (unshifted) window of the second input, one slab per 64-channel block
      for (int cb2 = 0; cb2 < p.cblocks2; ++cb2) {
        wait_bar(&emptyA[slot], phase ^ 1);
        uint8_t* dst = sA + static_cast<size_t>(slot) * p.slab_stride;
        if (ptx::elect_one()) {
          if (CG == 2) {
            if (rank == 0) ptx::mbar_expect_tx(&fullA[slot], 2u * p.slab_bytes);
            ptx::tma_load_5d_cg2(dst, &tmA2, ptx::mapa_u32(ptx::smem_u32(&fullA[slot]), 0), cb2 * 64, tc.w0, tc.h0, tc.t, xb);
          } else {
            ptx::mbar_expect_tx(&fullA[slot], p.slab_bytes);
            ptx::tma_load_5d(dst, &tmA2, &fullA[slot], cb2 * 64, tc.w0, tc.h0, tc.t, xb);
          }
        }
        __syncwarp();
        if (++slot == p.NA) {
          slot = 0;
          phase ^= 1;
        }
      }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------- B producer
    {
      int slot = 0;
      uint32_t phase = 0;
      if (p.wide) {
        auto load_w = [&](const CUtensorMap* tm, int c0, int tap) {
          wait_bar(&emptyB[slot], phase ^ 1);
          if (ptx::elect_one()) {
            if (CG == 2) {
              if (rank == 0) ptx::mbar_expect_tx(&fullB[slot], 2u * p.b_bytes);
              ptx::tma_load_3d_cg2(sB + static_cast<size_t>(slot) * p.b_bytes, tm, ptx::mapa_u32(ptx::smem_u32(&fullB[slot]), 0), c0,
                                   tc.n0 + rank * (p.N_cta / 2), tap);
            } else {
              ptx::mbar_expect_tx(&fullB[slot], p.b_bytes);
              ptx::tma_load_3d(sB + static_cast<size_t>(slot) * p.b_bytes, tm, &fullB[slot], c0, tc.n0, tap);
            }
          }
          __syncwarp();
          if (++slot == p.NB) {
            slot = 0;
            phase ^= 1;
          }
        };
        for_each_wslab(p, tc.t, [&](int kt, int ti, int cb) {
          for (int kh = 0; kh < p.KH; ++kh)
            for (int kw = 0; kw < p.KW; ++kw) load_w(&tmB, cb * 64, (kt * p.KH + kh) * p.KW + kw);
        });
        for (int cb2 = 0; cb2 < p.cblocks2; ++cb2) load_w(&tmB2, cb2 * 64, 0);
      } else {
      for_each_slab(p, tc.t, [&](int kt, int ti, int hg, int kw, int cb) {
        for (int khs = 0; khs < p.KHs; ++khs) {
          // batched GEMM: the "tap" axis of the weight tensor indexes the batch item (1x1x1 problems only)
          const int tap = (p.flags & CVVAE_CONV_W_PER_BATCH) ? tc.b : (kt * p.KH + hg * p.KHs + khs) * p.KW + kw;
          wait_bar(&emptyB[slot], phase ^ 1);
          if (ptx::elect_one()) {
            if (CG == 2) {
              // each CTA stages its half of the N_cta weight rows
              if (rank == 0) ptx::mbar_expect_tx(&fullB[slot], 2u * p.b_bytes);
              ptx::tma_load_3d_cg2(sB + static_cast<size_t>(slot) * p.b_bytes, &tmB, ptx::mapa_u32(ptx::smem_u32(&fullB[slot]), 0),
                                   cb * 64, tc.n0 + rank * (p.N_cta / 2), tap);
            } else {
              ptx::mbar_expect_tx(&fullB[slot], p.b_bytes);
              ptx::tma_load_3d(sB + static_cast<size_t>(slot) * p.b_bytes, &tmB, &fullB[slot], cb * 64, tc.n0, tap);
            }
          }
          __syncwarp();
          if (++slot == p.NB) {
            slot = 0;
            phase ^= 1;
          }
        }
      });
      for (int cb2 = 0; cb2 < p.cblocks2; ++cb2) {   // shortcut weights [Cout][Cin2]
        wait_bar(&emptyB[slot], phase ^ 1);
        if (ptx::elect_one()) {
          if (CG == 2) {
            if (rank == 0) ptx::mbar_expect_tx(&fullB[slot], 2u * p.b_bytes);
            ptx::tma_load_3d_cg2(sB + static_cast<size_t>(slot) * p.b_bytes, &tmB2, ptx::mapa_u32(ptx::smem_u32(&fullB[slot]), 0),
                                 cb2 * 64, tc.n0 + rank * (p.N_cta / 2), 0);
          } else {
            ptx::mbar_expect_tx(&fullB[slot], p.b_bytes);
            ptx::tma_load_3d(sB + static_cast<size_t>(slot) * p.b_bytes, &tmB2, &fullB[slot], cb2 * 64, tc.n0, 0);
          }
        }
        __syncwarp();
        if (++slot == p.NB) {
          slot = 0;
          phase ^= 1;
        }
      }
      }
    }
  } else if (warp == 2 && rank == 0) {
    // ------------------------------------------------------------- MMA issuer (the pair's leader when CG = 2)
    // Issue rate matters: one UTCHMMA covers only 64 (N=128) / 128 (N=256) tensor-pipe cycles, so the loop
    // around it must stay a handful of uniform-datapath instructions.  All 32 lanes run the control flow
    // (operands provably uniform -> no per-instruction ELECT/broadcast sequences), descriptors are a
    // precomputed 64-bit base whose low word advances by constants, and only the elected lane issues.
    {
      int slotA = 0, slotB = 0;
      uint32_t phaseA = 0, phaseB = 0;
      uint32_t accumulate = 0;
      const uint32_t sub_stride16 = (p.flat ? 16384u : static_cast<uint32_t>(p.ROWS * p.TW) * 128u) >> 4;
      const uint32_t tap_stride16 = (static_cast<uint32_t>(p.TW) * 128u) >> 4;
      const uint32_t idesc = p.idesc;
      const uint32_t ncta = static_cast<uint32_t>(p.N_cta);
      // descriptor high word: SBO = 1024 B (>>4 = 64) at [32,46), version 1 at [46,48), SWIZZLE_128B at [61,64)
      constexpr uint32_t kDescHi = 64u | (1u << 14) | (2u << 29);
      constexpr uint32_t kDescLoFlags = 1u << 16;  // LBO field (canonical 1 for swizzled K-major)
      bool first = true;
      if (p.wide) {
        // positions (A) operand: 16 groups of 8 rows per 128-row sub-tile, one group per image row of the 8-wide tile, PW * 128 B
        // apart; tap (kh, kw) and sub-tile s are start-address offsets ((kh + s * ROWS) * PW + kw) * 128 B into the one slab
        const uint32_t descHiA = static_cast<uint32_t>(p.PW * 8) | (1u << 14) | (2u << 29);
        auto mma_slab = [&](int ch_total, int cb, uint32_t off16_base, int n_taps_h, int n_taps_w) {
          wait_bar(&fullA[slotA], phaseA);
          if (traced && first && lane == 0) trc[2] = ptx::globaltimer_ns();
          const int ch_left = ch_total - cb * 64;
          const int ksteps = ch_left >= 64 ? 4 : (ch_left + 15) >> 4;
          const uint32_t a_lo0 = (((ptx::smem_u32(sA + static_cast<size_t>(slotA) * p.slab_stride) >> 4) & 0x3FFFu) | kDescLoFlags) + off16_base;
          for (int kh = 0; kh < n_taps_h; ++kh) {
            for (int kw = 0; kw < n_taps_w; ++kw) {
              wait_bar(&fullB[slotB], phaseB);
              ptx::tc_fence_after();
              if (traced && first && lane == 0) trc[3] = ptx::globaltimer_ns();
              first = false;
              const uint32_t b_lo0 = ((ptx::smem_u32(sB + static_cast<size_t>(slotB) * p.b_bytes) >> 4) & 0x3FFFu) | kDescLoFlags;
              if (ptx::elect_one()) {
                for (int s = 0; s < nacc_eff; ++s) {
                  const uint32_t a_lo = a_lo0 + static_cast<uint32_t>((kh + s * p.ROWS) * p.PW + kw) * 8u;
                  const uint32_t d = tmem_base + static_cast<uint32_t>(s) * ncta;
                  for (int k = 0; k < ksteps; ++k) {
                    if (CG == 2) ptx::umma_f16_lohi2_cg2(d, a_lo + 2 * k, descHiA, b_lo0 + 2 * k, kDescHi, idesc, accumulate | static_cast<uint32_t>(k));
                    else ptx::umma_f16_lohi2(d, a_lo + 2 * k, descHiA, b_lo0 + 2 * k, kDescHi, idesc, accumulate | static_cast<uint32_t>(k));
                  }
                }
                if (CG == 2) ptx::umma_commit_pair(&emptyB[slotB]); else ptx::umma_commit(&emptyB[slotB]);
              }
              __syncwarp();
              accumulate = 1;
              if (++slotB == p.NB) {
                slotB = 0;
                phaseB ^= 1;
              }
            }
          }
          if (ptx::elect_one()) {
            if (CG == 2) ptx::umma_commit_pair(&emptyA[slotA]); else ptx::umma_commit(&emptyA[slotA]);
          }
          __syncwarp();
          if (++slotA == p.NA) {
            slotA = 0;
            phaseA ^= 1;
          }
        };
        for_each_wslab(p, tc.t, [&](int kt, int ti, int cb) { mma_slab(p.Cin, cb, 0u, p.KH, p.KW); });
        for (int cb2 = 0; cb2 < p.cblocks2; ++cb2) mma_slab(p.Cin2, cb2, p.sc_off16, 1, 1);   // fused shortcut: the centre tap
      } else {
      for_each_slab(p, tc.t, [&](int kt, int ti, int hg, int kw, int cb) {
        wait_bar(&fullA[slotA], phaseA);
        if (traced && first && lane == 0) trc[2] = ptx::globaltimer_ns();
        // K = 16 per MMA; channels beyond Cin are TMA zero-fill in both operands, skip those MMAs entirely
        const int ch_left = p.Cin - cb * 64;
        const int ksteps = ch_left >= 64 ? 4 : (ch_left + 15) >> 4;
        const uint32_t a_lo0 = ((ptx::smem_u32(sA + static_cast<size_t>(slotA) * p.slab_stride) >> 4) & 0x3FFFu) | kDescLoFlags;
        for (int khs = 0; khs < p.KHs; ++khs) {
          wait_bar(&fullB[slotB], phaseB);
          ptx::tc_fence_after();
          if (traced && first && lane == 0) trc[3] = ptx::globaltimer_ns();
          first = false;
          const uint32_t b_lo0 = ((ptx::smem_u32(sB + static_cast<size_t>(slotB) * p.b_bytes) >> 4) & 0x3FFFu) | kDescLoFlags;
          const uint32_t a_lo1 = a_lo0 + static_cast<uint32_t>(khs) * tap_stride16;
          if (ptx::elect_one()) {
            for (int s = 0; s < nacc_eff; ++s) {
              const uint32_t a_lo = a_lo1 + static_cast<uint32_t>(s) * sub_stride16;
              const uint32_t d = tmem_base + static_cast<uint32_t>(s) * ncta;
              if (CG == 2) {
                for (int k = 0; k < ksteps; ++k)
                  ptx::umma_f16_lohi_cg2(d, a_lo + 2 * k, b_lo0 + 2 * k, kDescHi, idesc, accumulate | static_cast<uint32_t>(k));
              } else if (ksteps == 4) {
                ptx::umma_f16_lohi(d, a_lo, b_lo0, kDescHi, idesc, accumulate);
                ptx::umma_f16_lohi(d, a_lo + 2, b_lo0 + 2, kDescHi, idesc, 1);
                ptx::umma_f16_lohi(d, a_lo + 4, b_lo0 + 4, kDescHi, idesc, 1);
                ptx::umma_f16_lohi(d, a_lo + 6, b_lo0 + 6, kDescHi, idesc, 1);
              } else {
                for (int k = 0; k < ksteps; ++k)
                  ptx::umma_f16_lohi(d, a_lo + 2 * k, b_lo0 + 2 * k, kDescHi, idesc, accumulate | static_cast<uint32_t>(k));
              }
            }
            if (CG == 2) ptx::umma_commit_pair(&emptyB[slotB]); else ptx::umma_commit(&emptyB[slotB]);
          }
          __syncwarp();
          accumulate = 1;
          if (++slotB == p.NB) {
            slotB = 0;
            phaseB ^= 1;
          }
        }
        if (ptx::elect_one()) {
          if (CG == 2) ptx::umma_commit_pair(&emptyA[slotA]); else ptx::umma_commit(&emptyA[slotA]);
        }
        __syncwarp();
        if (++slotA == p.NA) {
          slotA = 0;
          phaseA ^= 1;
        }
      });
      for (int cb2 = 0; cb2 < p.cblocks2; ++cb2) {   // fused 1x1 shortcut: row-tap 0 of the unshifted window
        wait_bar(&fullA[slotA], phaseA);
        wait_bar(&fullB[slotB], phaseB);
        ptx::tc_fence_after();
        const int ch_left = p.Cin2 - cb2 * 64;
        const int ksteps = ch_left >= 64 ? 4 : (ch_left + 15) >> 4;
        const uint32_t a_lo0 = ((ptx::smem_u32(sA + static_cast<size_t>(slotA) * p.slab_stride) >> 4) & 0x3FFFu) | kDescLoFlags;
        const uint32_t b_lo0 = ((ptx::smem_u32(sB + static_cast<size_t>(slotB) * p.b_bytes) >> 4) & 0x3FFFu) | kDescLoFlags;
        if (ptx::elect_one()) {
          for (int s = 0; s < nacc_eff; ++s) {
            const uint32_t a_lo = a_lo0 + static_cast<uint32_t>(s) * sub_stride16;
            const uint32_t d = tmem_base + static_cast<uint32_t>(s) * ncta;
            for (int k = 0; k < ksteps; ++k) {
              if (CG == 2) ptx::umma_f16_lohi_cg2(d, a_lo + 2 * k, b_lo0 + 2 * k, kDescHi, idesc, accumulate | static_cast<uint32_t>(k));
              else ptx::umma_f16_lohi(d, a_lo + 2 * k, b_lo0 + 2 * k, kDescHi, idesc, accumulate | static_cast<uint32_t>(k));
            }
          }
          if (CG == 2) {
            ptx::umma_commit_pair(&emptyB[slotB]);
            ptx::umma_commit_pair(&emptyA[slotA]);
          } else {
            ptx::umma_commit(&emptyB[slotB]);
            ptx::umma_commit(&emptyA[slotA]);
          }
        }
        __syncwarp();
        accumulate = 1;
        if (++slotB == p.NB) {
          slotB = 0;
          phaseB ^= 1;
        }
        if (++slotA == p.NA) {
          slotA = 0;
          phaseA ^= 1;
        }
      }
      }
      if (ptx::elect_one()) {
        if (CG == 2) ptx::umma_commit_pair(accFull); else ptx::umma_commit(accFull);
      }
      __syncwarp();
      if (traced && lane == 0) trc[4] = ptx::globaltimer_ns();
    }
  }
  {
    // ------------------------------------------------------------- epilogue (all 8 warps)
    // Warps 4-7 arrive here at once, warps 0-2 when their role loops have issued everything, warp 3 after the
    // TMEM allocation.  Warp w may touch TMEM lanes 32*(w%4)..+31, so two warps share each lane quarter and
    // split the (sub-tile, 32-column chunk) work items between them.
    using E = Elem<DT>;
    const int q = warp & 3;                 // TMEM lane quarter
    const int grp = warp >> 2;              // which half of the work items
    const int r = q * 32 + lane;            // accumulator row owned by this thread
    wait_bar(accFull, 0);
    ptx::tc_fence_after();
    if (traced && threadIdx.x == 128) trc[5] = ptx::globaltimer_ns();
    const int chalf = p.up_time == 2 ? p.Cout / 2 : p.Cout;
    const int bias_b = (p.flags & CVVAE_CONV_W_PER_BATCH) ? 0 : tc.b;  // batched GEMM: a row bias is shared by the batch items
    int item = 0;
    if (p.tma_epi) {
      // ---- TMEM -> registers -> SWIZZLE_128B staging tile (32 positions x 64 channels, 4 KB) -> TMA store.
      // A warp's direct 16-byte stores would touch 32 different 128-byte lines per instruction (position stride
      // = C*2 bytes); the bulk tensor store writes full lines and clips partial tiles by itself.  The residual
      // tile comes in the same way (TMA load into the staging tile, added in place).  Staging reuses the drained
      // A ring: two 4 KB tiles per warp.
      uint8_t* stage = sA + static_cast<size_t>(warp) * 8192;
      uint32_t res_phase = 0;
      int nbuf = 0;
      const int r0 = q * 32;
      const uint32_t row_off = static_cast<uint32_t>(lane) * 128u;
      const uint32_t sw = static_cast<uint32_t>(lane & 7);
      for (int s = 0; s < nacc_eff; ++s) {
        int h, w, h_me, w_me;
        if (p.flat) {
          h = 0;
          w = tc.w0 + s * 128 + r0;
          h_me = 0;
          w_me = w + lane;
        } else {
          h = tc.h0 + s * p.ROWS + r0 / p.TW;
          w = tc.w0 + r0 % p.TW;
          h_me = tc.h0 + s * p.ROWS + (r0 + lane) / p.TW;
          w_me = tc.w0 + (r0 + lane) % p.TW;
        }
        float bias_m = 0.f;
        if (p.bias && (p.flags & CVVAE_CONV_BIAS_ALONG_M)) {
          const long long m_index =
              ((static_cast<long long>(bias_b) * p.T_out + tc.t) * p.H_out + h_me) * static_cast<long long>(p.W_out) + w_me;
          if (h_me < p.H_out && w_me < p.W_out) bias_m = __ldg(p.bias + m_index);
        }
        for (int c0 = 0; c0 < p.N_cta; c0 += 64) {
          const int cg0 = tc.n0 + c0;
          if (cg0 >= p.Cout) break;               // warp-uniform
          if (((item++) & 1) != grp) continue;    // warp-uniform
          int cbase = cg0, t_o = tc.t;
          if (p.up_time == 2) {
            const int n_il = cg0 / chalf;
            cbase = cg0 - n_il * chalf;
            t_o = 2 * tc.t + n_il - 1;
            if (t_o < 0) continue;
          }
          uint8_t* tile = stage + (nbuf & 1) * 4096;
          const uint32_t tile_u32 = ptx::smem_u32(tile);
          // the bulk store that last read this buffer (two items ago) must be done reading
          if (lane == 0) ptx::bulk_wait_read<1>();
          __syncwarp();
          if (p.residual) {
            if (lane == 0) {
              ptx::mbar_expect_tx(&resBar[warp], 4096);
              ptx::tma_load_5d(tile, &tmR, &resBar[warp], cbase, w, h, t_o, tc.b);
            }
            wait_bar(&resBar[warp], res_phase);
            res_phase ^= 1;
          }
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int cc0 = c0 + half * 32;
            uint32_t v[32];
            if (cc0 < p.N_cta) {
              ptx::tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(s * p.N_cta + cc0), v);
              ptx::tmem_ld_wait();
            } else {
#pragma unroll
              for (int c = 0; c < 32; ++c) v[c] = 0u;
            }
            float bv[32];
            const int cgh = tc.n0 + cc0;
            if (p.bias && !(p.flags & CVVAE_CONV_BIAS_ALONG_M) && cgh + 32 <= p.Cout) {
              if (p.bias_vec) {
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                  const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + cgh) + g);
                  bv[4 * g] = b4.x; bv[4 * g + 1] = b4.y; bv[4 * g + 2] = b4.z; bv[4 * g + 3] = b4.w;
                }
              } else {
#pragma unroll
                for (int c = 0; c < 32; ++c) bv[c] = __ldg(p.bias + cgh + c);
              }
            } else if (p.bias && !(p.flags & CVVAE_CONV_BIAS_ALONG_M)) {
#pragma unroll
              for (int c = 0; c < 32; ++c) bv[c] = (cgh + c < p.Cout) ? __ldg(p.bias + cgh + c) : 0.f;
            } else {
#pragma unroll
              for (int c = 0; c < 32; ++c) bv[c] = bias_m;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t chunk = static_cast<uint32_t>(half * 4 + j);
              const uint32_t addr = tile_u32 + row_off + ((chunk ^ sw) << 4);
              uint4 rv = make_uint4(0, 0, 0, 0);
              if (p.residual) rv = ptx::ld_shared_v4(addr);
              const uint32_t rw[4] = {rv.x, rv.y, rv.z, rv.w};
              uint32_t ow[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int c = j * 8 + e * 2;
                float a0 = fmaf(__uint_as_float(v[c]), p.alpha, bv[c]);
                float a1 = fmaf(__uint_as_float(v[c + 1]), p.alpha, bv[c + 1]);
                if (p.residual) {
                  const float2 rf = E::to_f2(rw[e]);
                  a0 += rf.x;
                  a1 += rf.y;
                }
                ow[e] = E::pack2(a0, a1);
              }
              ptx::st_shared_v4(addr, ow[0], ow[1], ow[2], ow[3]);
            }
          }
          if (p.gn_stats) {
            // GroupNorm statistics of the consumer, from the staged (already rounded) tile: lane l owns channels
            // 2l, 2l+1 of this 64-channel group and walks the 32 rows (conflict-free: one 128-byte row per step)
            __syncwarp();
            const unsigned valid = __ballot_sync(0xffffffffu, (h_me < p.H_out) && (w_me < p.W_out));
            float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
            const uint32_t chunk = static_cast<uint32_t>(lane >> 2), word = static_cast<uint32_t>(lane & 3) * 4u;
            for (int rr = 0; rr < 32; ++rr) {
              if (!((valid >> rr) & 1u)) continue;
              uint32_t u;
              asm volatile("ld.shared.b32 %0, [%1];" : "=r"(u) : "r"(tile_u32 + rr * 128u + ((chunk ^ (rr & 7u)) << 4) + word));
              const float2 f = E::to_f2(u);
              s0 += f.x; q0 = fmaf(f.x, f.x, q0);
              s1 += f.y; q1 = fmaf(f.y, f.y, q1);
            }
            const int ch = cbase + 2 * lane;
            if (p.gn_cpg >= 2) {
              float ts = s0 + s1, tq = q0 + q1;
              for (int o = 1; o < (p.gn_cpg >> 1) && o < 32; o <<= 1) {
                ts += __shfl_xor_sync(0xffffffffu, ts, o);
                tq += __shfl_xor_sync(0xffffffffu, tq, o);
              }
              const int lanes_per_group = min(p.gn_cpg >> 1, 32);
              if ((lane % lanes_per_group) == 0 && ch < p.yC) {
                atomicAdd(&gn_bins[(ch / p.gn_cpg) * 2], gn_fix(ts, kGnSumScale));
                atomicAdd(&gn_bins[(ch / p.gn_cpg) * 2 + 1], gn_fix(tq, kGnSqScale));
              }
            } else if (ch < p.yC) {  // one channel per group
              atomicAdd(&gn_bins[ch * 2], gn_fix(s0, kGnSumScale));
              atomicAdd(&gn_bins[ch * 2 + 1], gn_fix(q0, kGnSqScale));
              if (ch + 1 < p.yC) {
                atomicAdd(&gn_bins[(ch + 1) * 2], gn_fix(s1, kGnSumScale));
                atomicAdd(&gn_bins[(ch + 1) * 2 + 1], gn_fix(q1, kGnSqScale));
              }
            }
          }
          ptx::fence_proxy_async();   // generic-proxy writes -> visible to the TMA (async proxy)
          __syncwarp();
          if (lane == 0) {
            ptx::tma_store_5d(&tmY, tile, cbase, w, h, t_o, tc.b);
            ptx::bulk_commit();
          }
          ++nbuf;
        }
      }
      if (lane == 0) ptx::bulk_wait<0>();
      __syncwarp();
    } else
    for (int s = 0; s < nacc_eff; ++s) {
      int h, w;
      if (p.flat) {
        h = 0;
        w = tc.w0 + s * 128 + r;
      } else {
        h = tc.h0 + s * p.ROWS + r / p.TW;
        w = tc.w0 + r % p.TW;
      }
      const bool pix_ok = (h < p.H_out) && (w < p.W_out);
      const long long m_index =
          ((static_cast<long long>(bias_b) * p.T_out + tc.t) * p.H_out + h) * static_cast<long long>(p.W_out) + w;
      for (int c0 = 0; c0 < p.N_cta; c0 += 32) {
        const int cg0 = tc.n0 + c0;
        if (cg0 >= p.Cout) break;  // warp-uniform
        if (((item++) & 1) != grp) continue;  // warp-uniform
        uint32_t v[32];
        ptx::tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(s * p.N_cta + c0), v);
        ptx::tmem_ld_wait();
        if (!pix_ok) continue;
        // output coordinates (time interleave of Upsample3D folded in)
        int n_il = 0, cbase = cg0, t_o = tc.t;
        if (p.up_time == 2) {
          n_il = cg0 / chalf;
          cbase = cg0 - n_il * chalf;
          t_o = 2 * tc.t + n_il - 1;
          if (t_o < 0) continue;
        }
        const long long off = tc.b * p.ys_b + t_o * p.ys_t + h * p.ys_h + w * p.ys_w;
        const float bias_m = (p.bias && (p.flags & CVVAE_CONV_BIAS_ALONG_M)) ? __ldg(p.bias + m_index) : 0.f;
        const bool chunk_full = (cg0 + 32 <= p.Cout) && (p.up_time != 2 || (cbase + 32 <= chalf));
        if (p.flags & CVVAE_CONV_OUT_F32) {
          // fp32 logits (S = q k^T): no residual, no interleave
          float* yf = reinterpret_cast<float*>(p.y) + off;
          if (p.vec_ok && chunk_full) {
            float4* y4 = reinterpret_cast<float4*>(yf + cbase * p.ys_c);
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              float o4[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float a = __uint_as_float(v[g * 4 + j]) * p.alpha;
                if (p.bias) a += (p.flags & CVVAE_CONV_BIAS_ALONG_M) ? bias_m : __ldg(p.bias + cg0 + g * 4 + j);
                o4[j] = a;
              }
              y4[g] = make_float4(o4[0], o4[1], o4[2], o4[3]);
            }
          } else {
            for (int c = 0; c < 32 && cg0 + c < p.Cout; ++c) {
              float a = __uint_as_float(v[c]) * p.alpha;
              if (p.bias) a += (p.flags & CVVAE_CONV_BIAS_ALONG_M) ? bias_m : __ldg(p.bias + cg0 + c);
              yf[(cg0 + c) * p.ys_c] = a;
            }
          }
        } else if (p.vec_ok && chunk_full) {
          typename E::T* yp = reinterpret_cast<typename E::T*>(p.y) + off + cbase;
          const typename E::T* rp =
              p.residual ? reinterpret_cast<const typename E::T*>(p.residual) + off + cbase : nullptr;
          float bv[32];
          if (p.bias && !(p.flags & CVVAE_CONV_BIAS_ALONG_M)) {
            if (p.bias_vec) {
#pragma unroll
              for (int g = 0; g < 8; ++g) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + cg0) + g);
                bv[4 * g] = b4.x; bv[4 * g + 1] = b4.y; bv[4 * g + 2] = b4.z; bv[4 * g + 3] = b4.w;
              }
            } else {
#pragma unroll
              for (int c = 0; c < 32; ++c) bv[c] = __ldg(p.bias + cg0 + c);
            }
          } else {
#pragma unroll
            for (int c = 0; c < 32; ++c) bv[c] = bias_m;
          }
          // residual: issue all four 128-bit loads before the arithmetic
          uint4 rv4[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) rv4[g] = rp ? __ldg(reinterpret_cast<const uint4*>(rp) + g) : make_uint4(0, 0, 0, 0);
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const uint32_t rw[4] = {rv4[g].x, rv4[g].y, rv4[g].z, rv4[g].w};
            uint32_t ow[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int c = g * 8 + j * 2;
              float a0 = fmaf(__uint_as_float(v[c]), p.alpha, bv[c]);
              float a1 = fmaf(__uint_as_float(v[c + 1]), p.alpha, bv[c + 1]);
              if (rp) {
                float2 rf = E::to_f2(rw[j]);
                a0 += rf.x;
                a1 += rf.y;
              }
              ow[j] = E::pack2(a0, a1);
            }
            reinterpret_cast<uint4*>(yp)[g] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
          }
        } else {
          for (int c = 0; c < 32; ++c) {
            const int cg = cg0 + c;
            if (cg >= p.Cout) break;
            int cc = cg, tt = tc.t;
            if (p.up_time == 2) {
              const int n2 = cg / chalf;
              cc = cg - n2 * chalf;
              tt = 2 * tc.t + n2 - 1;
              if (tt < 0) continue;
            }
            const long long o2 = tc.b * p.ys_b + tt * p.ys_t + h * p.ys_h + w * p.ys_w + cc * p.ys_c;
            float a = __uint_as_float(v[c]) * p.alpha;
            if (p.bias) a += (p.flags & CVVAE_CONV_BIAS_ALONG_M) ? bias_m : __ldg(p.bias + cg);
            if (p.residual) a += E::to_f(reinterpret_cast<const typename E::T*>(p.residual)[o2]);
            reinterpret_cast<typename E::T*>(p.y)[o2] = E::from_f(a);
          }
        }
      }
    }
  }

  if (traced && threadIdx.x == 128) trc[6] = ptx::globaltimer_ns();
  ptx::tc_fence_before();
  if (CG == 2) ptx::cluster_sync(); else __syncthreads();  // the leader's MMAs wrote the peer's TMEM too
  if (p.gn_stats && static_cast<int>(threadIdx.x) < 2 * p.gn_groups) {
    const unsigned long long vsum = gn_bins[threadIdx.x];
    if (vsum != 0ull)
      atomicAdd(reinterpret_cast<unsigned long long*>(p.gn_stats) + static_cast<size_t>(tc.b) * 2 * p.gn_groups + threadIdx.x, vsum);
  }
  if (warp == 3) {
    ptx::tc_fence_after();
    if (CG == 2) ptx::tmem_dealloc_cg2(tmem_base, kTmemCols); else ptx::tmem_dealloc(tmem_base, kTmemCols);
    if (traced && lane == 0) {
      unsigned smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      trc[7] = (ptx::globaltimer_ns() & 0xFFFFFFFFFFFFull) | (static_cast<unsigned long long>(smid) << 48);
    }
  }
}


// ------------------------------------------------------------------------------------------------------------------
// Persistent, operand-swapped variant for the Cout == 128 layers (the full-resolution layers, where a CTA's mainloop is
// short: 11 us for a 1x3x3 conv).  One CTA per SM walks tiles of 256 output positions; the 128-channel x 256-position
// accumulator is double buffered in TMEM (2 x 256 columns), so the 8 epilogue warps drain tile i while the MMA warp
// already runs tile i+1 and the TMA producers prefetch ahead across tile boundaries: set-up, first-load latency and the
// whole epilogue leave the critical path.  Price: each staged weight tile now feeds one accumulator instead of two.
// Warps: 0 A producer, 1 B producer, 2 MMA issuer, 3 TMEM allocator, 4-11 epilogue (two per TMEM lane quarter).
static constexpr int kPersistThreads = 384;

template <int DT>
__global__ void __launch_bounds__(kPersistThreads, 1)
    conv_tc_psw_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                       const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmR,
                       const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
                       const ConvTcParams p) {
  using E = Elem<DT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = sA + static_cast<size_t>(p.NA) * p.slab_stride;
  uint8_t* sStage = sB + static_cast<size_t>(p.NB) * p.b_bytes;  // 8 warps x 2 x 2 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStage + 32768);
  uint64_t* fullA = bars;          // [8]
  uint64_t* emptyA = bars + 8;     // [8]
  uint64_t* fullB = bars + 16;     // [8]
  uint64_t* emptyB = bars + 24;    // [8]
  uint64_t* accFull = bars + 32;   // [2]
  uint64_t* accEmpty = bars + 34;  // [2]
  uint64_t* resBar = bars + 40;    // [8]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 36);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < p.NA; ++i) {
      ptx::mbar_init(&fullA[i], 1);
      ptx::mbar_init(&emptyA[i], 1);
    }
    for (int i = 0; i < p.NB; ++i) {
      ptx::mbar_init(&fullB[i], 1);
      ptx::mbar_init(&emptyB[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&accFull[i], 1);
      ptx::mbar_init(&accEmpty[i], 8);  // one arrival per epilogue warp
    }
    for (int i = 0; i < 8; ++i) ptx::mbar_init(&resBar[i], 1);
    ptx::fence_mbar_init();
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    ptx::prefetch_tmap(&tmY);
  }
  if (warp == 3) {
    ptx::tmem_alloc(tmem_slot, kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tile0 = blockIdx.x, tstep = gridDim.x;

  if (warp == 0) {
    // ------------------------------------------------------------- A producer (runs ahead across tiles)
    int slot = 0;
    uint32_t phase = 0;
    for (int tile = tile0; tile < p.n_tiles; tile += tstep) {
      const TileCoord tc = decode_tile<1>(p, 0, tile);
      if (p.wide) {
        for_each_wslab(p, tc.t, [&](int kt, int ti, int cb) {
          wait_bar(&emptyA[slot], phase ^ 1);
          if (ptx::elect_one()) {
            ptx::mbar_expect_tx(&fullA[slot], p.slab_bytes);
            ptx::tma_load_5d(sA + static_cast<size_t>(slot) * p.slab_stride, &tmA, &fullA[slot], cb * 64, tc.w0 + p.off_w,
                             tc.h0 + p.off_h, ti, tc.b);
          }
          __syncwarp();
          if (++slot == p.NA) {
            slot = 0;
            phase ^= 1;
          }
        });
        for (int cb2 = 0; cb2 < p.cblocks2; ++cb2) {   // fused 1x1 shortcut: same window (with its halo) of the second input
          wait_bar(&emptyA[slot], phase ^ 1);
          if (ptx::elect_one()) {
            ptx::mbar_expect_tx(&fullA[slot], p.slab_bytes);
            ptx::tma_load_5d(sA + static_cast<size_t>(slot) * p.slab_stride, &tmA2, &fullA[slot], cb2 * 64, tc.w0 + p.off_w,
                             tc.h0 + p.off_h, tc.t, tc.b);
          }
          __syncwarp();
          if (++slot == p.NA) {
            slot = 0;
            phase ^= 1;
          }
        }
        continue;
      }
      for_each_slab(p, tc.t, [&](int kt, int ti, int hg, int kw, int cb) {
        wait_bar(&emptyA[slot], phase ^ 1);
        if (ptx::elect_one()) {
          ptx::mbar_expect_tx(&fullA[slot], p.slab_bytes);
          ptx::tma_load_5d(sA + static_cast<size_t>(slot) * p.slab_stride, &tmA, &fullA[slot], cb * 64,
                           tc.w0 * p.sw + kw + p.off_w, tc.h0 * p.sh + hg * p.KHs + p.off_h, ti, tc.b);
        }
        __syncwarp();
        if (++slot == p.NA) {
          slot = 0;
          phase ^= 1;
        }
      });
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------- B producer
    int slot = 0;
    uint32_t phase = 0;
    for (int tile = tile0; tile < p.n_tiles; tile += tstep) {
      const TileCoord tc = decode_tile<1>(p, 0, tile);
      auto load_tap = [&](int tap, int cb) {
        wait_bar(&emptyB[slot], phase ^ 1);
        if (ptx::elect_one()) {
          ptx::mbar_expect_tx(&fullB[slot], p.b_bytes);
          ptx::tma_load_3d(sB + static_cast<size_t>(slot) * p.b_bytes, &tmB, &fullB[slot], cb * 64, tc.n0, tap);
        }
        __syncwarp();
        if (++slot == p.NB) {
          slot = 0;
          phase ^= 1;
        }
      };
      if (p.wide) {
        for_each_wslab(p, tc.t, [&](int kt, int ti, int cb) {
          for (int kh = 0; kh < p.KH; ++kh)
            for (int kw = 0; kw < p.KW; ++kw) load_tap((kt * p.KH + kh) * p.KW + kw, cb);
        });
        for (int cb2 = 0; cb2 < p.cblocks2; ++cb2) {   // shortcut weights [Cout][Cin2]
          wait_bar(&emptyB[slot], phase ^ 1);
          if (ptx::elect_one()) {
            ptx::mbar_expect_tx(&fullB[slot], p.b_bytes);
            ptx::tma_load_3d(sB + static_cast<size_t>(slot) * p.b_bytes, &tmB2, &fullB[slot], cb2 * 64, tc.n0, 0);
          }
          __syncwarp();
          if (++slot == p.NB) {
            slot = 0;
            phase ^= 1;
          }
        }
        continue;
      }
      for_each_slab(p, tc.t, [&](int kt, int ti, int hg, int kw, int cb) {
        for (int khs = 0; khs < p.KHs; ++khs) load_tap((kt * p.KH + hg * p.KHs + khs) * p.KW + kw, cb);
      });
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------- MMA issuer
    int slotA = 0, slotB = 0;
    uint32_t phaseA = 0, phaseB = 0;
    const uint32_t tap_stride16 = (static_cast<uint32_t>(p.TW) * 128u) >> 4;
    const uint32_t idesc = p.idesc;
    constexpr uint32_t kDescHi = 64u | (1u << 14) | (2u << 29);
    constexpr uint32_t kDescLoFlags = 1u << 16;
    int it = 0;
    for (int tile = tile0; tile < p.n_tiles; tile += tstep, ++it) {
      const TileCoord tc = decode_tile<1>(p, 0, tile);
      const int st = it & 1;
      wait_bar(&accEmpty[st], ((it >> 1) & 1) ^ 1);  // the epilogue has drained this TMEM stage (free on first use)
      ptx::tc_fence_after();
      const uint32_t d = tmem_base + static_cast<uint32_t>(st) * 256u;
      uint32_t accumulate = 0;
      if (p.wide) {
        // positions operand: 32 groups of 8 rows, one group per image row of the 8-wide tile, PW * 128 B apart
        const uint32_t descHiX = static_cast<uint32_t>(p.PW * 8) | (1u << 14) | (2u << 29);
        for_each_wslab(p, tc.t, [&](int kt, int ti, int cb) {
          wait_bar(&fullA[slotA], phaseA);
          const int ch_left = p.Cin - cb * 64;
          const int ksteps = ch_left >= 64 ? 4 : (ch_left + 15) >> 4;
          const uint32_t a_lo0 = ((ptx::smem_u32(sA + static_cast<size_t>(slotA) * p.slab_stride) >> 4) & 0x3FFFu) | kDescLoFlags;
          for (int kh = 0; kh < p.KH; ++kh) {
            for (int kw = 0; kw < p.KW; ++kw) {
              wait_bar(&fullB[slotB], phaseB);
              ptx::tc_fence_after();
              const uint32_t w_lo = ((ptx::smem_u32(sB + static_cast<size_t>(slotB) * p.b_bytes) >> 4) & 0x3FFFu) | kDescLoFlags;
              const uint32_t x_lo = a_lo0 + static_cast<uint32_t>(kh * p.PW + kw) * 8u;
              if (ptx::elect_one()) {
                for (int k = 0; k < ksteps; ++k)
                  ptx::umma_f16_lohi2(d, w_lo + 2 * k, kDescHi, x_lo + 2 * k, descHiX, idesc, accumulate | static_cast<uint32_t>(k));
                ptx::umma_commit(&emptyB[slotB]);
              }
              __syncwarp();
              accumulate = 1;
              if (++slotB == p.NB) {
                slotB = 0;
                phaseB ^= 1;
              }
            }
          }
          if (ptx::elect_one()) ptx::umma_commit(&emptyA[slotA]);
          __syncwarp();
          if (++slotA == p.NA) {
            slotA = 0;
            phaseA ^= 1;
          }
        });
        for (int cb2 = 0; cb2 < p.cblocks2; ++cb2) {   // fused 1x1 shortcut: the centre tap of the second input's slab
          wait_bar(&fullA[slotA], phaseA);
          wait_bar(&fullB[slotB], phaseB);
          ptx::tc_fence_after();
          const int ch_left = p.Cin2 - cb2 * 64;
          const int ksteps = ch_left >= 64 ? 4 : (ch_left + 15) >> 4;
          const uint32_t x_lo = (((ptx::smem_u32(sA + static_cast<size_t>(slotA) * p.slab_stride) >> 4) & 0x3FFFu) | kDescLoFlags) + p.sc_off16;
          const uint32_t w_lo = ((ptx::smem_u32(sB + static_cast<size_t>(slotB) * p.b_bytes) >> 4) & 0x3FFFu) | kDescLoFlags;
          if (ptx::elect_one()) {
            for (int k = 0; k < ksteps; ++k)
              ptx::umma_f16_lohi2(d, w_lo + 2 * k, kDescHi, x_lo + 2 * k, descHiX, idesc, accumulate | static_cast<uint32_t>(k));
            ptx::umma_commit(&emptyB[slotB]);
            ptx::umma_commit(&emptyA[slotA]);
          }
          __syncwarp();
          accumulate = 1;
          if (++slotB == p.NB) {
            slotB = 0;
            phaseB ^= 1;
          }
          if (++slotA == p.NA) {
            slotA = 0;
            phaseA ^= 1;
          }
        }
        if (ptx::elect_one()) ptx::umma_commit(&accFull[st]);
        __syncwarp();
        continue;
      }
      for_each_slab(p, tc.t, [&](int kt, int ti, int hg, int kw, int cb) {
        wait_bar(&fullA[slotA], phaseA);
        const int ch_left = p.Cin - cb * 64;
        const int ksteps = ch_left >= 64 ? 4 : (ch_left + 15) >> 4;
        const uint32_t a_lo0 = ((ptx::smem_u32(sA + static_cast<size_t>(slotA) * p.slab_stride) >> 4) & 0x3FFFu) | kDescLoFlags;
        for (int khs = 0; khs < p.KHs; ++khs) {
          wait_bar(&fullB[slotB], phaseB);
          ptx::tc_fence_after();
          const uint32_t w_lo = ((ptx::smem_u32(sB + static_cast<size_t>(slotB) * p.b_bytes) >> 4) & 0x3FFFu) | kDescLoFlags;
          const uint32_t x_lo = a_lo0 + static_cast<uint32_t>(khs) * tap_stride16;
          if (ptx::elect_one()) {
            for (int k = 0; k < ksteps; ++k)
              ptx::umma_f16_lohi(d, w_lo + 2 * k, x_lo + 2 * k, kDescHi, idesc, accumulate | static_cast<uint32_t>(k));
            ptx::umma_commit(&emptyB[slotB]);
          }
          __syncwarp();
          accumulate = 1;
          if (++slotB == p.NB) {
            slotB = 0;
            phaseB ^= 1;
          }
        }
        if (ptx::elect_one()) ptx::umma_commit(&emptyA[slotA]);
        __syncwarp();
        if (++slotA == p.NA) {
          slotA = 0;
          phaseA ^= 1;
        }
      });
      if (ptx::elect_one()) ptx::umma_commit(&accFull[st]);
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------- epilogue warps
    const int ew = warp - 4;           // 0..7
    const int q = warp & 3;            // TMEM lane quarter (warp id mod 4)
    const int grp = ew >> 2;           // which half of the 8 items of a tile
    uint8_t* stage = sStage + static_cast<size_t>(ew) * 4096;
    uint32_t res_phase = 0;
    int nbuf = 0;
    const int c_me = q * 32 + lane;    // output channel owned by this thread (n0 == 0: Cout == 128)
    const float bias_c = p.bias ? __ldg(p.bias + c_me) : 0.f;
    float gs = 0.f, gq = 0.f;
    int cur_b = -1;
    auto flush_stats = [&](int b) {
      if (!p.gn_stats || b < 0) return;
      float ts = gs, tq = gq;
      for (int o = 1; o < p.gn_cpg && o < 32; o <<= 1) {
        ts += __shfl_xor_sync(0xffffffffu, ts, o);
        tq += __shfl_xor_sync(0xffffffffu, tq, o);
      }
      const int lanes_per_group = min(p.gn_cpg, 32);
      if ((lane % lanes_per_group) == 0) {
        unsigned long long* o64 = reinterpret_cast<unsigned long long*>(p.gn_stats) + (static_cast<size_t>(b) * p.gn_groups + c_me / p.gn_cpg) * 2;
        atomicAdd(o64, gn_fix(ts, kGnSumScale));
        atomicAdd(o64 + 1, gn_fix(tq, kGnSqScale));
      }
      gs = gq = 0.f;
    };
    int it = 0;
    for (int tile = tile0; tile < p.n_tiles; tile += tstep, ++it) {
      const TileCoord tc = decode_tile<1>(p, 0, tile);
      const int st = it & 1;
      if (tc.b != cur_b) {
        flush_stats(cur_b);
        cur_b = tc.b;
      }
      wait_bar(&accFull[st], (it >> 1) & 1);
      ptx::tc_fence_after();
      const int rows_valid = min(p.TH, max(0, p.H_out - tc.h0));  // rows of this tile inside the image
      for (int jj = 0; jj < 4; ++jj) {
        const int j = grp * 4 + jj;                 // 32-position chunk of the 256-position tile
        const int f0 = j * 32;
        uint32_t v[32];
        ptx::tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(st * 256 + f0), v);
        ptx::tmem_ld_wait();
        if (jj == 3) {
          // last TMEM read of this tile by this warp: hand the stage back to the MMA warp before the stores
          ptx::tc_fence_before();
          if (lane == 0) ptx::mbar_arrive(&accEmpty[st]);
        }
        if (f0 / p.TW >= rows_valid) continue;       // chunk entirely below the image (warp-uniform)
        const int h = tc.h0 + f0 / p.TW, w = tc.w0 + f0 % p.TW;
        const int hi = tc.h0 + (f0 + lane) / p.TW, wi = tc.w0 + (f0 + lane) % p.TW;
        const unsigned valid = __ballot_sync(0xffffffffu, (hi < p.H_out) && (wi < p.W_out));
        uint8_t* tilebuf = stage + (nbuf & 1) * 2048;
        const uint32_t tile_u32 = ptx::smem_u32(tilebuf);
        if (lane == 0) ptx::bulk_wait_read<1>();
        __syncwarp();
        if (p.residual) {
          if (lane == 0) {
            ptx::mbar_expect_tx(&resBar[ew], 2048);
            ptx::tma_load_5d(tilebuf, &tmR, &resBar[ew], q * 32, w, h, tc.t, tc.b);
          }
          wait_bar(&resBar[ew], res_phase);
          res_phase ^= 1;
        }
        const uint32_t my = tile_u32 + static_cast<uint32_t>(lane) * 2u;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float a = fmaf(__uint_as_float(v[i]), p.alpha, bias_c);
          if (p.residual) {
            uint16_t r16;
            asm volatile("ld.shared.u16 %0, [%1];" : "=h"(r16) : "r"(my + i * 64u));
            a += E::to_f(*reinterpret_cast<const typename E::T*>(&r16));
          }
          const typename E::T o = E::from_f(a);
          if (p.gn_stats && ((valid >> i) & 1u)) {
            const float of = E::to_f(o);
            gs += of;
            gq = fmaf(of, of, gq);
          }
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(my + i * 64u), "h"(*reinterpret_cast<const uint16_t*>(&o)) : "memory");
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          ptx::tma_store_5d(&tmY, tilebuf, q * 32, w, h, tc.t, tc.b);
          ptx::bulk_commit();
        }
        ++nbuf;
      }
    }
    flush_stats(cur_b);
    if (lane == 0) ptx::bulk_wait<0>();
    __syncwarp();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 3) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------- host side
// cuTensorMapEncodeTiled is a pure function of its arguments and costs 1-2 us on the host; a network pass issues the same
// few hundred (pointer, shape) combinations call after call (the activation buffers come back from the caching allocator at
// the same addresses), so the encoded maps are memoised per thread, keyed by the full argument list (SURVEY 8b: "optional
// descriptor cache keyed by (ptr, shape)").
struct TmapKey {
  const void* ptr;
  uint32_t rank, swizzle;
  cuuint64_t dims[5], strides[4];
  cuuint32_t box[5], estr[5];
  bool operator==(const TmapKey& o) const { return memcmp(this, &o, sizeof(TmapKey)) == 0; }
};
struct TmapSlot {
  TmapKey key;
  CUtensorMap map;
  bool valid;
};
static constexpr int kTmapSlots = 1024;

static bool encode_map(CUtensorMap* m, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_b,
                       const cuuint32_t* box, const cuuint32_t* estr,
                       CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  static thread_local TmapSlot* cache = nullptr;
  if (!cache) cache = static_cast<TmapSlot*>(calloc(kTmapSlots, sizeof(TmapSlot)));
  TmapKey key;
  memset(&key, 0, sizeof(key));
  key.ptr = ptr;
  key.rank = static_cast<uint32_t>(rank);
  key.swizzle = static_cast<uint32_t>(swizzle);
  for (int i = 0; i < rank; ++i) {
    key.dims[i] = dims[i];
    key.box[i] = box[i];
    key.estr[i] = estr[i];
    if (i + 1 < rank) key.strides[i] = strides_b[i];
  }
  uint64_t h = 1469598103934665603ull;  // FNV-1a over the key bytes
  const unsigned char* kb = reinterpret_cast<const unsigned char*>(&key);
  for (size_t i = 0; i < sizeof(key); ++i) h = (h ^ kb[i]) * 1099511628211ull;
  TmapSlot* slot = cache ? &cache[h % kTmapSlots] : nullptr;
  if (slot && slot->valid && slot->key == key) {
    *m = slot->map;
    return true;
  }
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return false;
  }
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, rank, const_cast<void*>(ptr), dims, strides_b, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d): rank %d dims [%llu %llu %llu %llu %llu] box [%u %u %u %u %u]",
              (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
              (unsigned long long)(rank > 4 ? dims[4] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0,
              rank > 3 ? box[3] : 0, rank > 4 ? box[4] : 0);
    return false;
  }
  if (slot) {
    slot->key = key;
    slot->map = *m;
    slot->valid = true;
  }
  return true;
}

bool conv_tc_eligible(const cvvae_conv_desc* d, const char** why) {
  const cvvae_tensor5& x = d->x;
  auto fail = [&](const char* m) {
    if (why) *why = m;
    return false;
  };
  if (x.s_c != 1) return fail("input channel stride != 1");
  if (d->w_ld % 8 != 0 || (d->w_ld == 0 && x.C % 8 != 0)) return fail("weight row stride not a 16-byte multiple");
  if ((x.s_w % 8) || (x.s_h % 8) || (x.s_t % 8) || (x.s_b % 8)) return fail("input strides not 16-byte multiples");
  if (reinterpret_cast<uintptr_t>(x.ptr) % 16) return fail("input pointer not 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(d->w) % 16) return fail("weight pointer not 16-byte aligned");
  if (d->pad_hw != CVVAE_PAD_ZERO) {
    // replicate padding in H/W is only needed when a tap can actually leave the image
    const int lo_h = d->off_h, hi_h = (d->y.H - 1) * d->sh + d->KH - 1 + d->off_h;
    const int lo_w = d->off_w, hi_w = (d->y.W - 1) * d->sw + d->KW - 1 + d->off_w;
    if (lo_h < 0 || lo_w < 0 || hi_h >= x.H || hi_w >= x.W) return fail("replicate H/W padding needs a pre-padded input");
  }
  if (d->sh > 2 || d->sw > 2 || d->sh != d->sw) return fail("unsupported spatial stride");
  if (d->KH > 3 || d->KW > 3 || d->KT > 3) return fail("kernel extent > 3");
  if (d->up_time == 2 && (d->Cout % 2)) return fail("odd Cout with up_time");
  return true;
}

static unsigned long long* g_trace_buf = nullptr;
static int g_trace_n = 0;
void conv_tc_set_trace(unsigned long long* buf, int n) {
  g_trace_buf = buf;
  g_trace_n = n;
}

int conv_tc_launch(const cvvae_conv_desc* d, cudaStream_t stream) {
  const char* why = nullptr;
  if (!conv_tc_eligible(d, &why)) {
    set_error("cvvae_conv3d_tc: not eligible: %s", why);
    return CVVAE_E_UNSUPPORTED;
  }
  const cvvae_tensor5& x = d->x;
  const cvvae_tensor5& y = d->y;
  ConvTcParams p{};
  p.B = x.B;
  p.T_in = x.T;
  p.Cin = x.C;
  p.Cout = d->Cout;
  p.up_time = d->up_time == 2 ? 2 : 1;
  p.T_out = p.up_time == 2 ? (y.T + 1) / 2 : y.T;
  p.H_out = y.H;
  p.W_out = y.W;
  p.KT = d->KT; p.KH = d->KH; p.KW = d->KW;
  p.st = d->st; p.sh = d->sh; p.sw = d->sw;
  p.off_t = d->off_t; p.off_h = d->off_h; p.off_w = d->off_w;
  p.pad_t = d->pad_t;
  p.flags = d->flags;
  p.alpha = d->alpha;
  p.bias = d->bias;
  p.residual = d->residual;
  p.y = y.ptr;
  p.ys_b = y.s_b; p.ys_t = y.s_t; p.ys_h = y.s_h; p.ys_w = y.s_w; p.ys_c = y.s_c;
  p.yC = y.C; p.yT = y.T;
  p.trace = g_trace_buf;
  p.trace_n = g_trace_n;
  p.bias_vec = d->bias && (reinterpret_cast<uintptr_t>(d->bias) % 16 == 0);
  if (d->flags & CVVAE_CONV_X_SHARED) CVVAE_CHECK_ARG(x.B == 1, "conv: CVVAE_CONV_X_SHARED needs x.B == 1");
  else CVVAE_CHECK_ARG(y.B == x.B, "conv: batch mismatch");
  if (d->flags & CVVAE_CONV_W_PER_BATCH)
    CVVAE_CHECK_ARG(d->KT * d->KH * d->KW == 1 && p.up_time == 1 && !d->gn_stats, "conv: per-batch weights need a 1x1x1 problem");
  p.B = y.B;
  CVVAE_CHECK_ARG(y.C == (p.up_time == 2 ? d->Cout / 2 : d->Cout), "conv: y.C %d inconsistent with Cout %d / up_time %d",
                  y.C, d->Cout, p.up_time);
  p.vec_ok = (y.s_c == 1) && (y.s_w % 8 == 0) && (y.s_h % 8 == 0) && (y.s_t % 8 == 0) && (y.s_b % 8 == 0) &&
             (reinterpret_cast<uintptr_t>(y.ptr) % 16 == 0) &&
             (!d->residual || reinterpret_cast<uintptr_t>(d->residual) % 16 == 0) &&
             ((p.up_time == 2 ? d->Cout / 2 : d->Cout) % 8 == 0);

  if (d->flags & CVVAE_CONV_OUT_F32) {
    CVVAE_CHECK_ARG(!d->residual && p.up_time == 1, "conv: fp32 output excludes residual / up_time");
    p.vec_ok = (y.s_c == 1) && (y.s_w % 4 == 0) && (y.s_h % 4 == 0) && (y.s_t % 4 == 0) && (y.s_b % 4 == 0) &&
               (reinterpret_cast<uintptr_t>(y.ptr) % 16 == 0);
  }

  // ---- tiling
  int N_cta;
  if (p.Cout >= 256) N_cta = 256;
  else if (p.Cout > 64) N_cta = 128;
  else if (p.Cout > 32) N_cta = 64;
  else if (p.Cout > 16) N_cta = 32;
  else N_cta = 16;
  p.N_cta = N_cta;
  p.n_tiles_n = (p.Cout + N_cta - 1) / N_cta;
  p.NACC = (512 / N_cta) < 4 ? (512 / N_cta) : 4;
  p.flat = (p.H_out == 1 && d->KH == 1 && d->KW == 1 && d->sw == 1 && d->sh == 1 && x.H == 1) ? 1 : 0;
  if (d->flags & (CVVAE_CONV_W_PER_BATCH | CVVAE_CONV_X_SHARED))
    CVVAE_CHECK_ARG(p.flat, "conv: batched-GEMM flags need a flat problem (H == 1, 1x1x1, stride 1)");
  // persistent double-buffered kernel for the Cout == 128 layers: tiles of 256 positions (two 128-row sub-tiles)
  p.persist = (!p.flat && p.Cout == 128 && p.up_time == 1 && p.vec_ok &&
               !(d->flags & (CVVAE_CONV_BIAS_ALONG_M | CVVAE_CONV_OUT_F32)) && y.C % 32 == 0) ? 1 : 0;
  if (p.persist) p.NACC = 2;
  // wide slabs (one slab per (kt, channel block) for all KH x KW taps) for stride-1 spatial kernels, in the persistent
  // kernel and in the Cout >= 256 layers (non-persistent kernel, CTA pairs side by side along W)
  const bool wide_want = (p.persist || N_cta == 256) && !p.flat && d->sh == 1 && d->sw == 1 && d->KW > 1 && d->KW <= 3 &&
                         d->KH <= 3;
  p.cblocks = (p.Cin + 63) / 64;
  for (;;) {
  if (p.flat) {
    p.TW = 128; p.ROWS = 1; p.TH = 1;
    p.KHs = 1; p.n_hgroups = 1; p.slab_rows = p.NACC;
    p.tiles_w = (p.W_out + p.NACC * 128 - 1) / (p.NACC * 128);
    p.tiles_h = 1;
  } else {
    p.KHs = (d->sh == 1) ? d->KH : 1;
    p.n_hgroups = d->KH / p.KHs;
    long long best_cost = -1;
    int best_tw = 16;
    // CTA pairs (N_cta = 256) stack two tiles vertically: an odd tile count costs one whole padding tile per column of tiles
    const int cg_plan = N_cta == 256 ? 2 : 1;
    for (int tw = 8; tw <= 128; tw *= 2) {
      const int rows = 128 / tw;
      const int th = rows * p.NACC;
      if (tw * d->sw > 256 || (th + p.KHs - 1) * d->sh > 256) continue;
      const long long tiles_w = (p.W_out + tw - 1) / tw;
      long long subtiles_h = (p.H_out + rows - 1) / rows;
      long long tiles_h = (p.H_out + th - 1) / th;
      if (cg_plan == 2 && tiles_h >= 2 && (tiles_h & 1)) {
        tiles_h += 1;
        subtiles_h += p.NACC;
      }
      // MMA work ~ sub-tiles; slab traffic ~ (th + halo) rows per tile
      const long long cost = tiles_w * subtiles_h * 128 * 16 + tiles_w * tiles_h * (th + p.KHs - 1) * tw * 3;
      if (best_cost < 0 || cost < best_cost) {
        best_cost = cost;
        best_tw = tw;
      }
    }
    if (wide_want) best_tw = 8;   // one 8-row swizzle group per image row of the tile
    p.TW = best_tw;
    p.ROWS = 128 / p.TW;
    p.TH = p.ROWS * p.NACC;
    p.slab_rows = p.TH + p.KHs - 1;
    p.tiles_w = (p.W_out + p.TW - 1) / p.TW;
    p.tiles_h = (p.H_out + p.TH - 1) / p.TH;
  }
  // small problems (latent-resolution layers, single images, attention GEMMs): fewer accumulators per CTA = more CTAs.
  // The count is per SAMPLE so that the plan - hence every rounding - is independent of the batch size.
  const long long ctas_per_sample = 1ll * p.n_tiles_n * p.T_out * p.tiles_w * p.tiles_h;
  if (p.persist || p.NACC <= 1 || ctas_per_sample >= num_sms()) break;
  p.NACC /= 2;
  }
  p.slab_bytes = p.flat ? static_cast<uint32_t>(p.NACC) * 16384u : static_cast<uint32_t>(p.slab_rows * p.TW) * 128u;
  p.wide = 0;
  p.PW = p.TW;
  if (wide_want) {
    p.wide = 1;
    p.PW = 8 + d->KW - 1;
    p.slab_bytes = static_cast<uint32_t>(p.slab_rows * p.PW) * 128u;
  }
  p.slab_stride = (p.slab_bytes + 1023u) & ~1023u;
  // CTA pairs (cta_group::2) when there are at least two adjacent tiles to pair up.  Measured (tools/bench_conv.py): pairs
  // help the N_cta = 256 layers (half the weight bytes per CTA, up to +10 %) and cost 0-16 % on the N_cta = 128 layers,
  // so they are used for N_cta = 256 only
  p.pair_w = (p.wide && !p.persist) ? 1 : 0;   // wide slabs: 8-wide tiles, pair them along W (always plenty, never odd rows)
  const bool pair_ok = !p.flat && (p.pair_w ? p.tiles_w >= 2 : p.tiles_h >= 2);
  const int CG = (pair_ok && N_cta == 256) ? 2 : 1;
  p.tiles_hg = p.pair_w ? p.tiles_h : (p.tiles_h + CG - 1) / CG;
  p.tiles_wg = p.pair_w ? (p.tiles_w + CG - 1) / CG : p.tiles_w;
  p.b_bytes = static_cast<uint32_t>(N_cta / CG) * 128u;  // weight rows staged per CTA
  // the persistent kernel swaps the MMA operands: D = [128 channels][256 positions]
  p.idesc = p.persist ? ptx::umma_idesc_f16(d->dtype == CVVAE_BF16 ? 1 : 0, 128, 256)
                      : ptx::umma_idesc_f16(d->dtype == CVVAE_BF16 ? 1 : 0, 128 * CG, N_cta);

  // ---- shared memory budget: 227 KB - alignment slack - barriers
  const size_t budget = 232448 - 1024 - 1536 - (p.persist ? 32768 : 0);  // persistent kernel: own staging area
  int NB = 4;
  while (NB > 2 && static_cast<size_t>(NB) * p.b_bytes + 2ull * p.slab_stride > budget) --NB;
  size_t rest = budget - static_cast<size_t>(NB) * p.b_bytes;
  int NA = static_cast<int>(rest / p.slab_stride);
  if (p.wide && NA > 2) NA = 2;   // a wide slab lasts KH x KW weight tiles: two slots hide its load, the rest goes to weights
  if (NA > 4) NA = 4;
  CVVAE_CHECK_ARG(NA >= 2, "conv_tc: slab of %u bytes does not fit the shared-memory budget", p.slab_bytes);
  // spend what is left on more weight stages
  while (NB < 8 && static_cast<size_t>(NB + 1) * p.b_bytes + static_cast<size_t>(NA) * p.slab_stride <= budget) ++NB;
  p.NA = NA;
  p.NB = NB;
  const size_t smem = 1024 + static_cast<size_t>(NA) * p.slab_stride + static_cast<size_t>(NB) * p.b_bytes + 1536 +
                      (p.persist ? 32768 : 0);

  // ---- tensor maps
  CUtensorMap tmA, tmB;
  {
    cuuint64_t dims[5] = {(cuuint64_t)x.C, (cuuint64_t)x.W, (cuuint64_t)x.H, (cuuint64_t)x.T, (cuuint64_t)x.B};
    cuuint64_t strides[4] = {(cuuint64_t)x.s_w * 2, (cuuint64_t)x.s_h * 2, (cuuint64_t)x.s_t * 2, (cuuint64_t)x.s_b * 2};
    // degenerate dims may carry meaningless strides; TMA wants multiples of 16 and monotone-ish validity
    for (int i = 0; i < 4; ++i)
      if (dims[i + 1] == 1 && (strides[i] == 0 || strides[i] % 16)) strides[i] = (cuuint64_t)x.C * 2;
    cuuint32_t box[5], estr[5] = {1, (cuuint32_t)d->sw, (cuuint32_t)d->sh, 1, 1};
    box[0] = 64;
    if (p.flat) {
      box[1] = 128; box[2] = 1;
    } else {
      box[1] = (cuuint32_t)(p.wide ? p.PW : p.TW * d->sw);
      box[2] = (cuuint32_t)(p.slab_rows * d->sh);
    }
    box[3] = 1; box[4] = 1;
    if (!encode_map(&tmA, x.ptr, 5, dims, strides, box, estr)) return CVVAE_E_CUDA;
  }
  {
    const int taps = (d->flags & CVVAE_CONV_W_PER_BATCH) ? x.B > y.B ? x.B : y.B : d->KT * d->KH * d->KW;
    cuuint64_t dims[3] = {(cuuint64_t)p.Cin, (cuuint64_t)p.Cout, (cuuint64_t)taps};
    const cuuint64_t wld = d->w_ld ? (cuuint64_t)d->w_ld : (cuuint64_t)p.Cin;
    cuuint64_t strides[2] = {wld * 2, wld * p.Cout * 2};
    cuuint32_t box[3] = {64, (cuuint32_t)(N_cta / CG), 1}, estr[3] = {1, 1, 1};
    if (!encode_map(&tmB, d->w, 3, dims, strides, box, estr)) return CVVAE_E_CUDA;
  }

  // ---- fused 1x1 shortcut: a second input tensor (same positions as the output) and a [Cout][Cin2] matrix
  CUtensorMap tmA2 = tmA, tmB2 = tmB;
  p.Cin2 = 0;
  p.cblocks2 = 0;
  p.sc_off16 = 0;
  if (d->w2) {
    const cvvae_tensor5& x2 = d->x2;
    CVVAE_CHECK_ARG(tensor_ok(&x2) && x2.B == y.B && x2.T == y.T && x2.H == y.H && x2.W == y.W,
                    "conv: fused shortcut input must have the output's [B,T,H,W] extents");
    CVVAE_CHECK_ARG(x2.s_c == 1 && x2.C % 8 == 0 && !(x2.s_w % 8) && !(x2.s_h % 8) && !(x2.s_t % 8) && !(x2.s_b % 8) &&
                        reinterpret_cast<uintptr_t>(x2.ptr) % 16 == 0 && reinterpret_cast<uintptr_t>(d->w2) % 16 == 0,
                    "conv: fused shortcut operands must be 16-byte aligned channels-last views with C %% 8 == 0");
    CVVAE_CHECK_ARG(!p.flat && p.up_time == 1 && d->st == 1 && d->sh == 1 && d->sw == 1 && !d->residual &&
                        !(d->flags & (CVVAE_CONV_BIAS_ALONG_M | CVVAE_CONV_OUT_F32 | CVVAE_CONV_W_PER_BATCH | CVVAE_CONV_X_SHARED)),
                    "conv: a fused shortcut needs a stride-1 spatial convolution without residual / interleave");
    CVVAE_CHECK_ARG(-d->off_h >= 0 && -d->off_h < d->KH && -d->off_w >= 0 && -d->off_w < d->KW && d->off_t <= 0 && -d->off_t < d->KT,
                    "conv: fused shortcut needs the centre tap inside the kernel window");
    p.Cin2 = x2.C;
    p.cblocks2 = (x2.C + 63) / 64;
    if (p.wide) p.sc_off16 = static_cast<uint32_t>((-d->off_h) * p.PW + (-d->off_w)) * 8u;
    {
      cuuint64_t dims[5] = {(cuuint64_t)x2.C, (cuuint64_t)x2.W, (cuuint64_t)x2.H, (cuuint64_t)x2.T, (cuuint64_t)x2.B};
      cuuint64_t strides[4] = {(cuuint64_t)x2.s_w * 2, (cuuint64_t)x2.s_h * 2, (cuuint64_t)x2.s_t * 2, (cuuint64_t)x2.s_b * 2};
      for (int i = 0; i < 4; ++i)
        if (dims[i + 1] == 1 && (strides[i] == 0 || strides[i] % 16)) strides[i] = (cuuint64_t)x2.C * 2;
      cuuint32_t box[5] = {64, (cuuint32_t)(p.wide ? p.PW : p.TW), (cuuint32_t)p.slab_rows, 1, 1}, estr[5] = {1, 1, 1, 1, 1};
      if (!encode_map(&tmA2, x2.ptr, 5, dims, strides, box, estr)) return CVVAE_E_CUDA;
    }
    {
      cuuint64_t dims[3] = {(cuuint64_t)x2.C, (cuuint64_t)p.Cout, 1};
      cuuint64_t strides[2] = {(cuuint64_t)x2.C * 2, (cuuint64_t)x2.C * p.Cout * 2};
      cuuint32_t box[3] = {64, (cuuint32_t)(N_cta / CG), 1}, estr[3] = {1, 1, 1};
      if (!encode_map(&tmB2, d->w2, 3, dims, strides, box, estr)) return CVVAE_E_CUDA;
    }
  }

  // ---- epilogue through shared memory + TMA store where the output is a plain channels-last 16-bit tensor.  The
  // persistent kernel's transposing epilogue stages [32 positions][32 channels] tiles (64-byte rows, no swizzle).
  CUtensorMap tmY = tmA, tmR = tmA;
  p.tma_epi = 0;
  {
    const int chalf = p.up_time == 2 ? p.Cout / 2 : p.Cout;
    const bool ok = p.vec_ok && !(d->flags & CVVAE_CONV_OUT_F32) && (p.up_time == 1 || chalf % 64 == 0) &&
                    (static_cast<size_t>(NA) * p.slab_stride >= 65536);
    if (ok) {
      p.box_w = p.flat ? 32 : (p.TW < 32 ? p.TW : 32);
      cuuint64_t dims[5] = {(cuuint64_t)y.C, (cuuint64_t)y.W, (cuuint64_t)y.H, (cuuint64_t)y.T, (cuuint64_t)y.B};
      cuuint64_t strides[4] = {(cuuint64_t)y.s_w * 2, (cuuint64_t)y.s_h * 2, (cuuint64_t)y.s_t * 2, (cuuint64_t)y.s_b * 2};
      for (int i = 0; i < 4; ++i)
        if (dims[i + 1] == 1 && (strides[i] == 0 || strides[i] % 16)) strides[i] = (cuuint64_t)y.C * 2;
      cuuint32_t box[5] = {p.persist ? 32u : 64u, (cuuint32_t)p.box_w, (cuuint32_t)(32 / p.box_w), 1, 1}, estr[5] = {1, 1, 1, 1, 1};
      const CUtensorMapSwizzle swz = p.persist ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B;
      if (!encode_map(&tmY, y.ptr, 5, dims, strides, box, estr, swz)) return CVVAE_E_CUDA;
      if (d->residual && !encode_map(&tmR, d->residual, 5, dims, strides, box, estr, swz)) return CVVAE_E_CUDA;
      p.tma_epi = 1;
    }
  }
  // a persistent plan always qualifies: its output is 16-byte aligned channels-last, and its slabs hold at least
  // 256 positions x 128 B with NA >= 2
  CVVAE_CHECK_ARG(!p.persist || p.tma_epi, "conv_tc: internal: persistent plan without the TMA epilogue");
  // fused GroupNorm statistics need the TMA epilogue, power-of-two channels per group and one sample per CTA index
  p.gn_stats = nullptr;
  if (d->gn_stats) {
    const int cpg = d->gn_groups > 0 ? y.C / d->gn_groups : 0;
    const bool ok = p.tma_epi && d->gn_groups > 0 && d->gn_groups <= 64 && y.C % d->gn_groups == 0 && cpg >= 1 &&
                    (cpg & (cpg - 1)) == 0 && (cpg <= 64 ? 64 % cpg == 0 : cpg % 64 == 0);
    if (!ok) {
      set_error("conv_tc: fused GroupNorm statistics unsupported for this output (C=%d groups=%d tma_epi=%d)", y.C,
                d->gn_groups, p.tma_epi);
      return CVVAE_E_UNSUPPORTED;
    }
    p.gn_stats = d->gn_stats;
    p.gn_groups = d->gn_groups;
    p.gn_cpg = cpg;
  }

  if (p.cblocks2 && p.persist && !p.wide) {
    set_error("conv_tc: fused shortcut unsupported on the persistent kernel without wide slabs");
    return CVVAE_E_UNSUPPORTED;
  }
  const long long grid = 1ll * p.n_tiles_n * p.T_out * p.tiles_wg * p.tiles_hg * p.B * CG;
  CVVAE_CHECK_ARG(grid > 0 && grid < (1ll << 31), "conv_tc: grid size %lld out of range", grid);
  CVVAE_DISPATCH_DTYPE(d->dtype, {
    static PerDeviceOnce attr_set;   // the > 48 KB shared-memory opt-in is per device
    if (attr_set.need()) {
      CVVAE_CUDA(cudaFuncSetAttribute(conv_tc_kernel<DT, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
      CVVAE_CUDA(cudaFuncSetAttribute(conv_tc_kernel<DT, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
      CVVAE_CUDA(cudaFuncSetAttribute(conv_tc_psw_kernel<DT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
      attr_set.mark();
    }
    if (p.persist) {
      p.n_tiles = static_cast<int>(grid);
      const int ctas = p.n_tiles < num_sms() ? p.n_tiles : num_sms();
      conv_tc_psw_kernel<DT><<<ctas, kPersistThreads, smem, stream>>>(tmA, tmB, tmY, tmR, tmA2, tmB2, p);
    } else if (CG == 2) {
      cudaLaunchConfig_t cfg{};
      cfg.gridDim = dim3(static_cast<unsigned>(grid));
      cfg.blockDim = dim3(kThreads);
      cfg.dynamicSmemBytes = smem;
      cfg.stream = stream;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      CVVAE_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<DT, 2>, tmA, tmB, tmY, tmR, tmA2, tmB2, p));
    } else {
      conv_tc_kernel<DT, 1><<<static_cast<unsigned>(grid), kThreads, smem, stream>>>(tmA, tmB, tmY, tmR, tmA2, tmB2, p);
    }
  });
  CVVAE_LAUNCH_CHECK();
  return CVVAE_OK;
}

}  // namespace cvvae

extern "C" int cvvae_conv_tc_set_trace(void* device_buf, int32_t n_ctas) {
  cvvae::conv_tc_set_trace(static_cast<unsigned long long*>(device_buf), device_buf ? n_ctas : 0);
  return CVVAE_OK;
}

extern "C" int cvvae_conv3d_tc(const cvvae_conv_desc* d, void* stream) {
  CVVAE_CHECK_ARG(d && cvvae::tensor_ok(&d->x) && cvvae::tensor_ok(&d->y) && d->w, "cvvae_conv3d_tc: null argument");
  return cvvae::conv_tc_launch(d, static_cast<cudaStream_t>(stream));
}
