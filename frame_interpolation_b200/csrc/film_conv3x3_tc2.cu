// CTA-pair (tcgen05 cta_group::2) variant of the persistent 3x3 convolution (sm_100a).
//
// Two CTAs of a (2,1,1) cluster -- the two SMs of a TPC -- share every MMA: M = 256 output pixels
// (two vertically adjacent 16x8 tiles, one per CTA), N = BN.  Each CTA TMA-loads ITS OWN
// activation boxes and only HALF of the rows of every weight tap, so the weight bytes pulled from
// L2 per MAC halve (the N <= 128 layers are L2-bandwidth bound on re-streamed weights), and one
// instruction covers twice the work (the M=128 SS-mode instruction floor is ~72 cycles whatever N is).
//
// Protocol (CUTLASS PipelineTmaUmmaAsync 2-SM pattern):
//   * "full" barriers live in the LEADER (cluster rank 0): the leader arms expect_tx for the bytes of
//     BOTH CTAs; both producers issue cp.async.bulk.tensor...cta_group::2 whose complete_tx goes to
//     the leader's barrier.
//   * The leader's MMA warp issues tcgen05.mma.cta_group::2 and releases stages with
//     tcgen05.commit...multicast::cluster (mask 0b11): the same "empty" barrier offset in both CTAs.
//   * Accumulators: each CTA's TMEM holds its 128 rows; double-buffered.  t_full is multicast by the
//     leader; t_empty lives in the leader and collects the epilogue warps of both CTAs (the peer
//     arrives remotely through its shared::cluster address).
//   * 3-pass split product.  BN >= 128: unfused, 3 instructions per k-step (N = BN), each CTA loads
//     half of the W_hi rows and half of the W_lo rows (weight bytes per CTA x0.5).
//     BN <= 64 (instruction-bound): fused, 2 instructions per k-step.  The B operand of a
//     cta_group::2 MMA is split by rows across the pair, so for  A_hi x [W_hi ; W_lo]  (N = 2*BN) the
//     leader holds ALL of W_hi and the peer ALL of W_lo at the same smem offset; for  A_lo x W_hi
//     (N = BN) each CTA additionally holds its half of W_hi (weight bytes per CTA x0.75).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "film_conv.h"
#include "film_tc_ptx.cuh"

namespace film {
namespace {
using namespace tc;

constexpr int kEpiWarps = 8;
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kTileH = 16, kTileW = 8;
constexpr int kMaxRing = 8;
constexpr int kSmemLimit = 227 * 1024;
constexpr int kBarBytes = 8 * (4 * kMaxRing + 4);
constexpr int kFixedBytes = kBarBytes + 16 + 512 * 4 /*bias*/ + 64 /*src table*/ + 1024 /*align*/ + 64;

__host__ __device__ constexpr int a_stage_bytes2(int kc) { return 2 * (kTileH + 2) * kTileW * kc * 2; }
// Wide-halo mode: one box (KC ch, 10 px, 18 rows) per plane and chunk serves all nine taps.
constexpr int kHaloW = kTileW + 2;
__host__ __device__ constexpr int halo_box_bytes(int kc) { return (kTileH + 2) * kHaloW * kc * 2; }  // 23,040 (KC 64)
__host__ __device__ constexpr int halo_plane_bytes(int kc) { return (halo_box_bytes(kc) + 1023) & ~1023; }  // 1 KiB-aligned planes
__host__ __device__ constexpr int halo_stage_bytes(int kc) { return 2 * halo_plane_bytes(kc); }  // 46 KiB vs 3 x 36 KiB
// `planes` = 2 (hi + lo) or 1 (single-pass layers load the hi planes only)
__host__ __device__ constexpr int a_stage_bytes2h(int kc, int halo, int planes = 2) {
  return (halo ? halo_stage_bytes(kc) : a_stage_bytes2(kc)) / 2 * planes;
}
// bytes of one weight tap per CTA: unfused = half of W_hi + half of W_lo; fused (BN <= 64) = one full
// plane (W_hi in the leader, W_lo in the peer) + this CTA's half of W_hi
__host__ __device__ constexpr bool pair_fused(int bn) { return bn <= 64; }
// single-pass: this CTA's half of the W_hi rows only
__host__ __device__ constexpr int w_half_tap_bytes(int bn, int kc, int planes = 2) {
  return planes == 1 ? (bn / 2) * kc * 2 : pair_fused(bn) ? (bn + bn / 2) * kc * 2 : (bn / 2) * kc * 2 * 2;
}

template <int BN, int KC>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
    k_conv3x3_tc2(const ConvProblem* __restrict__ prob) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int kAPlane = (kTileH + 2) * kTileW * KC * 2;
  constexpr int kAStage = 2 * kAPlane;
  constexpr bool kFused = pair_fused(BN);
  constexpr int kWHalf = (BN / 2) * KC * 2;   // one plane, half of the rows
  constexpr int kWFull = BN * KC * 2;         // one plane, all rows of the N tile
  constexpr int kRowStep = kTileW * KC * 2;
  constexpr int kHaloBox = halo_box_bytes(KC), kHaloPlane = halo_plane_bytes(KC), kHaloStage = halo_stage_bytes(KC);
  constexpr uint32_t kAccCols = kFused ? 2 * BN : BN;
  // double-buffered accumulators; N tiles <= 128 reserve two SETS per buffer for the dual-item mode
  constexpr uint32_t kTmemCols = (BN <= 128) ? 4 * kAccCols : 2 * kAccCols;
  static_assert(kTmemCols >= 32 && kTmemCols <= 512, "TMEM budget");

  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;

  const int NA = prob->v2_na, NW = prob->v2_nw;
  const bool resident = prob->v2_resident != 0;
  const bool halo = prob->halo != 0;
  const bool one = prob->passes == 1;   // single-pass product A_hi x W_hi: hi planes only
  const int planes = one ? 1 : 2;
  const int kWTap = w_half_tap_bytes(BN, KC, planes);
  const int lo_plane = halo ? kHaloPlane : kAPlane;
  const int a_stage = planes * lo_plane;
  (void)kAStage; (void)kHaloStage;
  const int nsrc = prob->nsrc;
  const int tiles_x = prob->tiles_x, tiles_y = prob->tiles_y;
  const int pairs_y = (tiles_y + 1) / 2;
  const int pairs_per_img = pairs_y * tiles_x;
  const int cout = prob->cout;
  const int n_nt = (cout + BN - 1) / BN;
  const int nitems = prob->B * pairs_per_img * n_nt;   // work items: (tile pair, N tile), N fastest
  const int item0 = blockIdx.x >> 1, item_step = gridDim.x >> 1;
  // dual-item mode (host guarantees: streamed weights, wide halo, one N tile, BN <= 128, NA >= 2): a "super item" is
  // two consecutive spatial items sharing every weight tap
  const bool dual = prob->dual != 0;
  const int sub_n = dual ? 2 : 1;
  const int nsuper = dual ? (nitems + 1) / 2 : nitems;
  int nkb = 0;
  for (int s = 0; s < nsrc; ++s) nkb += prob->src[s].nchunk * 9;

  const FastDiv div_nt(n_nt, nitems), div_img(pairs_per_img, nitems), div_tx(tiles_x, nitems);   // item decode

  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* gen_base = smem_raw + (base - raw);
  const uint32_t a_base = base;
  const uint32_t w_base = a_base + (uint32_t)NA * a_stage;
  const uint32_t w_bytes = resident ? (uint32_t)nkb * kWTap : (uint32_t)NW * kWTap;
  const uint32_t tail = w_base + w_bytes;
  const uint32_t tail_off = (uint32_t)NA * a_stage + w_bytes;
  // barrier k at tail + 8k: a_full[0..7], a_empty[8..15], w_full[16..23], w_empty[24..31], t_full[32,33], t_empty[34,35]
  auto a_full = [&](int s) { return tail + 8u * s; };
  auto a_empty = [&](int s) { return tail + 8u * (kMaxRing + s); };
  auto w_full = [&](int s) { return tail + 8u * (2 * kMaxRing + s); };
  auto w_empty = [&](int s) { return tail + 8u * (3 * kMaxRing + s); };
  auto t_full = [&](int s) { return tail + 8u * (4 * kMaxRing + s); };
  auto t_empty = [&](int s) { return tail + 8u * (4 * kMaxRing + 2 + s); };
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(gen_base + tail_off + kBarBytes);
  float* bias_smem = reinterpret_cast<float*>(gen_base + tail_off + kBarBytes + 16);
  int* src_tab = reinterpret_cast<int*>(gen_base + tail_off + kBarBytes + 16 + 512 * 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kMaxRing; ++s) {
      mbar_init(a_full(s), 1);
      mbar_init(a_empty(s), 1);
      mbar_init(w_full(s), 1);
      mbar_init(w_empty(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(t_full(s), 1);
      mbar_init(t_empty(s), 2 * kEpiWarps);  // epilogue warps of BOTH CTAs (leader's copy is the one used)
    }
    for (int s = 0; s < kMaxSrc; ++s) {
      src_tab[2 * s] = s < nsrc ? prob->src[s].nchunk : 0;
      src_tab[2 * s + 1] = s < nsrc ? prob->src[s].c_off : 0;
      src_tab[2 * kMaxSrc + s] = s < nsrc ? prob->src[s].ksteps : 0;
      src_tab[3 * kMaxSrc + s] = s < nsrc ? prob->src[s].bswap : 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc_2sm(smem_u32(tmem_ptr_smem), kTmemCols);
  if (warp >= 2)
    for (int i = threadIdx.x - 64; i < n_nt * BN; i += 32 * kEpiWarps) bias_smem[i] = (i < cout) ? prob->bias[i] : 0.f;
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ============================ TMA producer (both CTAs) ============================
    const CUtensorMap* tm_w_hi = &prob->tm_w_hi_half;
    const CUtensorMap* tm_w_lo = &prob->tm_w_lo_half;
    const CUtensorMap* tm_w_full_hi = &prob->tm_w_hi;   // fused form: full-height boxes [BN x KC]
    const CUtensorMap* tm_w_full_lo = &prob->tm_w_lo;
    const int n_half = (int)rank * (BN / 2);
    if (resident) {
      if (elect_one()) {
        const uint32_t bar = map_to_cta(w_full(0), 0);
        if (leader) mbar_expect_tx(w_full(0), 2u * (uint32_t)nkb * kWTap);   // both CTAs' halves
        for (int kb = 0; kb < nkb; ++kb) {
          if (one) {
            tma_load_2d_2sm(w_base + kb * kWTap, tm_w_hi, bar, kb * KC, n_half);
          } else if constexpr (kFused) {
            tma_load_2d_2sm(w_base + kb * kWTap, leader ? tm_w_full_hi : tm_w_full_lo, bar, kb * KC, 0);
            tma_load_2d_2sm(w_base + kb * kWTap + kWFull, tm_w_hi, bar, kb * KC, n_half);
          } else {
            tma_load_2d_2sm(w_base + kb * kWTap, tm_w_hi, bar, kb * KC, n_half);
            tma_load_2d_2sm(w_base + kb * kWTap + kWHalf, tm_w_lo, bar, kb * KC, n_half);
          }
        }
      }
      __syncwarp();
    }
    RingPos ra, rw;   // activation / weight ring positions
    if (dual) {
      // chunk by chunk: the halo boxes of BOTH sub-items, then the nine weight taps they share
      for (int sit = item0; sit < nsuper; sit += item_step) {
        const int nsub = (2 * sit + 1 < nitems) ? 2 : 1;
        int kb = 0;
        for (int s = 0; s < nsrc; ++s) {
          const int nchunk = src_tab[2 * s], c_off = src_tab[2 * s + 1];
          const bool swap = src_tab[3 * kMaxSrc + s] != 0;
          const CUtensorMap* tm_hi = &prob->tm_a_hi[s];
          const CUtensorMap* tm_lo = &prob->tm_a_lo[s];
          for (int ch = 0; ch < nchunk; ++ch) {
            for (int sub = 0; sub < nsub; ++sub) {
              const int sp = 2 * sit + sub;   // n_nt == 1
              int b, rem, ty, tx;
              div_img.divmod(sp, b, rem);
              div_tx.divmod(rem, ty, tx);
              const int y0 = (2 * ty + (int)rank) * kTileH, x0 = tx * kTileW;
              const int bs = swap ? prob->B - 1 - b : b;
              const int st = ra.stage;
              mbar_wait(a_empty(st), ra.phase ^ 1u);
              if (elect_one()) {
                const uint32_t sa = a_base + st * a_stage;
                const uint32_t bar = map_to_cta(a_full(st), 0);
                if (leader) mbar_expect_tx(a_full(st), 2u * planes * kHaloBox);
                tma_load_4d_2sm(sa, tm_hi, bar, c_off + ch * KC, x0 - 1, y0 - 1, bs);
                if (!one) tma_load_4d_2sm(sa + kHaloPlane, tm_lo, bar, c_off + ch * KC, x0 - 1, y0 - 1, bs);
              }
              __syncwarp();
              ra.advance(NA);
            }
            for (int t = 0; t < 9; ++t, ++kb) {
              const int ws = rw.stage;
              mbar_wait(w_empty(ws), rw.phase ^ 1u);
              if (elect_one()) {
                const uint32_t sw = w_base + ws * kWTap;
                const uint32_t bar = map_to_cta(w_full(ws), 0);
                if (leader) mbar_expect_tx(w_full(ws), 2u * kWTap);
                if (one) {
                  tma_load_2d_2sm(sw, tm_w_hi, bar, kb * KC, n_half);
                } else if constexpr (kFused) {
                  tma_load_2d_2sm(sw, leader ? tm_w_full_hi : tm_w_full_lo, bar, kb * KC, 0);
                  tma_load_2d_2sm(sw + kWFull, tm_w_hi, bar, kb * KC, n_half);
                } else {
                  tma_load_2d_2sm(sw, tm_w_hi, bar, kb * KC, n_half);
                  tma_load_2d_2sm(sw + kWHalf, tm_w_lo, bar, kb * KC, n_half);
                }
              }
              __syncwarp();
              rw.advance(NW);
            }
          }
        }
      }
    } else {
    for (int item = item0; item < nitems; item += item_step) {
      int sp, nti, b, rem, ty, tx;
      div_nt.divmod(item, sp, nti);
      div_img.divmod(sp, b, rem);
      div_tx.divmod(rem, ty, tx);
      const int n0 = nti * BN;
      const int y0 = (2 * ty + (int)rank) * kTileH, x0 = tx * kTileW;
      int kb = 0;
      for (int s = 0; s < nsrc; ++s) {
        const int nchunk = src_tab[2 * s], c_off = src_tab[2 * s + 1];
        const int bs = src_tab[3 * kMaxSrc + s] ? prob->B - 1 - b : b;
        const CUtensorMap* tm_hi = &prob->tm_a_hi[s];
        const CUtensorMap* tm_lo = &prob->tm_a_lo[s];
        for (int ch = 0; ch < nchunk; ++ch) {
          // activation stages of this chunk: one wide halo box, or three dx-shifted boxes
          const int nst = halo ? 1 : 3;
          for (int dx = 0; dx < nst; ++dx) {
            const int st = ra.stage;
            mbar_wait(a_empty(st), ra.phase ^ 1u);
            if (elect_one()) {
              const uint32_t sa = a_base + st * a_stage;
              const uint32_t bar = map_to_cta(a_full(st), 0);
              if (halo) {
                if (leader) mbar_expect_tx(a_full(st), 2u * planes * kHaloBox);   // planes x two CTAs
                tma_load_4d_2sm(sa, tm_hi, bar, c_off + ch * KC, x0 - 1, y0 - 1, bs);
                if (!one) tma_load_4d_2sm(sa + kHaloPlane, tm_lo, bar, c_off + ch * KC, x0 - 1, y0 - 1, bs);
              } else {
                if (leader) mbar_expect_tx(a_full(st), 2u * planes * kAPlane);
                tma_load_4d_2sm(sa, tm_hi, bar, c_off + ch * KC, x0 + dx - 1, y0 - 1, bs);
                if (!one) tma_load_4d_2sm(sa + kAPlane, tm_lo, bar, c_off + ch * KC, x0 + dx - 1, y0 - 1, bs);
              }
            }
            __syncwarp();
            ra.advance(NA);
            if (!resident) {
              const int ntap = halo ? 9 : 3;   // weight taps consumed against this activation stage
              for (int t = 0; t < ntap; ++t, ++kb) {
                const int ws = rw.stage;
                mbar_wait(w_empty(ws), rw.phase ^ 1u);
                if (elect_one()) {
                  const uint32_t sw = w_base + ws * kWTap;
                  const uint32_t bar = map_to_cta(w_full(ws), 0);
                  if (leader) mbar_expect_tx(w_full(ws), 2u * kWTap);
                  if (one) {
                    tma_load_2d_2sm(sw, tm_w_hi, bar, kb * KC, n0 + n_half);
                  } else if constexpr (kFused) {
                    tma_load_2d_2sm(sw, leader ? tm_w_full_hi : tm_w_full_lo, bar, kb * KC, n0);
                    tma_load_2d_2sm(sw + kWFull, tm_w_hi, bar, kb * KC, n0 + n_half);
                  } else {
                    tma_load_2d_2sm(sw, tm_w_hi, bar, kb * KC, n0 + n_half);
                    tma_load_2d_2sm(sw + kWHalf, tm_w_lo, bar, kb * KC, n0 + n_half);
                  }
                }
                __syncwarp();
                rw.advance(NW);
              }
            }
          }
        }
      }
    }
    }  // one item per weight pass
  } else if (warp == 1) {
    // ============================ MMA issuer (leader CTA only) ============================
    if (leader) {
      const uint32_t idesc = make_idesc_m<BN, 256>();
      const uint32_t idesc2 = make_idesc_m<(kFused ? 2 * BN : BN), 256>();
      if (resident) {
        mbar_wait(w_full(0), 0);
        tc_fence_after();
      }
      // The item loop is instantiated per (partial sources, wide halo): see film_conv3x3_tc.cu.  Halo mode:
      // one activation stage per chunk carries all nine taps; tap t = 3*dx + dy (the K order of the packed
      // weights) reads the box at pixel offset (dy, dx), i.e. byte offset (dy * 10 + dx) * 128, with 8-row
      // groups (one tile row each) 1280 B apart.
      bool any_partial = false;
      for (int s = 0; s < kMaxSrc; ++s) any_partial |= src_tab[2 * s] > 0 && src_tab[2 * kMaxSrc + s] < KC / 16;
      auto run_items = [&](auto partial_tag, auto halo_tag, auto one_tag, auto res_tag) {
        constexpr bool kPartial = decltype(partial_tag)::value;
        constexpr bool kHalo = decltype(halo_tag)::value;
        constexpr bool kOne = decltype(one_tag)::value;   // single-pass product
        constexpr bool kRes = decltype(res_tag)::value;   // weights resident: one elected lane issues a whole stage
        constexpr int kWTapC = w_half_tap_bytes(BN, KC, kOne ? 1 : 2);
        constexpr int kStageTaps = kHalo ? 9 : 3;       // taps served by one activation stage
        constexpr int kSrcStages = kHalo ? 1 : 3;       // activation stages per chunk
        constexpr int kLoPlane = kHalo ? kHaloPlane : kAPlane;
        constexpr int kStageBytes = (kOne ? 1 : 2) * kLoPlane;
        const int nab = nkb / kStageTaps;
        RingPos ra, rw;   // activation / weight ring positions
        uint32_t it = 0;
        for (int item = item0; item < nitems; item += item_step, ++it) {
          const uint32_t acc = it & 1u;
          mbar_wait(t_empty(acc), ((it >> 1) & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * kAccCols;
          int kb = 0;
          [[maybe_unused]] int src_i = 0, src_left = src_tab[0] * kSrcStages;  // stages left in the current source
          for (int ab = 0; ab < nab; ++ab) {
            [[maybe_unused]] int ksteps = KC / 16;
            if constexpr (kPartial) {  // all-zero tail k-steps are skipped (exact)
              while (src_left == 0) {
                ++src_i;
                src_left = src_tab[2 * src_i] * kSrcStages;
              }
              --src_left;
              ksteps = src_tab[2 * kMaxSrc + src_i];
            }
            const int st = ra.stage;
            mbar_wait(a_full(st), ra.phase);
            tc_fence_after();
            const uint32_t sa = a_base + st * kStageBytes;
            if constexpr (kRes) {
              // resident weights: straight-line issue of all taps of the stage (see film_conv3x3_tc.cu)
              if (elect_one()) {
                constexpr uint32_t kPx = KC * 2;
                const uint64_t a0 = kHalo ? make_desc_sbo<KC>(sa, kHaloW * kPx) : make_desc_kc<KC>(sa);
                const uint64_t w0 = make_desc_kc<KC>(w_base + kb * kWTapC);
                const uint32_t first = (kb == 0) ? 0u : 1u;
#pragma unroll
                for (int t = 0; t < kStageTaps; ++t) {
                  const uint64_t a_hi = a0 + (uint64_t)((kHalo ? ((t % 3) * kHaloW + t / 3) * kPx : t * kRowStep) >> 4);
                  const uint64_t a_lo = a_hi + (uint64_t)(kLoPlane >> 4);
                  const uint64_t wt = w0 + (uint64_t)((t * kWTapC) >> 4);
#pragma unroll
                  for (int k = 0; k < KC / 16; ++k) {
                    if (!kPartial || k < ksteps) {
                      const uint64_t adv = (uint64_t)(k * 32 >> 4);
                      const uint32_t accf = (t == 0 && k == 0) ? first : 1u;
                      if constexpr (kOne) {
                        umma_2sm(d_tmem, a_hi + adv, wt + adv, idesc, accf);          // halves of the W_hi rows
                      } else if constexpr (kFused) {
                        umma_2sm(d_tmem, a_hi + adv, wt + adv, idesc2, accf);         // X: W_hi (leader) / W_lo (peer)
                        umma_2sm(d_tmem, a_lo + adv, wt + (uint64_t)(kWFull >> 4) + adv, idesc, 1u);   // Y: halves of W_hi
                      } else {
                        umma_2sm(d_tmem, a_lo + adv, wt + adv, idesc, accf);
                        umma_2sm(d_tmem, a_hi + adv, wt + (uint64_t)(kWHalf >> 4) + adv, idesc, 1u);
                        umma_2sm(d_tmem, a_hi + adv, wt + adv, idesc, 1u);
                      }
                    }
                  }
                }
                umma_commit_2sm_mc(a_empty(st));
                if (ab == nab - 1) umma_commit_2sm_mc(t_full(acc));
              }
              __syncwarp();
              kb += kStageTaps;
            } else {
            for (int t = 0; t < kStageTaps; ++t, ++kb) {
              uint32_t sw;
              int ws = 0;
              if (resident) {
                sw = w_base + kb * kWTap;
              } else {
                ws = rw.stage;
                mbar_wait(w_full(ws), rw.phase);
                tc_fence_after();
                sw = w_base + ws * kWTap;
              }
              if (elect_one()) {
                uint64_t a_hi, a_lo;
                if constexpr (kHalo) {
                  constexpr uint32_t kPx = KC * 2;   // bytes of one pixel row of the box
                  const uint32_t off = (uint32_t)((t % 3) * kHaloW + t / 3) * kPx;
                  a_hi = make_desc_sbo<KC>(sa + off, kHaloW * kPx);
                  a_lo = make_desc_sbo<KC>(sa + kLoPlane + off, kHaloW * kPx);
                } else {
                  a_hi = make_desc_kc<KC>(sa + t * kRowStep);
                  a_lo = make_desc_kc<KC>(sa + kLoPlane + t * kRowStep);
                }
                const uint32_t first = (kb == 0) ? 0u : 1u;
                if constexpr (kOne) {
                  // each CTA holds its half of the W_hi rows at `sw`
                  const uint64_t w_h = make_desc_kc<KC>(sw);
#pragma unroll
                  for (int k = 0; k < KC / 16; ++k) {
                    if constexpr (kPartial) {
                      if (k >= ksteps) break;
                    }
                    const uint64_t adv = (uint64_t)(k * 32 >> 4);
                    umma_2sm(d_tmem, a_hi + adv, w_h + adv, idesc, k == 0 ? first : 1u);
                  }
                } else if constexpr (kFused) {
                  // region X (leader: W_hi, peer: W_lo) is the 2*BN-row operand; region Y = halves of W_hi
                  const uint64_t w_x = make_desc_kc<KC>(sw), w_y = make_desc_kc<KC>(sw + kWFull);
#pragma unroll
                  for (int k = 0; k < KC / 16; ++k) {
                    if constexpr (kPartial) {
                      if (k >= ksteps) break;
                    }
                    const uint64_t adv = (uint64_t)(k * 32 >> 4);
                    umma_2sm(d_tmem, a_hi + adv, w_x + adv, idesc2, k == 0 ? first : 1u);
                    umma_2sm(d_tmem, a_lo + adv, w_y + adv, idesc, 1u);
                  }
                } else {
                  const uint64_t w_hi = make_desc_kc<KC>(sw), w_lo = make_desc_kc<KC>(sw + kWHalf);
#pragma unroll
                  for (int k = 0; k < KC / 16; ++k) {
                    if constexpr (kPartial) {
                      if (k >= ksteps) break;
                    }
                    const uint64_t adv = (uint64_t)(k * 32 >> 4);
                    umma_2sm(d_tmem, a_lo + adv, w_hi + adv, idesc, k == 0 ? first : 1u);
                    umma_2sm(d_tmem, a_hi + adv, w_lo + adv, idesc, 1u);
                    umma_2sm(d_tmem, a_hi + adv, w_hi + adv, idesc, 1u);
                  }
                }
                if (!resident) umma_commit_2sm_mc(w_empty(ws));
                if (t == kStageTaps - 1) umma_commit_2sm_mc(a_empty(st));
                if (t == kStageTaps - 1 && ab == nab - 1) umma_commit_2sm_mc(t_full(acc));
              }
              __syncwarp();
              if (!resident) rw.advance(NW);
            }
            }  // per-tap issue loop
            ra.advance(NA);
          }
        }
      };
      // dual-item mode: per chunk wait for the halo boxes of both sub-items, then every weight tap is used twice
      auto run_items_dual = [&](auto partial_tag, auto one_tag) {
        constexpr bool kPartial = decltype(partial_tag)::value;
        constexpr bool kOne = decltype(one_tag)::value;
        constexpr int kStageBytes = (kOne ? 1 : 2) * kHaloPlane;
        constexpr uint32_t kPx = KC * 2;
        const int nab = nkb / 9;
        RingPos ra, rw;
        uint32_t it = 0;
        for (int sit = item0; sit < nsuper; sit += item_step, ++it) {
          const int nsub = (2 * sit + 1 < nitems) ? 2 : 1;
          const uint32_t acc = it & 1u;
          mbar_wait(t_empty(acc), ((it >> 1) & 1u) ^ 1u);
          tc_fence_after();
          int kb = 0;
          [[maybe_unused]] int src_i = 0, src_left = src_tab[0];
          for (int ab = 0; ab < nab; ++ab) {
            [[maybe_unused]] int ksteps = KC / 16;
            if constexpr (kPartial) {
              while (src_left == 0) {
                ++src_i;
                src_left = src_tab[2 * src_i];
              }
              --src_left;
              ksteps = src_tab[2 * kMaxSrc + src_i];
            }
            int st2[2] = {0, 0};
            for (int sub = 0; sub < nsub; ++sub) {
              st2[sub] = ra.stage;
              mbar_wait(a_full(ra.stage), ra.phase);
              ra.advance(NA);
            }
            tc_fence_after();
            for (int t = 0; t < 9; ++t, ++kb) {
              const int ws = rw.stage;
              mbar_wait(w_full(ws), rw.phase);
              tc_fence_after();
              const uint32_t sw = w_base + ws * kWTap;
              if (elect_one()) {
                const uint32_t off = (uint32_t)((t % 3) * kHaloW + t / 3) * kPx;
                const uint32_t first = (kb == 0) ? 0u : 1u;
                for (int sub = 0; sub < nsub; ++sub) {
                  const uint32_t sa = a_base + st2[sub] * kStageBytes;
                  const uint32_t d_tmem = tmem_base + (acc * 2 + sub) * kAccCols;
                  const uint64_t a_hi = make_desc_sbo<KC>(sa + off, kHaloW * kPx);
                  const uint64_t a_lo = make_desc_sbo<KC>(sa + kHaloPlane + off, kHaloW * kPx);
#pragma unroll
                  for (int k = 0; k < KC / 16; ++k) {
                    if (!kPartial || k < ksteps) {
                      const uint64_t adv = (uint64_t)(k * 32 >> 4);
                      const uint32_t accf = k == 0 ? first : 1u;
                      if constexpr (kOne) {
                        umma_2sm(d_tmem, a_hi + adv, make_desc_kc<KC>(sw) + adv, idesc, accf);
                      } else if constexpr (kFused) {
                        umma_2sm(d_tmem, a_hi + adv, make_desc_kc<KC>(sw) + adv, idesc2, accf);
                        umma_2sm(d_tmem, a_lo + adv, make_desc_kc<KC>(sw + kWFull) + adv, idesc, 1u);
                      } else {
                        umma_2sm(d_tmem, a_lo + adv, make_desc_kc<KC>(sw) + adv, idesc, accf);
                        umma_2sm(d_tmem, a_hi + adv, make_desc_kc<KC>(sw + kWHalf) + adv, idesc, 1u);
                        umma_2sm(d_tmem, a_hi + adv, make_desc_kc<KC>(sw) + adv, idesc, 1u);
                      }
                    }
                  }
                }
                umma_commit_2sm_mc(w_empty(ws));
                if (t == 8) {
                  for (int sub = 0; sub < nsub; ++sub) umma_commit_2sm_mc(a_empty(st2[sub]));
                  if (ab == nab - 1) umma_commit_2sm_mc(t_full(acc));
                }
              }
              __syncwarp();
              rw.advance(NW);
            }
          }
        }
      };
      auto run_pass = [&](auto one_tag, auto res_tag) {
        if (halo) {
          if (any_partial) run_items(std::true_type{}, std::true_type{}, one_tag, res_tag);
          else run_items(std::false_type{}, std::true_type{}, one_tag, res_tag);
        } else {
          if (any_partial) run_items(std::true_type{}, std::false_type{}, one_tag, res_tag);
          else run_items(std::false_type{}, std::false_type{}, one_tag, res_tag);
        }
      };
      if (dual) {
        if (one) {
          if (any_partial) run_items_dual(std::true_type{}, std::true_type{});
          else run_items_dual(std::false_type{}, std::true_type{});
        } else {
          if (any_partial) run_items_dual(std::true_type{}, std::false_type{});
          else run_items_dual(std::false_type{}, std::false_type{});
        }
      } else if (resident && prob->straight) {
        if (one) run_pass(std::true_type{}, std::true_type{});
        else run_pass(std::false_type{}, std::true_type{});
      } else {
        if (one) run_pass(std::true_type{}, std::false_type{});
        else run_pass(std::false_type{}, std::false_type{});
      }
    }
  } else {
    // ============================ epilogue (warps 2..9, both CTAs) ============================
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int r = q * 32 + lane;
    const int H = prob->H, W = prob->W, out_H = prob->out_H, out_W = prob->out_W, out_C = prob->out_C;
    const int out_c_off = prob->out_c_off, act = prob->act;
    sp_t* const out_hi = prob->out_hi;
    sp_t* const out_lo = prob->out_lo;
    sp_t* const pool_hi = prob->pool_hi;
    sp_t* const pool_lo = prob->pool_lo;
    const int pool_C = prob->pool_C;
    const bool do_pool = pool_hi != nullptr;
    const bool lo_skip = prob->out_lo_skip != 0;
    const uint32_t t_empty_leader0 = map_to_cta(t_empty(0), 0), t_empty_leader1 = map_to_cta(t_empty(1), 0);
    uint32_t it = 0;
    for (int sit = item0; sit < nsuper; sit += item_step, ++it) {
      const uint32_t acc = it & 1u;
      mbar_wait(t_full(acc), (it >> 1) & 1u);
      tc_fence_after();
      const int nsub = (dual && 2 * sit + 1 < nitems) ? 2 : 1;
     for (int sub = 0; sub < nsub; ++sub) {
      const int item = dual ? 2 * sit + sub : sit;
      int sp, nti, b, rem, ty, tx;
      div_nt.divmod(item, sp, nti);
      div_img.divmod(sp, b, rem);
      div_tx.divmod(rem, ty, tx);
      const int n0 = nti * BN;
      const int py = (2 * ty + (int)rank) * kTileH + r / kTileW, px = tx * kTileW + r % kTileW;
      const bool valid = (py < H) && (px < W);
      const int64_t opix = ((int64_t)b * out_H + py) * out_W + px;
      sp_t* oh = out_hi + opix * out_C + out_c_off + n0;
      sp_t* ol = out_lo + opix * out_C + out_c_off + n0;
      const uint32_t t_addr = tmem_base + (acc * sub_n + sub) * kAccCols + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int cc = half; cc < BN / 16; cc += 2) {
        if (n0 + cc * 16 >= cout) break;
        uint32_t v[16];
        tmem_ld16(t_addr + (uint32_t)(cc * 16), v);
        if (kFused && !one) {
          uint32_t u[16];
          tmem_ld16(t_addr + (uint32_t)(BN + cc * 16), u);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
        } else {
          tmem_ld_wait();
        }
        {
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float x = __uint_as_float(v[j]) + bias_smem[n0 + cc * 16 + j];
            f[j] = act ? leaky(x) : x;
          }
          if (valid) {
            if (lo_skip) pack_store16_hi(f, oh + cc * 16);
            else pack_store16(f, oh + cc * 16, ol + cc * 16);   // two 32-byte stores
          }
          if (do_pool) {
            float pf[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float a = f[j] + __shfl_xor_sync(0xffffffffu, f[j], 1);
              pf[j] = (a + __shfl_xor_sync(0xffffffffu, a, 8)) * 0.25f;
            }
            // even-row, even-column lanes own the pooled pixel; VALID pooling floors (odd sizes drop the last row / column)
            if (!(lane & 1) && !(lane & 8) && (py >> 1) < (out_H >> 1) && (px >> 1) < (out_W >> 1)) {
              const int64_t ppix = ((int64_t)b * (out_H >> 1) + (py >> 1)) * (out_W >> 1) + (px >> 1);
              pack_store16(pf, pool_hi + ppix * pool_C + n0 + cc * 16, pool_lo + ppix * pool_C + n0 + cc * 16);
            }
          }
        }
      }
     }  // sub-items
      // this CTA's half of the accumulator is drained: tell the leader's MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(acc ? t_empty_leader1 : t_empty_leader0);
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // neither CTA may exit (or free TMEM) while the peer can still signal / read it
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, kTmemCols);
  }
}

int smem_bytes_for2(const ConvProblem& h, int bn) {
  const int nkb = h.ktot / h.kchunk;
  const int planes = h.passes == 1 ? 1 : 2;
  const int wt = w_half_tap_bytes(bn, h.kchunk, planes);
  const int w = h.v2_resident ? nkb * wt : h.v2_nw * wt;
  return h.v2_na * a_stage_bytes2h(h.kchunk, h.halo, planes) + w + kFixedBytes;
}

}  // namespace

int conv_tc_block_n(int cout);

bool conv3x3_tc2_plan(ConvProblem& h, int num_sms) {
  const int bn = h.bn;
  if (h.ntaps != 9 || h.tile_h != kTileH || h.tile_w != kTileW) return false;
  if (h.kchunk == 32 && bn != 32) return false;
  if (h.cout % bn) return false;            // whole N tiles only (the half-row boxes must not straddle Cout)
  const int nkb = h.ktot / h.kchunk;
  const int planes = h.passes == 1 ? 1 : 2;
  const int wtap = w_half_tap_bytes(bn, h.kchunk, planes);
  const int w_all = nkb * wtap;
  const bool can_resident = h.cout <= bn && 2 * (long)nkb * wtap < (1 << 20);
  // wide halo (the engine allows it per chunk size): resident weights win when both do not fit
  if (h.halo && can_resident && w_all + 2 * a_stage_bytes2h(h.kchunk, 0, planes) + kFixedBytes <= kSmemLimit &&
      w_all + 2 * a_stage_bytes2h(h.kchunk, 1, planes) + kFixedBytes > kSmemLimit)
    h.halo = 0;
  const int a_stage = a_stage_bytes2h(h.kchunk, h.halo, planes);
  h.v2_resident = 0;
  if (can_resident && w_all + 2 * a_stage + kFixedBytes <= kSmemLimit) {
    h.v2_resident = 1;
    int na = (kSmemLimit - kFixedBytes - w_all) / a_stage;
    const int na_max = h.halo ? 3 : 6;
    h.v2_na = na > na_max ? na_max : na;
    h.v2_nw = 1;
  } else {
    h.v2_na = h.halo ? 2 : 3;   // a halo stage feeds nine taps: two stages look further ahead than three did
    int nw = (kSmemLimit - kFixedBytes - h.v2_na * a_stage) / wtap;
    h.v2_nw = nw > kMaxRing ? kMaxRing : nw;
    if (h.v2_nw < 2) return false;
  }
  const int pairs_y = (h.tiles_y + 1) / 2;
  const int n_nt = (h.cout + bn - 1) / bn;
  int nitems = h.B * pairs_y * h.tiles_x * n_nt;
  // dual-item mode (the engine sets h.dual = 1 to ALLOW it): streamed weights, wide halo, one N tile, two accumulator
  // sets in TMEM (BN <= 128) and at least one activation stage per sub-item with two weight stages next to them
  if (h.dual) {
    bool ok = !h.v2_resident && h.halo && n_nt == 1 && bn <= 128 && nitems >= 4 * (num_sms / 2);
    if (ok) {
      int na = 4;
      if (na * a_stage + 2 * wtap + kFixedBytes > kSmemLimit) na = 2;
      ok = na * a_stage + 2 * wtap + kFixedBytes <= kSmemLimit;
      if (ok) {
        h.v2_na = na;
        int nw = (kSmemLimit - kFixedBytes - na * a_stage) / wtap;
        h.v2_nw = nw > kMaxRing ? kMaxRing : nw;
        nitems = (nitems + 1) / 2;
      }
    }
    h.dual = ok ? 1 : 0;
  }
  int grid = 2 * nitems;
  const int max_grid = num_sms & ~1;
  h.v2_grid = grid < max_grid ? grid : max_grid;
  h.pair = 1;
  return true;
}

cudaError_t conv3x3_tc2_configure() {
  cudaError_t e;
#define FILM_CFG(BN, KC)                                                                                      \
  e = cudaFuncSetAttribute(k_conv3x3_tc2<BN, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);   \
  if (e != cudaSuccess) return e;
  FILM_CFG(32, 64) FILM_CFG(64, 64) FILM_CFG(128, 64) FILM_CFG(256, 64) FILM_CFG(32, 32)
#undef FILM_CFG
  return cudaSuccess;
}

cudaError_t launch_conv3x3_tc2(const ConvProblem* d_prob, const ConvProblem& h, cudaStream_t st) {
  const int bn = h.bn;
  const int smem = smem_bytes_for2(h, bn);
  if (h.kchunk == 32) {
    k_conv3x3_tc2<32, 32><<<h.v2_grid, kThreads, smem, st>>>(d_prob);
    return cudaGetLastError();
  }
  switch (bn) {
    case 256: k_conv3x3_tc2<256, 64><<<h.v2_grid, kThreads, smem, st>>>(d_prob); break;
    case 128: k_conv3x3_tc2<128, 64><<<h.v2_grid, kThreads, smem, st>>>(d_prob); break;
    case 64: k_conv3x3_tc2<64, 64><<<h.v2_grid, kThreads, smem, st>>>(d_prob); break;
    default: k_conv3x3_tc2<32, 64><<<h.v2_grid, kThreads, smem, st>>>(d_prob); break;
  }
  return cudaGetLastError();
}

}  // namespace film
