// Persistent tcgen05 3x3 convolution with activation-tile reuse across taps (sm_100a).
//
// Why a second kernel: ncu on the generic kernel (profiles/r1_ncu_conv.md) shows the N <= 64
// layers re-loading the same activation pixels once per tap (9 x 32 KiB per 64-channel chunk and
// tile) and serialising prologue / mainloop / epilogue per tile.  Here:
//
//  * Tile = 16 rows x 8 columns of output pixels.  For a 64-channel chunk the producer loads
//    THREE boxes (dx = -1, 0, +1), each (64 ch, 8 px, 18 rows) of both planes: 144 pixel rows
//    of 128 B = 18 KiB per plane.  Because a tile row is exactly one 1024-byte swizzle atom
//    (8 px x 128 B), the operand of tap (dy, dx) is the SAME smem box at byte offset dy * 1024:
//    3 loads serve 9 taps (2.67x less L2 -> smem traffic) with plain, 1024-aligned UMMA descriptors.
//  * Weights: if the whole [Cout x K] hi+lo matrix fits (<= 144 KiB: 64->64, 128->32, 64->32 ...)
//    it is loaded ONCE per CTA and stays resident; otherwise it streams through its own ring,
//    one tap ([BN x 64] hi+lo) per stage.
//  * Persistent CTAs (grid = #SMs) walk a static tile list; the fp32 accumulator is double-buffered
//    in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.
//  * Fused-N product (BN <= 128): every M=128,K=16 SS-mode tcgen05.mma costs >= 72 cycles whatever
//    N <= 128 is (tools/ubench/mma_bench.cu, measured), so the 3-pass product is issued as TWO
//    instructions per k-step:  A_hi x [W_hi ; W_lo]  (N = 2*BN, the two weight planes are contiguous
//    in smem) and  A_lo x W_hi  accumulating into columns [0,BN).  The epilogue adds the halves.
//
// Roles (all role loops are warp-uniform, one elected lane issues): warp 0 = TMA producer
// (+ L2 prefetch of the next tile's boxes), warp 1 = TMEM allocator + MMA issuer, warps 2-9 = epilogue
// (two warps per TMEM lane quarter, alternating 16-column chunks).
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
// Tile shapes: tile_w must be a multiple of 8 pixels (one swizzle atom) and tile_h * tile_w = 128.
// 16x8 has the smallest halo (18/16); 8x16 and 4x32 exist to avoid wave quantisation on small levels.
__host__ __device__ constexpr int a_plane_bytes(int kc, int th, int tw) { return (th + 2) * tw * kc * 2; }
__host__ __device__ constexpr int a_stage_bytes(int kc, int th, int tw) { return 2 * a_plane_bytes(kc, th, tw); }
// Wide-halo mode (16x8 tiles, 64-channel chunks): ONE box (64 ch, 10 px, 18 rows) per plane and chunk serves
// all nine taps -- the UMMA descriptor of tap (dy, dx) starts (dy * 10 + dx) * 128 B into the box and steps
// 1280 B between 8-row groups (hardware check: tools/ubench/desc_offset_test.cu).  2.4x less L2 -> smem
// activation traffic than the three dx-shifted boxes.
constexpr int kHaloW = 10, kHaloRows = 18;
__host__ __device__ constexpr int halo_box_bytes(int kc) { return kHaloRows * kHaloW * kc * 2; }  // 23,040 for KC = 64
__host__ __device__ constexpr int halo_plane_bytes(int kc) { return (halo_box_bytes(kc) + 1023) & ~1023; }  // 1 KiB-aligned planes
__host__ __device__ constexpr int halo_stage_bytes(int kc) { return 2 * halo_plane_bytes(kc); }
// `planes` = 2 (hi + lo, three-pass product) or 1 (single-pass layers load the hi planes only)
__host__ __device__ constexpr int a_stage_bytes_h(int kc, int th, int tw, int halo, int planes = 2) {
  return planes * (halo ? halo_plane_bytes(kc) : a_plane_bytes(kc, th, tw));
}
constexpr int kMaxRing = 8;
constexpr int kSmemLimit = 227 * 1024;
constexpr int kBarBytes = 8 * (4 * kMaxRing + 4);
constexpr int kFixedBytes = kBarBytes + 16 + 512 * 4 /*bias*/ + 64 /*src table: 16 ints*/ + 1024 /*align*/ + 64;
// flow-head epilogue (epi_mode 3): partial sums [32 hidden][128 rows] + W3 [64][32] + b3 / W4 / b4, after the src table
constexpr int kHeadPart = 32 * 128 * 4, kHeadW3 = 64 * 32 * 4, kHeadMisc = 512;
constexpr int kHeadBytes = kHeadPart + kHeadW3 + kHeadMisc;

__host__ __device__ inline int w_tap_bytes(int bn, int kc, int planes = 2) { return bn * kc * 2 * planes; }  // [BN x KC] hi (+ lo)

template <int BN, int KC>
__global__ void __launch_bounds__(kThreads, 1) k_conv3x3_tc(const ConvProblem* __restrict__ prob) {
  extern __shared__ uint8_t smem_raw[];
  const bool one = prob->passes == 1;   // single-pass product A_hi x W_hi: hi planes only
  const int planes = one ? 1 : 2;
  constexpr int kWPlane = BN * KC * 2;  // one weight plane of one tap
  const int kWTap = kWPlane * planes;
  const int kTileH = prob->tile_h, kTileW = prob->tile_w;
  constexpr int kHaloBox = halo_box_bytes(KC), kHaloPlane = halo_plane_bytes(KC), kHaloStage = halo_stage_bytes(KC);
  const bool halo = prob->halo != 0;   // plan guarantees 16x8 tiles
  const int kAPlane = halo ? kHaloPlane : a_plane_bytes(KC, kTileH, kTileW);
  const int kAStage = planes * kAPlane;
  (void)kHaloStage;
  const int kRowStep = kTileW * KC * 2;  // one tile row of pixels = tile_w/8 swizzle atoms
  constexpr bool kFused = BN <= 128;
  constexpr uint32_t kAccCols = kFused ? 2 * BN : BN;
  constexpr uint32_t kTmemCols = 2 * kAccCols;

  // ---- problem fields -> registers, once (the asm "memory" clobbers would otherwise force a
  //      global reload of every P.* access inside the role loops)
  const int NA = prob->v2_na, NW = prob->v2_nw;
  const bool resident = prob->v2_resident != 0;
  const int nsrc = prob->nsrc;
  const int tiles_x = prob->tiles_x, tiles_per_img = prob->tiles_y * prob->tiles_x;
  const int cout = prob->cout;
  const int n_nt = (cout + BN - 1) / BN;                       // N tiles (Cout = 512 -> 2)
  const int ntiles = prob->B * tiles_per_img * n_nt;            // work items (spatial, N), N fastest
  int nkb = 0;                                                  // K blocks = (source, chunk, dx, dy)
  for (int s = 0; s < nsrc; ++s) nkb += prob->src[s].nchunk * 9;

  const FastDiv div_nt(n_nt, ntiles), div_img(tiles_per_img, ntiles), div_tx(tiles_x, ntiles);   // tile decode

  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* gen_base = smem_raw + (base - raw);
  const uint32_t a_base = base;
  const uint32_t w_base = a_base + (uint32_t)NA * kAStage;
  const uint32_t w_bytes = resident ? (uint32_t)nkb * kWTap : (uint32_t)NW * kWTap;
  const uint32_t tail = w_base + w_bytes;
  const uint32_t tail_off = (uint32_t)NA * kAStage + w_bytes;
  // barrier k lives at tail + 8k: a_full[0..7], a_empty[8..15], w_full[16..23], w_empty[24..31], t_full[32,33], t_empty[34,35]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(gen_base + tail_off + kBarBytes);
  float* bias_smem = reinterpret_cast<float*>(gen_base + tail_off + kBarBytes + 16);
  int* src_tab = reinterpret_cast<int*>(gen_base + tail_off + kBarBytes + 16 + 512 * 4);  // {nchunk, c_off} x 4

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kMaxRing; ++s) {
      mbar_init(tail + 8u * s, 1);
      mbar_init(tail + 8u * (kMaxRing + s), 1);
      mbar_init(tail + 8u * (2 * kMaxRing + s), 1);
      mbar_init(tail + 8u * (3 * kMaxRing + s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tail + 8u * (4 * kMaxRing + s), 1);
      mbar_init(tail + 8u * (4 * kMaxRing + 2 + s), kEpiWarps);  // one arrive per epilogue warp
    }
    for (int s = 0; s < kMaxSrc; ++s) {
      src_tab[2 * s] = s < nsrc ? prob->src[s].nchunk : 0;
      src_tab[2 * s + 1] = s < nsrc ? prob->src[s].c_off : 0;
      src_tab[2 * kMaxSrc + s] = s < nsrc ? prob->src[s].ksteps : 0;
      src_tab[3 * kMaxSrc + s] = s < nsrc ? prob->src[s].bswap : 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_ptr_smem), kTmemCols);
  if (warp >= 2)
    for (int i = threadIdx.x - 64; i < n_nt * BN; i += 32 * kEpiWarps) bias_smem[i] = (i < cout) ? prob->bias[i] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ============================ TMA producer (warp-uniform) ============================
    const CUtensorMap* tm_w_hi = &prob->tm_w_hi;
    const CUtensorMap* tm_w_lo = &prob->tm_w_lo;
    if (resident && elect_one()) {
      // whole weight matrix, once: nkb blocks of [BN x 64] hi then lo
      mbar_expect_tx(tail + 8u * (2 * kMaxRing), (uint32_t)nkb * kWTap);
      for (int kb = 0; kb < nkb; ++kb) {
        tma_load_2d(w_base + kb * kWTap, tm_w_hi, tail + 8u * (2 * kMaxRing), kb * KC, 0);
        if (!one) tma_load_2d(w_base + kb * kWTap + kWPlane, tm_w_lo, tail + 8u * (2 * kMaxRing), kb * KC, 0);
      }
    }
    __syncwarp();
    RingPos ra, rw;   // activation / weight ring positions
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      int sp, nti, b, rem, ty, tx;
      div_nt.divmod(tile, sp, nti);
      div_img.divmod(sp, b, rem);
      div_tx.divmod(rem, ty, tx);
      const int n0 = nti * BN, y0 = ty * kTileH, x0 = tx * kTileW;
      {
        // L2 prefetch of this CTA's NEXT spatial tile: first touch of an activation tile is DRAM
        const int nt = tile + gridDim.x;
        int nsp, nnt;
        div_nt.divmod(nt < ntiles ? nt : 0, nsp, nnt);
        if (nt < ntiles && nsp != sp && elect_one()) {
          int nb, nrem, nty, ntx;
          div_img.divmod(nsp, nb, nrem);
          div_tx.divmod(nrem, nty, ntx);
          const int ny0 = nty * kTileH, nx0 = ntx * kTileW;
          for (int s = 0; s < nsrc; ++s)
            for (int ch = 0; ch < src_tab[2 * s]; ++ch) {
              // the three dx boxes overlap: boxes at dx = 0 and dx = 2 cover the (tile_w + 2)-px-wide halo
              const int cc = src_tab[2 * s + 1] + ch * KC;
              tma_prefetch_4d(&prob->tm_a_hi[s], cc, nx0 - 1, ny0 - 1, nb);
              if (!one) tma_prefetch_4d(&prob->tm_a_lo[s], cc, nx0 - 1, ny0 - 1, nb);
              if (!halo) {  // (the wide box already spans the halo)
                tma_prefetch_4d(&prob->tm_a_hi[s], cc, nx0 + 1, ny0 - 1, nb);
                if (!one) tma_prefetch_4d(&prob->tm_a_lo[s], cc, nx0 + 1, ny0 - 1, nb);
              }
            }
        }
        __syncwarp();
      }
      int kb = 0;
      for (int s = 0; s < nsrc; ++s) {
        const int nchunk = src_tab[2 * s], c_off = src_tab[2 * s + 1];
        const int bs = src_tab[3 * kMaxSrc + s] ? prob->B - 1 - b : b;
        const CUtensorMap* tm_hi = &prob->tm_a_hi[s];
        const CUtensorMap* tm_lo = &prob->tm_a_lo[s];
        for (int ch = 0; ch < nchunk; ++ch) {
          const int nst = halo ? 1 : 3;   // activation stages of this chunk: one wide halo box or three dx boxes
          for (int dx = 0; dx < nst; ++dx) {
            const int st = ra.stage;
            mbar_wait(tail + 8u * (kMaxRing + st), ra.phase ^ 1u);
            if (elect_one()) {
              const uint32_t sa = a_base + st * kAStage, bar = tail + 8u * st;
              mbar_expect_tx(bar, halo ? (uint32_t)(planes * kHaloBox) : (uint32_t)kAStage);
              tma_load_4d(sa, tm_hi, bar, c_off + ch * KC, x0 + dx - 1, y0 - 1, bs);
              if (!one) tma_load_4d(sa + kAPlane, tm_lo, bar, c_off + ch * KC, x0 + dx - 1, y0 - 1, bs);
            }
            __syncwarp();
            ra.advance(NA);
            if (!resident) {
              const int ntap = halo ? 9 : 3;   // weight taps consumed against this activation stage
              for (int t = 0; t < ntap; ++t, ++kb) {
                const int ws = rw.stage;
                mbar_wait(tail + 8u * (3 * kMaxRing + ws), rw.phase ^ 1u);
                if (elect_one()) {
                  const uint32_t sw = w_base + ws * kWTap, bar = tail + 8u * (2 * kMaxRing + ws);
                  mbar_expect_tx(bar, kWTap);
                  tma_load_2d(sw, tm_w_hi, bar, kb * KC, n0);
                  if (!one) tma_load_2d(sw + kWPlane, tm_w_lo, bar, kb * KC, n0);
                }
                __syncwarp();
                rw.advance(NW);
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ============================ MMA issuer (warp-uniform, elected lane issues) ============================
    const uint32_t idesc = make_idesc<BN>();
    const uint32_t idesc2 = make_idesc<(kFused ? 2 * BN : BN)>();
    if (resident) {
      mbar_wait(tail + 8u * (2 * kMaxRing), 0);
      tc_fence_after();
    }
    // The item loop is instantiated twice: sources whose trailing 16-channel k-steps are zero padding in every
    // chunk (ConvSrc::ksteps < KC/16: the 10-of-64 "side" source, the 3-of-32 image block) skip those k-steps;
    // every other layer runs the loop without the bookkeeping (the issuing warp is issue-bound).
    bool any_partial = false;
    for (int s = 0; s < kMaxSrc; ++s) any_partial |= src_tab[2 * s] > 0 && src_tab[2 * kMaxSrc + s] < KC / 16;
    // Halo mode: one activation stage per chunk carries all nine taps; tap t = 3*dx + dy (the K order of the
    // packed weights) reads the box at byte offset (dy * 10 + dx) * 128, 8-row groups 1280 B apart.
    auto run_items = [&](auto partial_tag, auto halo_tag, auto one_tag, auto res_tag) {
      constexpr bool kPartial = decltype(partial_tag)::value;
      constexpr bool kHalo = decltype(halo_tag)::value;
      constexpr bool kOne = decltype(one_tag)::value;   // single-pass product
      constexpr bool kRes = decltype(res_tag)::value;   // weights resident in smem: no waits between the taps of a stage
      constexpr int kWTapC = kWPlane * (kOne ? 1 : 2);
      constexpr int kStageTaps = kHalo ? 9 : 3;   // taps served by one activation stage
      constexpr int kSrcStages = kHalo ? 1 : 3;   // activation stages per chunk
      const int nab = nkb / kStageTaps;           // activation stages per tile
      RingPos ra, rw;   // activation / weight ring positions
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const uint32_t acc = it & 1u;
        mbar_wait(tail + 8u * (4 * kMaxRing + 2 + acc), ((it >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kAccCols;
        int kb = 0;
        [[maybe_unused]] int src_i = 0, src_left = src_tab[0] * kSrcStages;  // stages left in the current source
        for (int ab = 0; ab < nab; ++ab) {
          [[maybe_unused]] int ksteps = KC / 16;
          if constexpr (kPartial) {
            while (src_left == 0) {
              ++src_i;
              src_left = src_tab[2 * src_i] * kSrcStages;
            }
            --src_left;
            ksteps = src_tab[2 * kMaxSrc + src_i];
          }
          const int st = ra.stage;
          mbar_wait(tail + 8u * st, ra.phase);
          tc_fence_after();
          const uint32_t sa = a_base + st * kAStage;
          if constexpr (kRes) {
            // Resident weights: nothing to wait for inside the stage, so ONE elected lane issues all of its taps as
            // straight-line code -- descriptors are a base plus compile-time offsets (the 14-bit address field
            // cannot carry: smem offsets are < 256 KiB), ~2 instructions per MMA instead of ~90 per tap.
            if (elect_one()) {
              constexpr uint32_t kPx = KC * 2;   // bytes of one pixel row of the box
              const uint64_t a0 = kHalo ? make_desc_sbo<KC>(sa, kHaloW * kPx) : make_desc_kc<KC>(sa);
              const uint64_t lo_delta = (uint64_t)((kHalo ? kHaloPlane : kAPlane) >> 4);
              const uint64_t row_delta = (uint64_t)(kRowStep >> 4);
              const uint64_t w0 = make_desc_kc<KC>(w_base + kb * kWTapC);
              const uint32_t first = (kb == 0) ? 0u : 1u;
#pragma unroll
              for (int t = 0; t < kStageTaps; ++t) {
                const uint64_t a_hi = a0 + (kHalo ? (uint64_t)((((t % 3) * kHaloW + t / 3) * kPx) >> 4) : (uint64_t)t * row_delta);
                const uint64_t a_lo = a_hi + lo_delta;
                const uint64_t w_hi = w0 + (uint64_t)((t * kWTapC) >> 4), w_lo = w_hi + (uint64_t)(kWPlane >> 4);
#pragma unroll
                for (int k = 0; k < KC / 16; ++k) {
                  if (!kPartial || k < ksteps) {
                    const uint64_t adv = (uint64_t)(k * 32 >> 4);
                    const uint32_t accf = (t == 0 && k == 0) ? first : 1u;
                    if constexpr (kOne) {
                      umma(d_tmem, a_hi + adv, w_hi + adv, idesc, accf);
                    } else if constexpr (kFused) {
                      umma(d_tmem, a_hi + adv, w_hi + adv, idesc2, accf);  // N = 2*BN: [W_hi ; W_lo]
                      umma(d_tmem, a_lo + adv, w_hi + adv, idesc, 1u);
                    } else {
                      umma(d_tmem, a_lo + adv, w_hi + adv, idesc, accf);
                      umma(d_tmem, a_hi + adv, w_lo + adv, idesc, 1u);
                      umma(d_tmem, a_hi + adv, w_hi + adv, idesc, 1u);
                    }
                  }
                }
              }
              umma_commit(tail + 8u * (kMaxRing + st));
              if (ab == nab - 1) umma_commit(tail + 8u * (4 * kMaxRing + acc));
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
              mbar_wait(tail + 8u * (2 * kMaxRing + ws), rw.phase);
              tc_fence_after();
              sw = w_base + ws * kWTap;
            }
            if (elect_one()) {
              uint64_t a_hi, a_lo;
              if constexpr (kHalo) {
                constexpr uint32_t kPx = KC * 2;   // bytes of one pixel row of the box
                const uint32_t off = (uint32_t)((t % 3) * kHaloW + t / 3) * kPx;
                a_hi = make_desc_sbo<KC>(sa + off, kHaloW * kPx);
                a_lo = make_desc_sbo<KC>(sa + kHaloPlane + off, kHaloW * kPx);
              } else {
                a_hi = make_desc_kc<KC>(sa + t * kRowStep);
                a_lo = make_desc_kc<KC>(sa + kAPlane + t * kRowStep);
              }
              const uint64_t w_hi = make_desc_kc<KC>(sw), w_lo = make_desc_kc<KC>(sw + kWPlane);
              const uint32_t first = (kb == 0) ? 0u : 1u;
  #pragma unroll
              for (int k = 0; k < KC / 16; ++k) {
                if constexpr (kPartial) {
                  if (k >= ksteps) break;
                }
                const uint64_t adv = (uint64_t)(k * 32 >> 4);
                if constexpr (kOne) {
                  umma(d_tmem, a_hi + adv, w_hi + adv, idesc, k == 0 ? first : 1u);
                } else if constexpr (kFused) {
                  umma(d_tmem, a_hi + adv, w_hi + adv, idesc2, k == 0 ? first : 1u);  // N = 2*BN: [W_hi ; W_lo]
                  umma(d_tmem, a_lo + adv, w_hi + adv, idesc, 1u);
                } else {
                  umma(d_tmem, a_lo + adv, w_hi + adv, idesc, k == 0 ? first : 1u);
                  umma(d_tmem, a_hi + adv, w_lo + adv, idesc, 1u);
                  umma(d_tmem, a_hi + adv, w_hi + adv, idesc, 1u);
                }
              }
              if (!resident) umma_commit(tail + 8u * (3 * kMaxRing + ws));
              if (t == kStageTaps - 1) umma_commit(tail + 8u * (kMaxRing + st));
              if (t == kStageTaps - 1 && ab == nab - 1) umma_commit(tail + 8u * (4 * kMaxRing + acc));
            }
            __syncwarp();
            if (!resident) rw.advance(NW);
          }
          }  // per-tap issue loop
          ra.advance(NA);
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
    if (resident && prob->straight) {
      if (one) run_pass(std::true_type{}, std::true_type{});
      else run_pass(std::false_type{}, std::true_type{});
    } else {
      if (one) run_pass(std::true_type{}, std::false_type{});
      else run_pass(std::false_type{}, std::false_type{});
    }
  } else {
    // ============================ epilogue (warps 2..9) ============================
    const int q = warp & 3;              // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;    // which 16-column chunks (even / odd) this warp drains
    const int r = q * 32 + lane;
    const int r_y = r / kTileW, r_x = r % kTileW;   // position of this thread's pixel inside the tile (tile-invariant)
    const int H = prob->H, W = prob->W, out_H = prob->out_H, out_W = prob->out_W, out_C = prob->out_C;
    const int out_c_off = prob->out_c_off, act = prob->act;
    sp_t* const out_hi = prob->out_hi;
    sp_t* const out_lo = prob->out_lo;
    // fused 2x2/2 average pool: only for 16x8 tiles (a warp's 32 lanes = 4 tile rows x 8 columns, so
    // the 2x2 partners of lane l are l^1, l^8, l^9 -> three warp shuffles on the fp32 values)
    sp_t* const pool_hi = prob->pool_hi;
    sp_t* const pool_lo = prob->pool_lo;
    const int pool_C = prob->pool_C;
    const bool do_pool = pool_hi != nullptr;
    const bool lo_skip = prob->out_lo_skip != 0;
    // RGB-head mode: channel partial sums of the 1x1 64 -> 3 conv; the two warps of a lane quarter own 32 channels each
    // and combine through shared memory (named barrier per quarter)
    const bool rgb = prob->epi_mode == 2;
    const float* const head_w = prob->head_w4;
    float* const rgb_out = prob->head_v;
    const int crop_y = prob->crop_y, crop_x = prob->crop_x, crop_h = prob->crop_h, crop_w = prob->crop_w;
    const int64_t crop_pitch = prob->crop_pitch;
    float* const part = bias_smem + 64;   // [128 rows][3] (bias_smem holds 64 biases in this mode, 512 floats in all)
    // flow-head mode (BN <= 64): hidden units = BN / 2; each warp of a lane quarter accumulates the partial sums of its
    // channels for every hidden unit, the pair combines through smem ([hidden][row]: conflict-free) and finishes the head
    const bool fhead = prob->epi_mode == 3;
    constexpr int kHid = BN <= 64 ? BN / 2 : 1;
    float* const hpart = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(src_tab) + 64);   // [kHid][128]
    float* const w3s = hpart + kHeadPart / 4;                                                   // [BN][kHid]
    float* const hmisc = w3s + kHeadW3 / 4;                                                     // b3[kHid] | w4[kHid][2] | b4[2]
    if (fhead) {
      if constexpr (BN <= 64) {
        for (int i = threadIdx.x - 64; i < BN * kHid; i += 32 * kEpiWarps) w3s[i] = prob->head_w3[i];
        for (int i = threadIdx.x - 64; i < kHid; i += 32 * kEpiWarps) hmisc[i] = prob->head_b3[i];
        for (int i = threadIdx.x - 64; i < 2 * kHid; i += 32 * kEpiWarps) hmisc[kHid + i] = prob->head_w4[i];
        if (threadIdx.x - 64 < 2) hmisc[3 * kHid + threadIdx.x - 64] = prob->head_b4[threadIdx.x - 64];
      }
      asm volatile("bar.sync 5, %0;" ::"r"(32 * kEpiWarps) : "memory");   // epilogue warps only
    }
    const float* const head_vup = prob->head_vup;
    float* const head_res = prob->head_res;
    float* const head_vout = prob->head_v;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const uint32_t acc = it & 1u;
      int sp, nti, b, rem, ty, tx;
      div_nt.divmod(tile, sp, nti);
      div_img.divmod(sp, b, rem);
      div_tx.divmod(rem, ty, tx);
      const int n0 = nti * BN;
      const int py = ty * kTileH + r_y, px = tx * kTileW + r_x;
      const bool valid = (py < H) && (px < W);
      const int64_t opix = ((int64_t)b * out_H + py) * out_W + px;
      sp_t* oh = out_hi + opix * out_C + out_c_off + n0;
      sp_t* ol = out_lo + opix * out_C + out_c_off + n0;
      mbar_wait(tail + 8u * (4 * kMaxRing + acc), (it >> 1) & 1u);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + acc * kAccCols + ((uint32_t)(q * 32) << 16);
      float r0 = 0.f, r1 = 0.f, r2 = 0.f;
      [[maybe_unused]] float hp[kHid];
      if constexpr (BN <= 64) {
#pragma unroll
        for (int hh = 0; hh < kHid; ++hh) hp[hh] = 0.f;
      }
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
          if (fhead) {
            if constexpr (BN <= 64) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float4* wr = reinterpret_cast<const float4*>(w3s + (cc * 16 + j) * kHid);   // broadcast reads
#pragma unroll
                for (int h4 = 0; h4 < kHid / 4; ++h4) {
                  const float4 wv = wr[h4];
                  hp[4 * h4] = fmaf(f[j], wv.x, hp[4 * h4]);
                  hp[4 * h4 + 1] = fmaf(f[j], wv.y, hp[4 * h4 + 1]);
                  hp[4 * h4 + 2] = fmaf(f[j], wv.z, hp[4 * h4 + 2]);
                  hp[4 * h4 + 3] = fmaf(f[j], wv.w, hp[4 * h4 + 3]);
                }
              }
            }
          } else if (rgb) {
            const float* hw = head_w + (n0 + cc * 16) * 3;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              r0 = fmaf(f[j], __ldg(hw + 3 * j), r0);
              r1 = fmaf(f[j], __ldg(hw + 3 * j + 1), r1);
              r2 = fmaf(f[j], __ldg(hw + 3 * j + 2), r2);
            }
          } else if (valid) {
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
            // lanes with even tile row and even tile column own the pooled pixel; VALID pooling floors, so on an
            // odd-sized level the last row / column has no pooled pixel (its 2x2 window would leave the grid)
            if (!(lane & 1) && !(lane & 8) && (py >> 1) < (out_H >> 1) && (px >> 1) < (out_W >> 1)) {
              const int64_t ppix = ((int64_t)b * (out_H >> 1) + (py >> 1)) * (out_W >> 1) + (px >> 1);
              pack_store16(pf, pool_hi + ppix * pool_C + n0 + cc * 16, pool_lo + ppix * pool_C + n0 + cc * 16);
            }
          }
        }
      }
      // accumulator drained: hand the TMEM buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tail + 8u * (4 * kMaxRing + 2 + acc));
      if (fhead) {
        if constexpr (BN <= 64) {
          if (half == 1) {
#pragma unroll
            for (int hh = 0; hh < kHid; ++hh) hpart[hh * 128 + r] = hp[hh];
          }
          asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
          if (half == 0 && valid) {
            float f0 = hmisc[3 * kHid], f1 = hmisc[3 * kHid + 1];
#pragma unroll
            for (int hh = 0; hh < kHid; ++hh) {
              const float x = leaky(hp[hh] + hpart[hh * 128 + r] + hmisc[hh]);     // conv_3: bias + LeakyReLU
              f0 = fmaf(x, hmisc[kHid + 2 * hh], f0);                                  // conv_4: linear
              f1 = fmaf(x, hmisc[kHid + 2 * hh + 1], f1);
            }
            float2 res = make_float2(f0, f1), tot = res;
            if (head_vup) {
              const float2 u = reinterpret_cast<const float2*>(head_vup)[opix];
              tot.x += u.x;
              tot.y += u.y;
            }
            reinterpret_cast<float2*>(head_res)[opix] = res;
            reinterpret_cast<float2*>(head_vout)[opix] = tot;
          }
          asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");   // hpart[] is rewritten by the next tile
        }
      } else if (rgb) {
        if (half == 1) {
          part[r * 3] = r0;
          part[r * 3 + 1] = r1;
          part[r * 3 + 2] = r2;
        }
        asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
        if (half == 0) {
          const int oy = py - crop_y, ox = px - crop_x;
          if (valid && oy >= 0 && oy < crop_h && ox >= 0 && ox < crop_w) {
            float* o = rgb_out + (int64_t)oy * crop_pitch + (int64_t)ox * 3;
            o[0] = r0 + part[r * 3] + __ldg(prob->head_b4);
            o[1] = r1 + part[r * 3 + 1] + __ldg(prob->head_b4 + 1);
            o[2] = r2 + part[r * 3 + 2] + __ldg(prob->head_b4 + 2);
          }
        }
        asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");   // part[] is rewritten by the next tile
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

int smem_bytes_for(const ConvProblem& h, int bn) {
  const int nkb = h.ktot / h.kchunk;
  const int planes = h.passes == 1 ? 1 : 2;
  const int w = h.v2_resident ? nkb * w_tap_bytes(bn, h.kchunk, planes) : h.v2_nw * w_tap_bytes(bn, h.kchunk, planes);
  return h.v2_na * a_stage_bytes_h(h.kchunk, h.tile_h, h.tile_w, h.halo, planes) + w + kFixedBytes +
         (h.epi_mode == 3 ? kHeadBytes : 0);
}

}  // namespace

int conv_tc_block_n(int cout);

// Tile shape: fewest waves over the SMs first (a 151st tile costs a whole extra wave on a small
// level), then the smallest halo.  16x8 is required by the fused pool.
void conv3x3_tc_pick_tile(int H, int W, int B, int cout, int num_sms, int& tile_h, int& tile_w) {
  static const int cand[3][2] = {{16, 8}, {8, 16}, {4, 32}};
  const int bn = conv_tc_block_n(cout);
  const int n_nt = (cout + bn - 1) / bn;
  double best = 1e30;
  for (auto& c : cand) {
    const long tiles = (long)B * ((H + c[0] - 1) / c[0]) * ((W + c[1] - 1) / c[1]) * n_nt;
    const long waves = (tiles + num_sms - 1) / num_sms;
    const double cost = (double)waves * (c[0] + 2.0) / c[0] * (1.0 + 1e-3 * (c[1] / 8));
    if (cost < best) {
      best = cost;
      tile_h = c[0];
      tile_w = c[1];
    }
  }
}

// Chooses resident/streamed weights and the ring depths for one 3x3 problem.
void conv3x3_tc_plan(ConvProblem& h, int num_sms) {
  const int bn = h.bn;
  const int nkb = h.ktot / h.kchunk;
  const int planes = h.passes == 1 ? 1 : 2;
  const int wtap = w_tap_bytes(bn, h.kchunk, planes);
  const int w_all = nkb * wtap;
  const bool can_resident = h.cout <= bn;
  const int kLimit = kSmemLimit - (h.epi_mode == 3 ? kHeadBytes : 0);   // flow-head epilogue scratch
  // wide halo (the engine allows it per chunk size): 16x8 tiles only; resident weights win when both do not fit
  if (h.halo && (h.tile_h != 16 || h.tile_w != 8 ||
                 (can_resident && w_all + 2 * a_stage_bytes_h(h.kchunk, h.tile_h, h.tile_w, 0, planes) + kFixedBytes <= kLimit &&
                  w_all + 2 * a_stage_bytes_h(h.kchunk, h.tile_h, h.tile_w, 1, planes) + kFixedBytes > kLimit)))
    h.halo = 0;
  const int kAStage = a_stage_bytes_h(h.kchunk, h.tile_h, h.tile_w, h.halo, planes);
  h.v2_resident = 0;
  if (can_resident && w_all + 2 * kAStage + kFixedBytes <= kLimit) {
    h.v2_resident = 1;
    int na = (kLimit - kFixedBytes - w_all) / kAStage;
    const int na_max = h.halo ? 3 : 6;
    h.v2_na = na > na_max ? na_max : na;
    h.v2_nw = 1;
  } else {
    h.v2_na = h.halo ? 2 : (bn >= 128 ? 2 : 3);
    int nw = (kLimit - kFixedBytes - h.v2_na * kAStage) / wtap;
    h.v2_nw = nw > kMaxRing ? kMaxRing : nw;
  }
  const int ntiles = h.B * h.tiles_y * h.tiles_x * ((h.cout + bn - 1) / bn);
  h.v2_grid = ntiles < num_sms ? ntiles : num_sms;
}

cudaError_t conv3x3_tc_configure() {
  cudaError_t e;
#define FILM_CFG(BN, KC)                                                                                     \
  e = cudaFuncSetAttribute(k_conv3x3_tc<BN, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);   \
  if (e != cudaSuccess) return e;
  FILM_CFG(32, 64) FILM_CFG(64, 64) FILM_CFG(128, 64) FILM_CFG(256, 64) FILM_CFG(32, 32) FILM_CFG(64, 32)
#undef FILM_CFG
  return cudaSuccess;
}

cudaError_t launch_conv3x3_tc(const ConvProblem* d_prob, const ConvProblem& h, cudaStream_t st) {
  const int bn = h.bn;
  const int smem = smem_bytes_for(h, bn);
  if (h.kchunk == 32) {  // 32-channel K blocks: the 32 -> 32 flow convs and the 3(32) -> 64 first conv
    if (bn == 32) k_conv3x3_tc<32, 32><<<h.v2_grid, kThreads, smem, st>>>(d_prob);
    else if (bn == 64) k_conv3x3_tc<64, 32><<<h.v2_grid, kThreads, smem, st>>>(d_prob);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
  }
  switch (bn) {
    case 256: k_conv3x3_tc<256, 64><<<h.v2_grid, kThreads, smem, st>>>(d_prob); break;
    case 128: k_conv3x3_tc<128, 64><<<h.v2_grid, kThreads, smem, st>>>(d_prob); break;
    case 64: k_conv3x3_tc<64, 64><<<h.v2_grid, kThreads, smem, st>>>(d_prob); break;
    default: k_conv3x3_tc<32, 64><<<h.v2_grid, kThreads, smem, st>>>(d_prob); break;
  }
  return cudaGetLastError();
}

}  // namespace film
