// Host side of the FILM B200 engine: weight loading + repacking, per-shape execution plans
// (arena, TMA tensor maps, static kernel schedule captured in a CUDA graph) and the C ABI of
// include/film_b200.h.  Network wiring follows the reference graph,
// models/film_net/interpolator.py:120-207; each step cites the lines it replaces.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/film_b200.h"
#include "film_conv.h"
#include "film_kernels.h"

namespace film {
int conv_tc_block_n(int cout);

// ----------------------------------------------------------------------------------------
// architecture constants (training/config/film_net-Style.gin:17-23)
// ----------------------------------------------------------------------------------------
constexpr int kLevels = 7, kFusionLevels = 5, kSpecialized = 3, kSubLevels = 4, kFilters = 64;
static const int kFlowFilters[4] = {32, 64, 128, 256};
static const char* kPredictorNames[4] = {"flow_predictor_0", "flow_predictor_1", "flow_predictor_2",
                                         "flow_predictor_shared"};
static int feat_channels(int l) {
  int c = 0;
  for (int j = 0; j <= (l < kSubLevels - 1 ? l : kSubLevels - 1); ++j) c += kFilters << j;
  return c;
}
static int fusion_filters(int l) { return l < kSpecialized ? (kFilters << l) : (kFilters << kSpecialized); }
static int round_up(int a, int b) { return (a + b - 1) / b * b; }

struct Error {
  int code;
  std::string msg;
};

// ----------------------------------------------------------------------------------------
// Precision plan.  Every tensor-core conv call site belongs to a STAGE; bit s of the plan's one-pass mask
// selects the single-pass product (A_hi x W_hi: fp16 operands, fp32 accumulate) for stage s, otherwise the
// three-pass split product (fp32-grade).  The flow heads and the RGB head are always three-pass / fp32.
// The default mask is the outcome of the measured per-stage error study (tools/precision_study.py,
// profiles/r2_precision_study_1080p.md, DESIGN.md section 3).
// ----------------------------------------------------------------------------------------
enum Stage {
  ST_FE_I0_K01 = 0, ST_FE_I0_K23, ST_FE_I0_K45, ST_FE_I0_K67,  // sub-tree of image level 0: conv pairs
  ST_FE_I1, ST_FE_I2, ST_FE_I3P,                                // sub-trees of image levels 1, 2, 3..6
  ST_FLOW_L0,                                                    // + pyramid level (7 levels): conv_0..2
  ST_FUS = ST_FLOW_L0 + kLevels,                                 // + 3 * fusion level + conv index
  ST_COUNT = ST_FUS + 3 * (kFusionLevels - 1),
  ST_NONE = -1
};
static std::string stage_name(int s) {
  static const char* fe[] = {"fe_i0_k01", "fe_i0_k23", "fe_i0_k45", "fe_i0_k67", "fe_i1", "fe_i2", "fe_i3p"};
  if (s < 0 || s >= ST_COUNT) return "";
  if (s < ST_FLOW_L0) return fe[s];
  if (s < ST_FUS) return "flow_L" + std::to_string(s - ST_FLOW_L0);
  return "fus" + std::to_string((s - ST_FUS) / 3) + "_c" + std::to_string((s - ST_FUS) % 3);
}
static int fe_stage(int image_level, int conv_k) {
  if (image_level == 0) return ST_FE_I0_K01 + conv_k / 2;
  return image_level == 1 ? ST_FE_I1 : image_level == 2 ? ST_FE_I2 : ST_FE_I3P;
}
// default: flow levels 0-4, the three deeper conv pairs of the level-0 sub-tree, fusion levels 2 and 3
constexpr uint32_t kDefaultOnepassMask =
    (1u << ST_FE_I0_K23) | (1u << ST_FE_I0_K45) | (1u << ST_FE_I0_K67) |
    (0x1Fu << ST_FLOW_L0) | (0x3Fu << (ST_FUS + 6));
#define FILM_CUDA(expr)                                                                       \
  do {                                                                                        \
    cudaError_t e__ = (expr);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      throw Error{FILM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)};        \
  } while (0)

// ----------------------------------------------------------------------------------------
// weight file (FILMW1, frame_interpolation_b200/weights.py)
// ----------------------------------------------------------------------------------------
struct HostTensor {
  std::vector<int> dims;
  std::vector<float> data;
};
typedef std::map<std::string, HostTensor> WeightMap;

static WeightMap read_weight_file(const char* path) {
  FILE* f = fopen(path, "rb");
  if (!f) throw Error{FILM_ERR_WEIGHTS, std::string("cannot open weight file ") + path};
  WeightMap m;
  auto fail = [&](const char* why) {
    fclose(f);
    throw Error{FILM_ERR_WEIGHTS, std::string(path) + ": " + why};
  };
  char magic[8];
  if (fread(magic, 1, 8, f) != 8 || memcmp(magic, "FILMW1\0\0", 8) != 0) fail("bad magic");
  uint32_t n;
  if (fread(&n, 4, 1, f) != 1) fail("truncated");
  for (uint32_t i = 0; i < n; ++i) {
    uint32_t ln, nd;
    if (fread(&ln, 4, 1, f) != 1 || ln > 4096) fail("bad name length");
    std::string name(ln, '\0');
    if (fread(&name[0], 1, ln, f) != ln) fail("truncated");
    if (fread(&nd, 4, 1, f) != 1 || nd > 8) fail("bad rank");
    HostTensor t;
    size_t cnt = 1;
    for (uint32_t d = 0; d < nd; ++d) {
      uint32_t v;
      if (fread(&v, 4, 1, f) != 1) fail("truncated");
      t.dims.push_back((int)v);
      cnt *= v;
    }
    t.data.resize(cnt);
    if (fread(t.data.data(), 4, cnt, f) != cnt) fail("truncated tensor data");
    m[name] = std::move(t);
  }
  fclose(f);
  return m;
}

static const HostTensor& get_tensor(const WeightMap& m, const std::string& name, std::vector<int> dims) {
  auto it = m.find(name);
  if (it == m.end()) throw Error{FILM_ERR_WEIGHTS, "missing tensor " + name};
  if (it->second.dims != dims) throw Error{FILM_ERR_WEIGHTS, "shape mismatch for " + name};
  return it->second;
}

// ----------------------------------------------------------------------------------------
// host-side rounding to the 16-bit split format (round-to-nearest-even, like the device)
// ----------------------------------------------------------------------------------------
static uint16_t f32_to_bf16(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static float bf16_to_f32(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
static uint16_t f32_to_sp(float f) {
#ifdef FILM_SPLIT_FP16
  __half h = __float2half_rn(f);
  uint16_t u;
  memcpy(&u, &h, 2);
  return u;
#else
  return f32_to_bf16(f);
#endif
}
static float sp_to_f32(uint16_t h) {
#ifdef FILM_SPLIT_FP16
  __half v;
  memcpy(&v, &h, 2);
  return __half2float(v);
#else
  return bf16_to_f32(h);
#endif
}

// ----------------------------------------------------------------------------------------
// packed weights of one tensor-core conv call-site type
// ----------------------------------------------------------------------------------------
struct PackedConv {
  sp_t* w_hi = nullptr;
  sp_t* w_lo = nullptr;
  float* bias = nullptr;
  int cout = 0, ktot = 0, cin_ref = 0;
  int kchunk = kChunk;          // channels per K block (64, or 32 for the 32-channel layers)
  std::vector<int> src_chunks;  // K-block chunks per source
  std::vector<int> src_ksteps;  // 16-channel k-steps per chunk that hold at least one real channel
  int ntaps = 0;
  int tap_dy[kMaxTaps], tap_dx[kMaxTaps];
};

struct TapSpec {
  int dy, dx;                               // offset on the input grid
  std::vector<std::pair<int, int>> terms;   // kernel positions (ky,kx) summed into this tap
};

// kernel: HWIO [kh][kw][cin][cout].  src_maps[s][slot] = reference input channel or -1 (zero).
// K order = (source, 64-chunk, tap, channel-in-chunk), matching the kernels' K loop.
static PackedConv pack_conv(const HostTensor& kernel, const HostTensor& bias,
                            const std::vector<std::vector<int>>& src_maps,
                            const std::vector<TapSpec>& taps, std::vector<void*>& allocs, int chunk = kChunk) {
  const int kw = kernel.dims[1], cin = kernel.dims[2], cout = kernel.dims[3];
  PackedConv pc;
  pc.cout = cout;
  pc.cin_ref = cin;
  pc.kchunk = chunk;
  pc.ntaps = (int)taps.size();
  for (size_t t = 0; t < taps.size(); ++t) {
    pc.tap_dy[t] = taps[t].dy;
    pc.tap_dx[t] = taps[t].dx;
  }
  int ktot = 0;
  for (auto& sm : src_maps) {
    if (sm.size() % chunk) throw Error{FILM_ERR_WEIGHTS, "source channel map not a multiple of the K chunk"};
    pc.src_chunks.push_back((int)sm.size() / chunk);
    // k-steps whose 16 channels are zero padding in EVERY chunk of the source are never issued (exact):
    // the 10-of-64 "side" source runs 1 of 4 k-steps, the 3-of-32 image block 1 of 2
    int ks = 1;
    for (size_t i = 0; i < sm.size(); ++i)
      if (sm[i] >= 0) ks = std::max(ks, (int)(i % chunk) / 16 + 1);
    pc.src_ksteps.push_back(ks);
    ktot += (int)sm.size() * (int)taps.size();
  }
  pc.ktot = ktot;
  std::vector<uint16_t> hi((size_t)cout * ktot), lo((size_t)cout * ktot);
  int kbase = 0;
  for (auto& sm : src_maps) {
    const int nchunk = (int)sm.size() / chunk;
    for (int ch = 0; ch < nchunk; ++ch) {
      for (size_t t = 0; t < taps.size(); ++t, kbase += chunk) {
        for (int c = 0; c < chunk; ++c) {
          const int ref = sm[ch * chunk + c];
          for (int n = 0; n < cout; ++n) {
            float w = 0.f;
            if (ref >= 0) {
              if (ref >= cin) throw Error{FILM_ERR_WEIGHTS, "channel map out of range"};
              for (auto& term : taps[t].terms)
                w += kernel.data[(((size_t)term.first * kw + term.second) * cin + ref) * cout + n];
            }
            const uint16_t h = f32_to_sp(w);
            const uint16_t l = f32_to_sp(w - sp_to_f32(h));
            hi[(size_t)n * ktot + kbase + c] = h;
            lo[(size_t)n * ktot + kbase + c] = l;
          }
        }
      }
    }
  }
  FILM_CUDA(cudaMalloc(&pc.w_hi, hi.size() * 2));
  allocs.push_back(pc.w_hi);
  FILM_CUDA(cudaMalloc(&pc.w_lo, lo.size() * 2));
  allocs.push_back(pc.w_lo);
  FILM_CUDA(cudaMalloc(&pc.bias, cout * 4));
  allocs.push_back(pc.bias);
  FILM_CUDA(cudaMemcpy(pc.w_hi, hi.data(), hi.size() * 2, cudaMemcpyHostToDevice));
  FILM_CUDA(cudaMemcpy(pc.w_lo, lo.data(), lo.size() * 2, cudaMemcpyHostToDevice));
  FILM_CUDA(cudaMemcpy(pc.bias, bias.data.data(), cout * 4, cudaMemcpyHostToDevice));
  return pc;
}

// dx-major tap order (kx outer, ky inner): the persistent 3x3 kernel consumes the three dy taps of
// one dx-shifted activation box back to back (film_conv3x3_tc.cu); the generic kernel is order-agnostic.
static std::vector<TapSpec> taps_3x3() {
  std::vector<TapSpec> t;
  for (int kx = 0; kx < 3; ++kx)
    for (int ky = 0; ky < 3; ++ky) t.push_back({ky - 1, kx - 1, {{ky, kx}}});
  return t;
}
// fusion.py:133-135: NN 2x upsample followed by a 2x2 SAME conv (pad bottom/right), evaluated on
// the COARSE grid per output parity (py,px): fine tap (fy,fx) reads coarse offset ((py+fy)/2,
// (px+fx)/2); taps that hit the same coarse pixel have their weights pre-summed.
static std::vector<TapSpec> taps_up2x2(int py, int px) {
  std::vector<TapSpec> t;
  for (int dy = 0; dy <= py; ++dy)
    for (int dx = 0; dx <= px; ++dx) {
      TapSpec s{dy, dx, {}};
      for (int fy = 0; fy < 2; ++fy)
        for (int fx = 0; fx < 2; ++fx)
          if ((py + fy) / 2 == dy && (px + fx) / 2 == dx) s.terms.push_back({fy, fx});
      t.push_back(s);
    }
  return t;
}
// the same 2x2 SAME conv on the fine grid (tap (ky,kx) reads offset (ky,kx); the bottom/right pad is the zero
// fill of out-of-bounds reads): the decoder's general path, used where the fine level is not twice the coarse one
static std::vector<TapSpec> taps_2x2() {
  std::vector<TapSpec> t;
  for (int ky = 0; ky < 2; ++ky)
    for (int kx = 0; kx < 2; ++kx) t.push_back({ky, kx, {{ky, kx}}});
  return t;
}
static std::vector<int> iota_map(int start, int n, int padded) {
  std::vector<int> m(padded, -1);
  for (int i = 0; i < n; ++i) m[i] = start + i;
  return m;
}
// side tensor slots (film_kernels.h launch_fusion_side) -> channels of the reference's aligned
// pyramid [img0w(3), feat0w(C), img1w(3), feat1w(C), bwd(2), fwd(2)] (interpolator.py:167-183)
static std::vector<int> side_map(int C) {
  std::vector<int> m(kChunk, -1);
  for (int c = 0; c < 3; ++c) m[c] = c;
  for (int c = 0; c < 3; ++c) m[3 + c] = 3 + C + c;
  m[6] = 6 + 2 * C;
  m[7] = 7 + 2 * C;
  m[8] = 8 + 2 * C;
  m[9] = 9 + 2 * C;
  return m;
}

// ----------------------------------------------------------------------------------------
// model weights on the device
// ----------------------------------------------------------------------------------------
struct Model {
  std::vector<void*> allocs;
  float *conv0_w = nullptr, *conv0_b = nullptr;  // cfeat_conv_0 [27][64]
  PackedConv fe[8];                              // fe[0] = 1x1 over im2col channels, fe[1..7] = 3x3
  PackedConv fe0_3x3;                            // cfeat_conv_0 as a 3x3 conv over a 32-channel-padded image
  PackedConv flow[4][3];                         // predictor p, 3x3 conv k
  PackedConv flow_c3[4];                         // predictor p, 1x1 conv_3 (tensor-core, fused head)
  float *flow_w3[4], *flow_b3[4], *flow_w4[4], *flow_b4[4];
  PackedConv fus_up[4][4];                       // level i, parity class py*2+px
  PackedConv fus_up_full[4];                     // level i, plain 2x2 conv on the fine grid (general path)
  PackedConv fus_c1[4], fus_c2[4];
  float *rgb_w = nullptr, *rgb_b = nullptr;

  float* upload(const HostTensor& t) {
    float* d;
    FILM_CUDA(cudaMalloc(&d, t.data.size() * 4));
    allocs.push_back(d);
    FILM_CUDA(cudaMemcpy(d, t.data.data(), t.data.size() * 4, cudaMemcpyHostToDevice));
    return d;
  }

  void load(const WeightMap& w) {
    const std::string fe_pre = "feat_net/sub_extractor/cfeat_conv_";
    conv0_w = upload(get_tensor(w, fe_pre + "0/kernel", {3, 3, 3, 64}));
    conv0_b = upload(get_tensor(w, fe_pre + "0/bias", {64}));
    {
      // tensor-core version of cfeat_conv_0: the HWIO kernel [3][3][3][64] flattened to a 1x1 conv over
      // the 27 im2col channels (k = (ky*3+kx)*3 + ci, film_kernels.cu k_im2col3x3), one 32-channel K block
      HostTensor k0 = get_tensor(w, fe_pre + "0/kernel", {3, 3, 3, 64});
      k0.dims = {1, 1, 27, 64};
      fe[0] = pack_conv(k0, get_tensor(w, fe_pre + "0/bias", {64}), {iota_map(0, 27, 32)},
                        {TapSpec{0, 0, {{0, 0}}}}, allocs, 32);
      // ... or directly as a 3x3 conv whose 32-channel K block holds the 3 image channels + 29 zeros
      fe0_3x3 = pack_conv(get_tensor(w, fe_pre + "0/kernel", {3, 3, 3, 64}), get_tensor(w, fe_pre + "0/bias", {64}),
                          {iota_map(0, 3, 32)}, taps_3x3(), allocs, 32);
    }
    int cin = 64;
    for (int k = 1; k < 8; ++k) {
      const int c = kFilters << (k / 2);
      fe[k] = pack_conv(get_tensor(w, fe_pre + std::to_string(k) + "/kernel", {3, 3, cin, c}),
                        get_tensor(w, fe_pre + std::to_string(k) + "/bias", {c}),
                        {iota_map(0, cin, cin)}, taps_3x3(), allocs);
      cin = c;
    }
    for (int p = 0; p < 4; ++p) {
      const std::string pre = std::string("predict_flow/") + kPredictorNames[p] + "/conv_";
      const int nf = kFlowFilters[p], C = feat_channels(p);
      flow[p][0] = pack_conv(get_tensor(w, pre + "0/kernel", {3, 3, 2 * C, nf}),
                             get_tensor(w, pre + "0/bias", {nf}),
                             {iota_map(0, C, C), iota_map(C, C, C)}, taps_3x3(), allocs);
      const int kc = nf < kChunk ? 32 : kChunk;  // the 32-filter predictor uses 32-channel K blocks
      for (int k = 1; k < 3; ++k)
        flow[p][k] = pack_conv(get_tensor(w, pre + std::to_string(k) + "/kernel", {3, 3, nf, nf}),
                               get_tensor(w, pre + std::to_string(k) + "/bias", {nf}),
                               {iota_map(0, nf, round_up(nf, kc))}, taps_3x3(), allocs, kc);
      flow_c3[p] = pack_conv(get_tensor(w, pre + "3/kernel", {1, 1, nf, nf / 2}),
                             get_tensor(w, pre + "3/bias", {nf / 2}), {iota_map(0, nf, round_up(nf, kc))},
                             {TapSpec{0, 0, {{0, 0}}}}, allocs, kc);
      flow_w3[p] = upload(get_tensor(w, pre + "3/kernel", {1, 1, nf, nf / 2}));
      flow_b3[p] = upload(get_tensor(w, pre + "3/bias", {nf / 2}));
      flow_w4[p] = upload(get_tensor(w, pre + "4/kernel", {1, 1, nf / 2, 2}));
      flow_b4[p] = upload(get_tensor(w, pre + "4/bias", {2}));
    }
    for (int i = 0; i < kFusionLevels - 1; ++i) {
      const std::string pre = "fusion/level_" + std::to_string(i) + "/conv_";
      const int nf = fusion_filters(i), C = feat_channels(i);
      const bool from_pyr = (i == kFusionLevels - 2);
      const int Cc = feat_channels(i + 1);
      const int coarse_c = from_pyr ? 2 * (3 + Cc) + 4 : fusion_filters(i + 1);
      const HostTensor& k0 = get_tensor(w, pre + "0/kernel", {2, 2, coarse_c, nf});
      const HostTensor& b0 = get_tensor(w, pre + "0/bias", {nf});
      std::vector<std::vector<int>> up_src;
      if (from_pyr)
        up_src = {iota_map(3, Cc, Cc), iota_map(6 + Cc, Cc, Cc), side_map(Cc)};
      else
        up_src = {iota_map(0, coarse_c, coarse_c)};
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px)
          fus_up[i][py * 2 + px] = pack_conv(k0, b0, up_src, taps_up2x2(py, px), allocs);
      fus_up_full[i] = pack_conv(k0, b0, up_src, taps_2x2(), allocs);
      const int a_c = 2 * (3 + C) + 4;
      fus_c1[i] = pack_conv(get_tensor(w, pre + "1/kernel", {3, 3, a_c + nf, nf}),
                            get_tensor(w, pre + "1/bias", {nf}),
                            {iota_map(3, C, C), iota_map(6 + C, C, C), side_map(C),
                             iota_map(a_c, nf, round_up(nf, kChunk))},
                            taps_3x3(), allocs);
      fus_c2[i] = pack_conv(get_tensor(w, pre + "2/kernel", {3, 3, nf, nf}),
                            get_tensor(w, pre + "2/bias", {nf}),
                            {iota_map(0, nf, round_up(nf, kChunk))}, taps_3x3(), allocs);
    }
    rgb_w = upload(get_tensor(w, "fusion/output_conv/kernel", {1, 1, 64, 3}));
    rgb_b = upload(get_tensor(w, "fusion/output_conv/bias", {3}));
  }
  ~Model() {
    for (void* p : allocs) cudaFree(p);
  }
};

// ----------------------------------------------------------------------------------------
// TMA tensor maps (driver entry point fetched through the runtime: no -lcuda link)
// ----------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    FILM_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !p)
      throw Error{FILM_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available"};
    fn = (EncodeTiledFn)p;
  }
  return fn;
}
#ifdef FILM_SPLIT_FP16
static const CUtensorMapDataType kTmType = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
#else
static const CUtensorMapDataType kTmType = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
#endif

static void make_act_map(CUtensorMap* tm, const sp_t* base, int B, int H, int W, int C, int th, int tw, int kc) {
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)kc, (cuuint32_t)tw, (cuuint32_t)th, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = get_encode_fn()(tm, kTmType, 4, (void*)base, dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, kc == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw Error{FILM_ERR_CUDA, "cuTensorMapEncodeTiled(activation) failed: " + std::to_string((int)r)};
}
static void make_w_map(CUtensorMap* tm, const sp_t* base, int cout, int ktot, int bn, int kc) {
  cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)cout};
  cuuint64_t strides[1] = {(cuuint64_t)ktot * 2};
  cuuint32_t box[2] = {(cuuint32_t)kc, (cuuint32_t)bn};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = get_encode_fn()(tm, kTmType, 2, (void*)base, dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, kc == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw Error{FILM_ERR_CUDA, "cuTensorMapEncodeTiled(weights) failed: " + std::to_string((int)r)};
}

// ----------------------------------------------------------------------------------------
// execution plan for one (h, w, align) shape
// ----------------------------------------------------------------------------------------
struct SplitBuf {
  sp_t* hi = nullptr;
  sp_t* lo = nullptr;
  int B = 0, H = 0, W = 0, C = 0;
  int64_t pixels() const { return (int64_t)B * H * W; }
};
struct SrcRef {
  const SplitBuf* buf;
  int c_off;
  int bswap;  // read with the batch index swapped (ConvSrc::bswap); 0 when omitted from a braced initialiser
};
struct DebugTensor {
  bool split;
  const void* p0;
  const void* p1;
  int64_t npix;
  int C, c_off, Cn;
  bool recycled = false;  // the buffer is reused later in the same plan (readable only with keep_debug = 1)
};

struct Plan {
  int h, w, H, W, off_y, off_x;
  int conv_impl;
  int conv3x3_v2 = 1, num_sms = 148, conv3x3_2cta = 0;
  int conv3x3_halo = 0;  // 1: pair kernel, 2: + single-CTA persistent kernel, 3: + 32-channel-chunk layers
  uint32_t onepass_mask = 0;  // precision plan: stages on the single-pass product
  int fe_conv0_tc = 0;        // 1: cfeat_conv_0 on the tensor cores (32-channel-padded image), 0: fp32 FMA kernel
  int fuse_rgb_head = 1;      // RGB head + crop in the epilogue of the decoder's last conv
  int conv3x3_dual = 0;       // CTA-pair kernel: two spatial items per streamed weight pass
  int fuse_flow_head = 1;     // flow head (conv_3, conv_4, residual add) in conv_2 epilogue: 1 = level 0, 2 = levels 0 and 1
  int plane_skip = 1;         // lo planes that no consumer reads are neither gathered nor written
  int mma_straight = 1;       // straight-line MMA issue for resident weights
  std::vector<void*> allocs;
  int64_t arena_bytes = 0;
  std::vector<ConvProblem> h_probs;
  ConvProblem* d_probs = nullptr;
  struct Op {
    std::function<cudaError_t(cudaStream_t)> fn;
    int category;      // 0 = tcgen05 conv, 1 = warp gather, 2 = other bandwidth kernels
    std::string name;
    double flops;      // reference-graph FLOPs (convs) of this op
    double bytes;      // algorithmic bytes (gathers)
    int lane;                  // stream lane the op is enqueued on
    std::vector<int> waits;    // tokens (events) the op waits for before it starts
    std::vector<int> signals;  // tokens recorded after the op
  };
  std::vector<Op> ops;
  std::vector<float> op_ms;  // filled by timed eager runs
  // Lanes: independent branches of the graph (the 7 per-scale feature-extractor chains, the
  // coarse-to-fine flow chain) are enqueued on different streams so that latency-bound coarse
  // levels overlap with the large fine-level kernels; cross-lane dependencies are tokens (events).
  static constexpr int kNumLanes = 8;
  int cur_lane = 0, num_tokens = 0, tok_end = -1;
  std::vector<int> pending_waits;
  int new_token() { return num_tokens++; }
  void add_op(int category, const std::string& name, std::function<cudaError_t(cudaStream_t)> fn,
              double flops = 0, double bytes = 0) {
    ops.push_back(Op{std::move(fn), category, name, flops, bytes, cur_lane, pending_waits, {}});
    pending_waits.clear();
  }
  void signal_last(int token) { ops.back().signals.push_back(token); }
  std::map<std::string, DebugTensor> debug;
  float* xin = nullptr;   // [2][h][w][3] unpadded inputs
  float* xout = nullptr;  // [h][w][3]
  cudaGraphExec_t graph = nullptr;
  double conv_flops = 0, mma_flops = 0, warp_bytes = 0, last_conv_bytes = 0;

  // Activation arena with liveness-based reuse.  The schedule is built in execution order and replayed on ONE
  // stream (or as the graph captured from it), so a buffer released at build position i may back any buffer
  // allocated at a position >= i: release() returns a block to the pool, alloc() takes the best-fitting free
  // block (at most 2x the request) before it asks the driver.  `pinned` buffers (network inputs/outputs, flows,
  // tensors whose zero-initialised padding channels are never rewritten) are never recycled.  Reuse is off
  // when intermediates must stay readable (keep_debug) or when branches run on concurrent streams (use_lanes).
  bool reuse = true;
  std::map<void*, int64_t> block_bytes;
  std::multimap<int64_t, void*> free_blocks;
  template <class T>
  T* alloc(int64_t count, bool pinned = false) {
    const int64_t bytes = std::max<int64_t>(count * (int64_t)sizeof(T), 256);
    if (reuse && !pinned) {
      auto it = free_blocks.lower_bound(bytes);
      if (it != free_blocks.end() && it->first <= 2 * bytes) {
        void* p = it->second;
        free_blocks.erase(it);
        return (T*)p;
      }
    }
    void* p;
    FILM_CUDA(cudaMalloc(&p, bytes));
    allocs.push_back(p);
    FILM_CUDA(cudaMemset(p, 0, bytes));
    arena_bytes += bytes;
    if (!pinned) block_bytes[p] = bytes;
    return (T*)p;
  }
  // the buffer's last reader has been added to the schedule
  void release(void* p) {
    if (!reuse || !p) return;
    auto it = block_bytes.find(p);
    if (it != block_bytes.end()) free_blocks.insert({it->second, p});
  }
  void release(const SplitBuf* s) {
    if (!s) return;
    release((void*)s->hi);
    release((void*)s->lo);
  }
  SplitBuf* split(int B, int H_, int W_, int C, bool pinned = false) {
    bufs.emplace_back(new SplitBuf);
    SplitBuf* s = bufs.back().get();
    s->B = B;
    s->H = H_;
    s->W = W_;
    s->C = C;
    s->hi = alloc<sp_t>((int64_t)B * H_ * W_ * C, pinned);
    s->lo = alloc<sp_t>((int64_t)B * H_ * W_ * C, pinned);
    return s;
  }
  std::vector<std::unique_ptr<SplitBuf>> bufs;

  ~Plan() {
    if (graph) cudaGraphExecDestroy(graph);
    for (void* p : allocs) cudaFree(p);
  }
};

static void pick_tile(int H, int W, int& th, int& tw) {
  static const int cand[][2] = {{8, 16}, {16, 8}, {4, 32}, {32, 4}, {2, 64}, {64, 2}, {1, 128}, {128, 1}};
  long best = -1;
  for (auto& c : cand) {
    long tiles = (long)((H + c[0] - 1) / c[0]) * ((W + c[1] - 1) / c[1]);
    if (best < 0 || tiles < best) {
      best = tiles;
      th = c[0];
      tw = c[1];
    }
  }
}

// Adds one conv call site to the plan.  The GEMM-M grid is the grid of sources[0].
static size_t add_conv(Plan& P, const std::string& tag, double ref_macs_per_px, const PackedConv& pc,
                       const std::vector<SrcRef>& sources, int act, const SplitBuf* out, int out_c_off,
                       int stage, int consumer, int sy = 1, int sx = 1, int oy = 0, int ox = 0,
                       const SplitBuf* pool_out = nullptr, bool no_op = false, int epi_mode = 0) {
  // `stage`: precision-plan stage of this conv.  `consumer`: stage of the ONLY reader of the destination when that
  // reader is a conv (ST_NONE otherwise): a single-pass reader never touches the lo plane, so it is not written.
  ConvProblem cp;
  memset(&cp, 0, sizeof(cp));
  cp.passes = (stage >= 0 && P.conv_impl == 0 && ((P.onepass_mask >> stage) & 1u)) ? 1 : 3;
  cp.out_lo_skip = (consumer >= 0 && P.conv_impl == 0 && !pool_out && P.plane_skip && ((P.onepass_mask >> consumer) & 1u)) ? 1 : 0;
  cp.straight = P.mma_straight;
  const SplitBuf* s0 = sources[0].buf;
  cp.nsrc = (int)sources.size();
  if (cp.nsrc != (int)pc.src_chunks.size()) throw Error{FILM_ERR_WEIGHTS, "source count mismatch"};
  cp.B = s0->B;
  cp.H = s0->H;
  cp.W = s0->W;
  // 3x3 SAME convs with a unit-stride destination run on the persistent tap-reuse kernel
  const int kc = pc.kchunk;
  cp.kchunk = kc;
  const bool v2 = P.conv3x3_v2 && P.conv_impl == 0 && pc.ntaps == 9 && (out || epi_mode >= 2) && sy == 1 && sx == 1 &&
                  (kc == kChunk || pc.cout <= 64);
  cp.epi_mode = epi_mode;
  int box_h, box_w;
  // CTA-pair kernel: large levels only (it needs 16x8 tiles and enough tile pairs to fill the SM pairs)
  const bool want_pair = v2 && P.conv3x3_2cta && epi_mode < 2 &&   // (the RGB / flow-head epilogues live in the single-CTA kernel)
                         (P.conv3x3_2cta >= 2 ||  // >= 2: every eligible layer (testing)
                          (long)cp.B * ((cp.H + 15) / 16) * ((cp.W + 7) / 8) >= 4L * P.num_sms);
  if (v2) {
    if (pool_out || want_pair) {
      cp.tile_h = 16;  // the fused pool maps 2x2 partners to lanes l^1 / l^8 of a 16x8 tile
      cp.tile_w = 8;
    } else {
      conv3x3_tc_pick_tile(cp.H, cp.W, cp.B, pc.cout, P.num_sms, cp.tile_h, cp.tile_w);
    }
    box_h = cp.tile_h + 2;
    box_w = cp.tile_w;
  } else {
    pick_tile(cp.H, cp.W, cp.tile_h, cp.tile_w);
    box_h = cp.tile_h;
    box_w = cp.tile_w;
  }
  cp.tiles_y = (cp.H + cp.tile_h - 1) / cp.tile_h;
  cp.tiles_x = (cp.W + cp.tile_w - 1) / cp.tile_w;
  for (int s = 0; s < cp.nsrc; ++s) {
    const SplitBuf* b = sources[s].buf;
    if (b->B != cp.B || b->H != cp.H || b->W != cp.W) throw Error{FILM_ERR_ARG, "conv source grid mismatch"};
    cp.src[s].hi = b->hi;
    cp.src[s].lo = b->lo;
    cp.src[s].C = b->C;
    cp.src[s].c_off = sources[s].c_off;
    cp.src[s].nchunk = pc.src_chunks[s];
    cp.src[s].ksteps = pc.src_ksteps[s];
    cp.src[s].bswap = sources[s].bswap;
    if (sources[s].c_off + pc.src_chunks[s] * kc > b->C) throw Error{FILM_ERR_ARG, "conv source channel overrun"};
    make_act_map(&cp.tm_a_hi[s], b->hi, b->B, b->H, b->W, b->C, box_h, box_w, kc);
    make_act_map(&cp.tm_a_lo[s], b->lo, b->B, b->H, b->W, b->C, box_h, box_w, kc);
  }
  cp.ntaps = pc.ntaps;
  for (int t = 0; t < pc.ntaps; ++t) {
    cp.tap_dy[t] = pc.tap_dy[t];
    cp.tap_dx[t] = pc.tap_dx[t];
  }
  cp.ktot = pc.ktot;
  cp.w_hi = pc.w_hi;
  cp.w_lo = pc.w_lo;
  cp.bias = pc.bias;
  cp.cout = pc.cout;
  cp.act = act;
  int bn = conv_tc_block_n(pc.cout);
  if (out && !pool_out) {
    // tiny pyramid levels: a 17x30 level has 8 tiles but K = 17280 -- split N into smaller tiles so the
    // K-serial work spreads over more SMs (and BN <= 128 tiles use the 2-instruction product)
    auto items = [&](int b) { return (long)cp.B * cp.tiles_y * cp.tiles_x * ((pc.cout + b - 1) / b); };
    while (bn > 64 && 2 * items(bn) <= P.num_sms) bn /= 2;  // only while under half of the SMs have work
  }
  cp.bn = bn;
  make_w_map(&cp.tm_w_hi, pc.w_hi, pc.cout, pc.ktot, bn, kc);
  make_w_map(&cp.tm_w_lo, pc.w_lo, pc.cout, pc.ktot, bn, kc);
  make_w_map(&cp.tm_w_hi_half, pc.w_hi, pc.cout, pc.ktot, bn / 2, kc);
  make_w_map(&cp.tm_w_lo_half, pc.w_lo, pc.cout, pc.ktot, bn / 2, kc);
  if (out) {
    cp.out_hi = out->hi;
    cp.out_lo = out->lo;
    cp.out_C = out->C;
    cp.out_H = out->H;
    cp.out_W = out->W;
  } else {  // flow-head mode: no split output, pixel index == input grid index
    cp.out_C = 0;
    cp.out_H = cp.H;
    cp.out_W = cp.W;
  }
  cp.out_c_off = out_c_off;
  cp.out_sy = sy;
  cp.out_sx = sx;
  cp.out_oy = oy;
  cp.out_ox = ox;
  if (out && (out->B != cp.B || out_c_off + pc.cout > out->C)) throw Error{FILM_ERR_ARG, "conv destination mismatch"};
  if (pool_out) {
    if (!v2) throw Error{FILM_ERR_UNSUPPORTED, "fused pool needs the persistent 3x3 kernel"};
    cp.pool_hi = pool_out->hi;
    cp.pool_lo = pool_out->lo;
    cp.pool_C = pool_out->C;
  }
  cp.group = 1;
  cp.pair = 0;
  bool pair = false;
  // wide halo level: 1 = pair kernel, 2 = + single-CTA kernel (64-channel chunks), 3 = + 32-channel chunks
  // (SWIZZLE_64B descriptor offsets verified by tools/ubench/desc_offset_test.cu; kernels not yet timed)
  int halo_ok = (v2 && cp.tile_h == 16 && cp.tile_w == 8) ? P.conv3x3_halo : 0;
  if (kc != kChunk && halo_ok < 3) halo_ok = 0;
  cp.halo = halo_ok >= 2;
  if (v2) conv3x3_tc_plan(cp, P.num_sms);
  // the pair kernel pays off where weights are re-streamed per tile (halved weight bytes per CTA);
  // layers whose weights stay resident in one CTA's smem are faster on the single-CTA fused kernel
  // (measured at 1080p, profiles/r1k: resident 9-K-block layers lose ~15 % on the pair kernel, the
  // 18-K-block 128->32 flow conv gains 28 %)
  if (want_pair && (!cp.v2_resident || cp.ktot / cp.kchunk >= 18 || P.conv3x3_2cta >= 2)) {
    ConvProblem alt = cp;
    alt.halo = halo_ok >= 1;
    alt.dual = P.conv3x3_dual;
    if (conv3x3_tc2_plan(alt, P.num_sms)) {
      cp = alt;
      pair = true;
    }
  }
  if (cp.halo) {  // the chosen kernel loads (tile_w + 2)-pixel-wide halo boxes
    for (int s = 0; s < cp.nsrc; ++s) {
      const SplitBuf* b = sources[s].buf;
      make_act_map(&cp.tm_a_hi[s], b->hi, b->B, b->H, b->W, b->C, box_h, box_w + 2, kc);
      make_act_map(&cp.tm_a_lo[s], b->lo, b->B, b->H, b->W, b->C, box_h, box_w + 2, kc);
    }
  }
  const size_t idx = P.h_probs.size();
  P.h_probs.push_back(cp);
  // issued tensor-core work: 3 passes over the padded K and the padded tile grid
  double k_issued = 0;  // skipped all-zero k-steps are not issued work
  for (size_t si = 0; si < pc.src_chunks.size(); ++si)
    k_issued += (double)pc.src_chunks[si] * pc.ntaps * ((v2 || pair) ? pc.src_ksteps[si] * 16 : pc.kchunk);
  P.mma_flops += (double)cp.passes * 2.0 * (double)cp.B * cp.tiles_y * cp.tiles_x * kTileM * k_issued *
                 (double)(((pc.cout + bn - 1) / bn) * bn);
  // algorithmic HBM bytes of this call site: every source plane it consumes read once, every destination plane written once
  double alg_bytes = 0;
  {
    const double px = (double)cp.B * cp.H * cp.W, planes_in = cp.passes == 1 ? 1.0 : 2.0;
    for (size_t si = 0; si < pc.src_chunks.size(); ++si) alg_bytes += px * pc.src_chunks[si] * pc.kchunk * 2.0 * planes_in;
    if (out) alg_bytes += px * pc.cout * 2.0 * (cp.out_lo_skip ? 1.0 : 2.0);
    if (pool_out) alg_bytes += px / 4.0 * pc.cout * 4.0;
    if (epi_mode == 2) alg_bytes += px * 12.0;
    if (!out && epi_mode != 2) alg_bytes += px * 24.0;   // flow heads: v_up read, residual and flow written
    alg_bytes += (double)pc.cout * pc.ktot * 2.0 * planes_in;
  }
  P.last_conv_bytes = alg_bytes;
  if (no_op) return idx;  // the caller launches this problem as part of a group
  Plan* pp = &P;
  const int impl = P.conv_impl;
  P.add_op(0, tag, [pp, idx, impl, v2, pair](cudaStream_t st) {
    if (impl == 1) return launch_conv_simt(pp->d_probs + idx, pp->h_probs[idx], st);
    if (pair) return launch_conv3x3_tc2(pp->d_probs + idx, pp->h_probs[idx], st);
    return v2 ? launch_conv3x3_tc(pp->d_probs + idx, pp->h_probs[idx], st)
              : launch_conv_tc(pp->d_probs + idx, pp->h_probs[idx], st);
  }, 2.0 * ref_macs_per_px * (double)cp.B * cp.H * cp.W, alg_bytes);
  return idx;
}

// eval/interpolator.py:30-63: network size (H, W) of an (h, w) frame and the offset of the frame inside it
static void padded_size(int h, int w, int align, int& H, int& W, int& off_y, int& off_x) {
  int ph = 0, pw = 0;
  if (align > 0) {
    ph = (h % align) ? align - h % align : 0;
    pw = (w % align) ? align - w % align : 0;
  }
  H = h + ph;
  W = w + pw;
  off_y = ph / 2;
  off_x = pw / 2;
}

// The reference graph accepts any size (VALID pooling floors, flows and the decoder resize to each level's size), and so
// does this engine when the handle option "any_size" is on.  Without it a padded size that is not a multiple of 64 (what
// the CLI default --align 64, eval/interpolator_cli.py:103, always gives) is refused.
static void check_supported_size(int H, int W, bool any_size) {
  if (!any_size && (H % 64 || W % 64))
    throw Error{FILM_ERR_UNSUPPORTED,
                "padded frame size must be a multiple of 64 (2^(pyramid_levels-1)) in this engine; use align=64"};
}

static std::unique_ptr<Plan> build_plan(const Model& M, int h, int w, int align, int conv_impl, bool keep_debug,
                                        int conv3x3_v2, int num_sms, int conv3x3_2cta, int conv3x3_halo,
                                        uint32_t onepass_mask, bool use_lanes, int fe_conv0_tc, bool any_size) {
  std::unique_ptr<Plan> pl(new Plan);
  Plan& P = *pl;
  P.fe_conv0_tc = fe_conv0_tc & 1;
  P.fuse_rgb_head = (fe_conv0_tc & 2) ? 0 : 1;
  P.conv3x3_dual = (fe_conv0_tc & 4) ? 1 : 0;
  P.plane_skip = (fe_conv0_tc & 8) ? 0 : 1;
  P.fuse_flow_head = (fe_conv0_tc & 64) ? 0 : ((fe_conv0_tc & 128) ? 2 : 1);
  P.mma_straight = (fe_conv0_tc & 16) ? 0 : 1;
  P.onepass_mask = onepass_mask;
  P.reuse = !keep_debug && !use_lanes && !(fe_conv0_tc & 32);
  P.h = h;
  P.w = w;
  P.conv_impl = conv_impl;
  P.conv3x3_v2 = conv3x3_v2;
  P.conv3x3_2cta = conv3x3_2cta;
  P.conv3x3_halo = conv3x3_halo;
  P.num_sms = num_sms;
  padded_size(h, w, align, P.H, P.W, P.off_y, P.off_x);
  check_supported_size(P.H, P.W, any_size);
  int Hs[kLevels], Ws[kLevels];
  for (int l = 0; l < kLevels; ++l) {
    Hs[l] = P.H >> l;
    Ws[l] = P.W >> l;
  }
  if (Hs[kLevels - 2] < 2 || Ws[kLevels - 2] < 2) throw Error{FILM_ERR_ARG, "frame too small"};

  P.xin = P.alloc<float>((int64_t)2 * h * w * 3, true);
  P.xout = P.alloc<float>((int64_t)h * w * 3, true);
  Plan* pp = &P;

  // ---- image pyramids (util.py:23-45), both images batched: img[l] = [2][H_l][W_l][3]
  float* img[kLevels];
  for (int l = 0; l < kLevels; ++l) img[l] = P.alloc<float>((int64_t)2 * Hs[l] * Ws[l] * 3, true);
  for (int k = 0; k < 2; ++k) {
    float* dst = img[0] + (int64_t)k * P.H * P.W * 3;
    const float* src = P.xin + (int64_t)k * h * w * 3;
    P.add_op(2, "pad_image", [=](cudaStream_t st) {
      return launch_pad_image(src, (int64_t)pp->w * 3, pp->h, pp->w, dst, pp->H, pp->W, pp->off_y, pp->off_x, st);
    });
  }
  // image pyramid (util.py:38-44): fused into the first conv of each scale when that conv is the FMA kernel (it has the
  // input patch in shared memory anyway); stand-alone pools otherwise (tensor-core first layer, validation path, lanes)
  const bool fuse_img_pool = P.conv_impl == 0 && !P.fe_conv0_tc && !use_lanes;
  for (int l = 0; l + 1 < kLevels && !fuse_img_pool; ++l) {
    const float* in = img[l];
    float* out = img[l + 1];
    const int hh = Hs[l], ww = Ws[l];
    P.add_op(2, "image_pool@L" + std::to_string(l), [=](cudaStream_t st) { return launch_image_pool(in, out, 2, hh, ww, st); });
  }

  const int tok_img = P.new_token();
  P.signal_last(tok_img);

  // ---- feature extractor (feature_extractor.py:125-193), Siamese: batch = image index
  SplitBuf* feat[kLevels];
  for (int l = 0; l < kLevels; ++l) feat[l] = P.split(2, Hs[l], Ws[l], feat_channels(l));
  static const int slice_off[4] = {0, 64, 192, 448};
  int tok_feat[kLevels][kSubLevels];  // token of the conv that completes slice j of feat[i + j]
  for (int i = 0; i < kLevels; ++i) {
    const int depth = (kLevels - i) < kSubLevels ? (kLevels - i) : kSubLevels;
    SplitBuf* pooled = nullptr;
    P.cur_lane = i;  // one lane per image-pyramid level (independent chains sharing only weights)
    if (i > 0) P.pending_waits = {tok_img};
    for (int j = 0; j < depth; ++j) {
      const int r = i + j, c = kFilters << j;
      SplitBuf* t1 = P.split(2, Hs[r], Ws[r], c);
      if (j == 0 && P.conv_impl == 0 && !P.fe_conv0_tc) {
        // cfeat_conv_0 (K = 27) on the FMA pipes, straight from the fp32 image level (exact fp32 arithmetic)
        const float* im = img[i];
        const int hh = Hs[r], ww = Ws[r];
        const float *w0 = M.conv0_w, *b0 = M.conv0_b;
        sp_t *oh = t1->hi, *ol = t1->lo;
        const bool lo_skip = P.plane_skip && ((P.onepass_mask >> fe_stage(i, 1)) & 1u);   // only reader: cfeat_conv_1 of this sub-tree
        float* pool_dst = (fuse_img_pool && i + 1 < kLevels) ? img[i + 1] : nullptr;   // next pyramid level
        P.add_op(2, std::string(pool_dst ? "fe_conv0+pool@L" : "fe_conv0@L") + std::to_string(r),
                 [=](cudaStream_t st) { return launch_fe_conv0(im, 2, hh, ww, w0, b0, oh, ol, lo_skip, pool_dst, st); },
                 2.0 * 27 * 64 * 2.0 * hh * ww, 2.0 * hh * ww * (3 * 4 + 64 * (lo_skip ? 2.0 : 4.0)));
      } else if (j == 0 && P.conv_impl == 0 && P.conv3x3_v2) {
        // cfeat_conv_0 on the persistent 3x3 tensor-core kernel: the image is widened to a 32-channel
        // split tensor (3 real channels), K = 9 taps x one 32-channel block
        const float* im = img[i];
        const int hh = Hs[r], ww = Ws[r];
        SplitBuf* im32 = P.split(2, hh, ww, 32, true);  // channels 8..31 stay zero: never recycled
        P.add_op(2, "fe_split32@L" + std::to_string(r),
                 [=](cudaStream_t st) { return launch_image_to_split32(im, 2, hh, ww, im32->hi, im32->lo, st); }, 0,
                 2.0 * hh * ww * (12 + 32.0));
        add_conv(P, "fe_conv0@L" + std::to_string(r), 27.0 * 64, M.fe0_3x3, {{im32, 0}}, 1, t1, 0, fe_stage(i, 0), fe_stage(i, 1));
      } else if (j == 0 && P.conv_impl == 0) {
        // generic-kernel variant: im2col-lite (27 -> 32 channels) + a 1x1 conv, K = 32
        const float* im = img[i];
        const int hh = Hs[r], ww = Ws[r];
        SplitBuf* col = P.split(2, hh, ww, 32, true);
        P.add_op(2, "fe_im2col@L" + std::to_string(r),
                 [=](cudaStream_t st) { return launch_im2col3x3(im, 2, hh, ww, col->hi, col->lo, st); }, 0,
                 2.0 * hh * ww * (12 + 128.0));
        add_conv(P, "fe_conv0@L" + std::to_string(r), 27.0 * 64, M.fe[0], {{col, 0}}, 1, t1, 0, fe_stage(i, 0), fe_stage(i, 1));
      } else if (j == 0) {
        const float* im = img[i];
        const int hh = Hs[r], ww = Ws[r];
        const float *w0 = M.conv0_w, *b0 = M.conv0_b;
        sp_t *oh = t1->hi, *ol = t1->lo;
        P.add_op(2, "fe_conv0@L" + std::to_string(r),
                 [=](cudaStream_t st) { return launch_conv0_c3(im, 2, hh, ww, w0, b0, oh, ol, 64, 0, st); },
                 2.0 * 27 * 64 * 2.0 * hh * ww, 2.0 * hh * ww * (3 + 64) * 4.0);
      } else {
        add_conv(P, "fe_conv" + std::to_string(2 * j) + "@L" + std::to_string(r), 9.0 * (c / 2) * c, M.fe[2 * j],
                 {{pooled, 0}}, 1, t1, 0, fe_stage(i, 2 * j), fe_stage(i, 2 * j + 1));
        P.release(pooled);  // consumed by this conv only
      }
      // second conv of the pair writes straight into the cascaded feature tensor slice
      // (replaces the tf.concat at feature_extractor.py:191)
      SplitBuf* pool_target = nullptr;
      const bool fuse_pool = (j < depth - 1) && P.conv_impl == 0 && P.conv3x3_v2;
      if (j < depth - 1) pool_target = P.split(2, Hs[r + 1], Ws[r + 1], c);
      add_conv(P, "fe_conv" + std::to_string(2 * j + 1) + "@L" + std::to_string(r), 9.0 * c * c, M.fe[2 * j + 1],
               {{t1, 0}}, 1, feat[r], slice_off[j], fe_stage(i, 2 * j + 1), ST_NONE, 1, 1, 0, 0,
               fuse_pool ? pool_target : nullptr);
      P.release(t1);
      tok_feat[i][j] = P.new_token();
      P.signal_last(tok_feat[i][j]);
      if (fuse_pool) {
        pooled = pool_target;  // written by the conv epilogue (feature_extractor.py:138-146 fused)
      } else if (j < depth - 1) {
        pooled = pool_target;
        const SplitBuf* f = feat[r];
        const SplitBuf* po = pooled;
        const int so = slice_off[j];
        P.add_op(2, "fe_pool@L" + std::to_string(r), [=](cudaStream_t st) {
          return launch_act_pool(f->hi, f->lo, f->C, so, 2, f->H, f->W, c, po->hi, po->lo, po->C, st);
        });
      }
    }
  }
  for (int l = 0; l < kLevels; ++l)
    for (int k = 0; k < 2; ++k)
      P.debug["feat" + std::to_string(k) + "/" + std::to_string(l)] =
          DebugTensor{true, feat[l]->hi + (int64_t)k * Hs[l] * Ws[l] * feat[l]->C,
                      feat[l]->lo + (int64_t)k * Hs[l] * Ws[l] * feat[l]->C, (int64_t)Hs[l] * Ws[l], feat[l]->C, 0,
                      feat[l]->C};

  // ---- pyramid flow estimator, both directions batched (pyramid_flow_estimator.py:125-163)
  // batch d = 0: forward (a = feat of image 0, b = image 1); d = 1: backward.
  float* v[kLevels];
  float* res[kLevels];
  for (int l = 0; l < kLevels; ++l) {
    v[l] = P.alloc<float>((int64_t)2 * Hs[l] * Ws[l] * 2, true);
    res[l] = P.alloc<float>((int64_t)2 * Hs[l] * Ws[l] * 2, true);
  }
  P.cur_lane = Plan::kNumLanes - 1;  // flow + fusion tail lane
  for (int l = kLevels - 1; l >= 0; --l) {
    const int p = l < kSpecialized ? l : kSpecialized;
    const int nf = kFlowFilters[p], C = feat_channels(l), hh = Hs[l], ww = Ws[l];
    // feat[l] is complete once every sub-pyramid contribution (image level i, depth l - i) is written
    for (int i = (l - (kSubLevels - 1) > 0 ? l - (kSubLevels - 1) : 0); i <= l; ++i) P.pending_waits.push_back(tok_feat[i][l - i]);
    const SplitBuf* second;  // second operand of concat(a, b)
    float* vup = nullptr;
    if (l == kLevels - 1) {
      // coarsest level: b = features of the other image, unwarped = the same tensor read at the other batch
      // index (ConvSrc::bswap: a TMA coordinate, no copy)
      second = nullptr;
    } else {
      SplitBuf* warped = P.split(2, hh, ww, C);
      vup = P.alloc<float>((int64_t)2 * hh * ww * 2);
      const float* vprev = v[l + 1];
      const SplitBuf* f = feat[l];
      const int hc = Hs[l + 1], wc = Ws[l + 1];
      float* vu = vup;
      // the warped features feed flow_conv0 of this level only: a single-pass consumer reads hi planes alone
      const bool hi_only = P.conv_impl == 0 && P.plane_skip && ((P.onepass_mask >> (ST_FLOW_L0 + l)) & 1u);
      const double wbytes = 2.0 * hh * ww * (double)C * (hi_only ? 4.0 : 8.0);
      P.add_op(1, "flow_warp@L" + std::to_string(l), [=](cudaStream_t st) {
        return launch_flow_warp(vprev, hc, wc, f->hi, f->lo, hh, ww, C, vu, warped->hi, warped->lo, hi_only, st);
      }, 0, wbytes);
      P.warp_bytes += wbytes;
      second = warped;
      // parity hooks: the flow-stage warp output (d = 0: features of image 1 warped by the forward flow) and the
      // upsampled flow it was gathered with
      for (int d = 0; d < 2; ++d) {
        P.debug["flow_warped" + std::to_string(d) + "/" + std::to_string(l)] =
            DebugTensor{true, warped->hi + (int64_t)d * hh * ww * C, warped->lo + (int64_t)d * hh * ww * C, (int64_t)hh * ww,
                        C, 0, C};
        P.debug["flow_vup" + std::to_string(d) + "/" + std::to_string(l)] =
            DebugTensor{false, vup + (int64_t)d * hh * ww * 2, nullptr, (int64_t)hh * ww, 2, 0, 2};
      }
    }
    const int cpad = round_up(nf, nf < kChunk ? 32 : kChunk);
    SplitBuf* c0 = P.split(2, hh, ww, cpad);
    SplitBuf* c1 = P.split(2, hh, ww, cpad);
    SplitBuf* c2 = P.split(2, hh, ww, cpad);
    const std::string lt = "@L" + std::to_string(l);
    std::vector<SrcRef> flow_src(2);
    flow_src[0].buf = feat[l];
    flow_src[0].c_off = 0;
    flow_src[1].buf = second ? second : feat[l];
    flow_src[1].c_off = 0;
    flow_src[1].bswap = second ? 0 : 1;
    add_conv(P, "flow_conv0" + lt, 9.0 * 2 * C * nf, M.flow[p][0], flow_src, 1, c0, 0, ST_FLOW_L0 + l, ST_FLOW_L0 + l);
    add_conv(P, "flow_conv1" + lt, 9.0 * nf * nf, M.flow[p][1], {{c0, 0}}, 1, c1, 0, ST_FLOW_L0 + l, ST_FLOW_L0 + l);
    // level 0 (32-filter predictor): conv_3, conv_4 and the residual add run in conv_2's epilogue.  The kernel supports
    // nf <= 64, but per-op timing (profiles/r2e) shows the 64-filter level 1 epilogue-bound (32 x 32 FMAs per thread):
    // 0.253 ms fused vs 0.224 ms as two launches, while level 0 gains (0.502 vs 0.566 ms) -- so only level 0 is fused.
    const bool fuse_head = P.conv_impl == 0 && P.conv3x3_v2 && P.fuse_flow_head && nf <= (P.fuse_flow_head >= 2 ? 64 : 32);
    if (fuse_head) {
      const size_t ci = add_conv(P, "flow_conv2+head" + lt, 9.0 * nf * nf + 1.0 * nf * (nf / 2) + (nf / 2) * 2.0, M.flow[p][2],
                                 {{c1, 0}}, 1, nullptr, 0, ST_FLOW_L0 + l, ST_NONE, 1, 1, 0, 0, nullptr, false, 3);
      ConvProblem& hp = P.h_probs[ci];
      if (hp.bn != nf || hp.pair) throw Error{FILM_ERR_UNSUPPORTED, "flow-head epilogue expects one N tile on the single-CTA kernel"};
      hp.head_w3 = M.flow_w3[p];
      hp.head_b3 = M.flow_b3[p];
      hp.head_w4 = M.flow_w4[p];
      hp.head_b4 = M.flow_b4[p];
      hp.head_vup = vup;
      hp.head_res = res[l];
      hp.head_v = v[l];
    } else {
      add_conv(P, "flow_conv2" + lt, 9.0 * nf * nf, M.flow[p][2], {{c1, 0}}, 1, c2, 0, ST_FLOW_L0 + l, ST_NONE);
    }
    if (fuse_head) {
    } else if (P.conv_impl == 1) {
      // CUDA-core validation path keeps the standalone fp32 head kernel
      const float *w3 = M.flow_w3[p], *b3 = M.flow_b3[p], *w4 = M.flow_w4[p], *b4 = M.flow_b4[p];
      float *rr = res[l], *vv = v[l];
      const float* vu = vup;
      const int npix = 2 * hh * ww;
      P.add_op(2, "flow_head" + lt, [=](cudaStream_t st) {
        return launch_flow_head(c2->hi, c2->lo, c2->C, nf, npix, w3, b3, w4, b4, vu, rr, vv, st);
      });
    } else {
      // conv_3 (1x1, nf -> nf/2) on the tensor cores; conv_4 + residual add in its epilogue
      const size_t ci = add_conv(P, "flow_head" + lt, 1.0 * nf * (nf / 2) + (nf / 2) * 2.0, M.flow_c3[p], {{c2, 0}}, 1,
                                 nullptr, 0, ST_NONE, ST_NONE);
      ConvProblem& hp = P.h_probs[ci];
      hp.epi_mode = 1;
      hp.head_w4 = M.flow_w4[p];
      hp.head_b4 = M.flow_b4[p];
      hp.head_vup = vup;
      hp.head_res = res[l];
      hp.head_v = v[l];
    }
    // this level's temporaries are dead; so are the feature levels the fusion stage does not warp
    P.release(second);
    P.release(vup);
    P.release(c0);
    P.release(c1);
    P.release(c2);
    if (l >= kFusionLevels) P.release(feat[l]);
    const int64_t np = (int64_t)hh * ww;
    P.debug["flow_fwd/" + std::to_string(l)] = DebugTensor{false, v[l], nullptr, np, 2, 0, 2};
    P.debug["flow_bwd/" + std::to_string(l)] = DebugTensor{false, v[l] + np * 2, nullptr, np, 2, 0, 2};
    P.debug["res_fwd/" + std::to_string(l)] = DebugTensor{false, res[l], nullptr, np, 2, 0, 2};
    P.debug["res_bwd/" + std::to_string(l)] = DebugTensor{false, res[l] + np * 2, nullptr, np, 2, 0, 2};
  }

  // ---- fusion-stage warps (interpolator.py:153-183).  v[l] already equals the synthesised flow
  // pyramid of util.py:106-117 (same arithmetic, same order), so that pass is not repeated.
  SplitBuf* wf[kFusionLevels];
  SplitBuf* side[kFusionLevels];
  for (int l = 0; l < kFusionLevels; ++l) {
    const int C = feat_channels(l), hh = Hs[l], ww = Ws[l];
    wf[l] = P.split(2, hh, ww, C);
    side[l] = P.split(1, hh, ww, kChunk, true);  // channels 16..63 stay zero: never recycled
    const float* vv = v[l];
    const float* im = img[l];
    const SplitBuf *f = feat[l], *o = wf[l], *sd = side[l];
    // consumers of the warped level: fusion_conv1 of the level (fusion_up of level 3 for the coarsest one)
    const int cons = l == kFusionLevels - 1 ? ST_FUS + 3 * (l - 1) : ST_FUS + 3 * l + 1;
    const bool hi_only = P.conv_impl == 0 && P.plane_skip && ((P.onepass_mask >> cons) & 1u);
    const double wbytes = 2.0 * hh * ww * (double)C * (hi_only ? 4.0 : 8.0);
    P.add_op(1, "fusion_warp@L" + std::to_string(l), [=](cudaStream_t st) {
      return launch_fusion_warp(vv, f->hi, f->lo, hh, ww, C, o->hi, o->lo, hi_only, st);
    }, 0, wbytes);
    P.add_op(2, "fusion_side@L" + std::to_string(l), [=](cudaStream_t st) {
      return launch_fusion_side(vv, im, hh, ww, sd->hi, sd->lo, sd->C, st);
    });
    P.warp_bytes += wbytes + 2.0 * hh * ww * 3.0 * 8.0;
    P.release(feat[l]);  // the fusion-stage warp is the last reader of the feature level
    P.debug["aligned_side/" + std::to_string(l)] =
        DebugTensor{true, sd->hi, sd->lo, (int64_t)hh * ww, sd->C, 0, 10};
    for (int k = 0; k < 2; ++k)
      P.debug["warped" + std::to_string(k) + "/" + std::to_string(l)] =
          DebugTensor{true, o->hi + (int64_t)k * hh * ww * C, o->lo + (int64_t)k * hh * ww * C, (int64_t)hh * ww, C, 0, C};
  }
  // The fusion convs see one frame (B = 1): views of the two warped feature batches.
  auto batch_view = [&](const SplitBuf* b, int k) {
    P.bufs.emplace_back(new SplitBuf(*b));
    SplitBuf* s = P.bufs.back().get();
    s->B = 1;
    s->hi = b->hi + (int64_t)k * b->H * b->W * b->C;
    s->lo = b->lo + (int64_t)k * b->H * b->W * b->C;
    return (const SplitBuf*)s;
  };

  // ---- fusion decoder (fusion.py:103-140)
  const SplitBuf* net = nullptr;
  for (int i = kFusionLevels - 2; i >= 0; --i) {
    const int nf = fusion_filters(i), hh = Hs[i], ww = Ws[i];
    const int cpad = round_up(nf, kChunk);
    SplitBuf* up = P.split(1, hh, ww, cpad);
    std::vector<SrcRef> up_src;
    if (i == kFusionLevels - 2)
      up_src = {{batch_view(wf[i + 1], 0), 0}, {batch_view(wf[i + 1], 1), 0}, {side[i + 1], 0}};
    else
      up_src = {{net, 0}};
    if (hh != 2 * Hs[i + 1] || ww != 2 * Ws[i + 1]) {
      // general path (a level of odd size below it: the fine grid is not twice the coarse one): every source is resized
      // by nearest neighbour onto the fine grid, then the plain 2x2 SAME conv runs there (both conv_impl values)
      const bool hi_only = P.conv_impl == 0 && P.plane_skip && ((P.onepass_mask >> (ST_FUS + 3 * i)) & 1u);
      std::vector<SplitBuf*> resized;
      for (size_t s = 0; s < up_src.size(); ++s) {
        const SplitBuf* src = up_src[s].buf;
        SplitBuf* dst = P.split(src->B, hh, ww, src->C);
        const double rbytes = (double)src->B * src->C * 2.0 * (hi_only ? 1.0 : 2.0) * ((double)hh * ww + (double)src->H * src->W);
        P.add_op(2, "fusion_resize" + std::to_string(s) + "@L" + std::to_string(i), [=](cudaStream_t st) {
          return launch_resize_nearest(src->hi, src->lo, src->B, src->H, src->W, src->C, dst->hi, dst->lo, hh, ww, hi_only, st);
        }, 0, rbytes);
        P.debug["fusion_resized" + std::to_string(s) + "/" + std::to_string(i)] =
            DebugTensor{true, dst->hi, dst->lo, (int64_t)hh * ww, dst->C, 0, dst->C};
        up_src[s].buf = dst;
        resized.push_back(dst);
      }
      add_conv(P, "fusion_up2x2@L" + std::to_string(i), 4.0 * M.fus_up_full[i].cin_ref * nf, M.fus_up_full[i], up_src, 0, up,
               0, ST_FUS + 3 * i, ST_FUS + 3 * i + 1);
      for (SplitBuf* r : resized) P.release(r);
    } else if (P.conv_impl == 0) {
      // the four parity classes share the grid: ONE launch, grid.z = class
      size_t first = 0;
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) {
          const size_t ci = add_conv(P, "", 0, M.fus_up[i][py * 2 + px], up_src, 0, up, 0, ST_FUS + 3 * i, ST_FUS + 3 * i + 1, 2, 2,
                                     py, px, nullptr, true);
          if (py == 0 && px == 0) first = ci;
        }
      P.h_probs[first].group = 4;
      const double up_bytes = 4.0 * P.last_conv_bytes;   // four parity classes, each reads the coarse sources once
      Plan* pq = &P;
      const double fl = 2.0 * 16.0 * M.fus_up[i][0].cin_ref * nf * (double)Hs[i + 1] * Ws[i + 1];
      P.add_op(0, "fusion_up@L" + std::to_string(i), [pq, first](cudaStream_t st) {
        return launch_conv_tc(pq->d_probs + first, pq->h_probs[first], st);
      }, fl, up_bytes);
    } else {
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px)
          add_conv(P, "fusion_up" + std::to_string(py * 2 + px) + "@L" + std::to_string(i),
                   4.0 * M.fus_up[i][0].cin_ref * nf, M.fus_up[i][py * 2 + px], up_src, 0, up, 0, ST_FUS + 3 * i,
                   ST_FUS + 3 * i + 1, 2, 2, py, px);
    }
    const bool fuse_rgb = (i == 0) && P.conv_impl == 0 && P.conv3x3_v2 && P.fuse_rgb_head && !keep_debug;
    SplitBuf* f1 = P.split(1, hh, ww, cpad);
    SplitBuf* f2 = fuse_rgb ? nullptr : P.split(1, hh, ww, cpad);
    add_conv(P, "fusion_conv1@L" + std::to_string(i), 9.0 * M.fus_c1[i].cin_ref * nf, M.fus_c1[i],
             {{batch_view(wf[i], 0), 0}, {batch_view(wf[i], 1), 0}, {side[i], 0}, {up, 0}}, 1, f1, 0, ST_FUS + 3 * i + 1,
             ST_FUS + 3 * i + 2);
    if (fuse_rgb) {
      // last decoder conv with the RGB head (fusion.py:100-101,139) and the crop (eval/interpolator.py:175) in its
      // epilogue: the 64-channel activation is never written
      const size_t ci = add_conv(P, "fusion_conv2+rgb@L0", 9.0 * nf * nf + 64.0 * 3, M.fus_c2[i], {{f1, 0}}, 1, nullptr, 0,
                                 ST_FUS + 3 * i + 2, ST_NONE, 1, 1, 0, 0, nullptr, false, 2);
      ConvProblem& hp = P.h_probs[ci];
      if (hp.cout != 64 || hp.bn != 64) throw Error{FILM_ERR_UNSUPPORTED, "RGB-head epilogue expects a 64-channel N tile"};
      hp.head_w4 = M.rgb_w;
      hp.head_b4 = M.rgb_b;
      hp.head_v = P.xout;
      hp.crop_y = P.off_y;
      hp.crop_x = P.off_x;
      hp.crop_h = P.h;
      hp.crop_w = P.w;
      hp.crop_pitch = (int64_t)P.w * 3;
    } else {
      add_conv(P, "fusion_conv2@L" + std::to_string(i), 9.0 * nf * nf, M.fus_c2[i], {{f1, 0}}, 1, f2, 0, ST_FUS + 3 * i + 2,
               i > 0 ? ST_FUS + 3 * (i - 1) : ST_NONE);
    }
    if (i == kFusionLevels - 2) P.release(wf[i + 1]);   // the coarsest aligned level fed fusion_up only
    else P.release(net);                                // previous level's output, consumed by fusion_up
    P.release(wf[i]);
    P.release(up);
    P.release(f1);
    net = f2;
    if (f2) P.debug["fusion_net/" + std::to_string(i)] = DebugTensor{true, f2->hi, f2->lo, (int64_t)hh * ww, f2->C, 0, nf};
    P.debug["fusion_up/" + std::to_string(i)] = DebugTensor{true, up->hi, up->lo, (int64_t)hh * ww, up->C, 0, nf};
  }
  {
    const float *rw = M.rgb_w, *rb = M.rgb_b;
    if (!(P.conv_impl == 0 && P.conv3x3_v2 && P.fuse_rgb_head && !keep_debug))
      P.add_op(2, "rgb_head", [=](cudaStream_t st) {
        return launch_rgb_head(net->hi, net->lo, net->C, pp->H, pp->W, rw, rb, pp->xout, (int64_t)pp->w * 3, pp->off_y,
                               pp->off_x, pp->h, pp->w, st);
      });
    P.debug["image"] = DebugTensor{false, P.xout, nullptr, (int64_t)h * w, 3, 0, 3};
    P.tok_end = P.new_token();
    P.signal_last(P.tok_end);
  }

  // reference-graph conv FLOPs (frame_interpolation_b200/spec.py conv_macs, SURVEY.md 8d)
  {
    double fe = 0, fl = 0, fu = 0;
    for (int i = 0; i < kLevels; ++i) {
      const int depth = (kLevels - i) < kSubLevels ? (kLevels - i) : kSubLevels;
      int cin = 3;
      for (int j = 0; j < depth; ++j) {
        const double c = kFilters << j;
        fe += (double)Hs[i + j] * Ws[i + j] * 9.0 * (cin * c + c * c);
        cin = (int)c;
      }
    }
    fe *= 2;
    for (int l = 0; l < kLevels; ++l) {
      const double nf = kFlowFilters[l < kSpecialized ? l : kSpecialized], cin = 2.0 * feat_channels(l);
      fl += (double)Hs[l] * Ws[l] * (9 * cin * nf + 18 * nf * nf + nf * nf / 2 + nf);
    }
    fl *= 2;
    for (int i = 0; i < kFusionLevels - 1; ++i) {
      const double nf = fusion_filters(i), a_c = 2.0 * (3 + feat_channels(i)) + 4;
      const double cc = (i == kFusionLevels - 2) ? 2.0 * (3 + feat_channels(i + 1)) + 4 : fusion_filters(i + 1);
      fu += (double)Hs[i] * Ws[i] * (4 * cc * nf + 9 * (a_c + nf) * nf + 9 * nf * nf);
    }
    fu += (double)Hs[0] * Ws[0] * 64 * 3;
    P.conv_flops = 2.0 * (fe + fl + fu);
  }

  if (P.reuse)
    for (auto& kv : P.debug)
      if (P.block_bytes.count((void*)kv.second.p0) ||
          kv.first.compare(0, 4, "feat") == 0 || kv.first.compare(0, 6, "warped") == 0 ||
          kv.first.compare(0, 11, "flow_warped") == 0 || kv.first.compare(0, 8, "flow_vup") == 0)
        kv.second.recycled = true;  // (batch views point into the middle of a recycled block)
  FILM_CUDA(cudaMalloc(&P.d_probs, P.h_probs.size() * sizeof(ConvProblem)));
  P.allocs.push_back(P.d_probs);
  FILM_CUDA(cudaMemcpy(P.d_probs, P.h_probs.data(), P.h_probs.size() * sizeof(ConvProblem), cudaMemcpyHostToDevice));
  (void)keep_debug;
  return pl;
}

}  // namespace film

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace film;

struct film_handle {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  std::unique_ptr<Model> model;
  std::map<std::string, std::unique_ptr<Plan>> plans;
  Plan* last_plan = nullptr;
  std::string err;
  int conv_impl = 0, use_graph = 1, keep_debug = 0, time_ops = 0;
  bool dev_events_valid = false;  // ev[1]/ev[2] bracket the last device-pointer call
  cudaStream_t copy_stream = nullptr;   // H2D / D2H of tile t+1 / t-1 overlaps the network call of tile t
  float* stage_in[2] = {nullptr, nullptr};
  float* stage_out[2] = {nullptr, nullptr};
  size_t stage_bytes = 0;
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr},
              ev_out[2] = {nullptr, nullptr};
  cudaStream_t lane_streams[Plan::kNumLanes] = {};  // lane 0 = the origin stream of the call
  std::vector<cudaEvent_t> token_events;
  cudaEvent_t fork_event = nullptr;
  int use_lanes = 0;   // stream lanes measured no gain at 1080p (smem-saturating kernels cannot co-reside)
  int conv3x3_v2 = 1;  // persistent tap-reuse kernel for 3x3 convs
  int conv3x3_2cta = 1;  // CTA-pair (cta_group::2) kernel for streamed-weight 3x3 convs on the large levels
  int conv3x3_halo = 3;  // wide halo boxes (one 10-px box per chunk serves nine taps): 0 off, 1 pair kernel, 2 both
                         // persistent kernels, 3 also the 32-channel-chunk layers (default: validated on hardware in
                         // round 2, -0.6 % / -2.0 % step time in two same-box A/Bs, profiles/r2c|r2d_variants_ab.md)
  uint32_t onepass_mask = kDefaultOnepassMask;  // precision plan (see `enum Stage`)
  int fe_conv0_tc = 0;  // cfeat_conv_0: 0 = register-tiled fp32 FMA kernel straight from the fp32 image (default: exact fp32,
                        // no widened image tensor; K = 27 is not tensor-core work), 1 = tensor-core kernel over the
                        // 32-channel-padded image (per-op timing of profiles/r2e: 0.78 ms over the 7 levels against 0.87 ms,
                        // i.e. 0.6 % of the step -- inside the run-to-run noise of the whole-step A/B)
  int fuse_rgb_head = 1;  // 1 = RGB head + crop in the epilogue of fusion_conv2@L0 (default), 0 = separate kernel
  int conv3x3_dual = 1;   // 1 = CTA-pair kernel serves two spatial items per streamed weight pass (default: -2.3 % step
                          // time in the same-box A/B of profiles/r2d_variants_ab.md)
  int plane_skip = 1, mma_straight = 1, arena_reuse = 1;   // round-2 optimisations, individually switchable (A/B, bisecting)
  int fuse_flow_head = 1;
  int any_size = 0;     // 1 = padded frame sizes that are not multiples of 64 are computed (the reference graph's general
                        // case); 0 (default) = they are refused with FILM_ERR_UNSUPPORTED.  Never changes a 64-aligned plan.
  uint8_t* u8_stage = nullptr;  // film_interpolate_u8: [x0][x1][out] on the device
  size_t u8_bytes = 0;
  int num_sms = 148;
  std::vector<cudaEvent_t> op_events;
  film_profile_t prof;
};

static std::string g_create_error;

static int fail(film_handle* h, const Error& e) noexcept {
  try {
    if (h) h->err = e.msg; else g_create_error = e.msg;
  } catch (...) {
  }
  return e.code;
}
// No C++ exception may unwind through an extern "C" entry point into the caller (ctypes / cgo / JNI):
// everything is turned into a status code; film_last_error() carries the text.
#define FILM_CATCH_ALL(h)                                                                                     \
  catch (const Error& e) { return fail(h, e); }                                                               \
  catch (const std::bad_alloc&) { return fail(h, Error{FILM_ERR_CUDA, "out of host memory"}); }               \
  catch (const std::exception& e) { return fail(h, Error{FILM_ERR_CUDA, std::string("internal error: ") + e.what()}); } \
  catch (...) { return fail(h, Error{FILM_ERR_CUDA, "unknown internal error"}); }

// Enqueues the whole schedule with `origin` as lane 0: fork the other lanes from it, express
// cross-lane dependencies with events, join everything back into `origin`.  Works both eagerly and
// under stream capture (the events become graph edges).
static void enqueue_plan(film_handle* h, Plan* P, cudaStream_t origin) {
  if (!h->use_lanes) {
    for (auto& op : P->ops) FILM_CUDA(op.fn(origin));
    return;
  }
  if (!h->fork_event) FILM_CUDA(cudaEventCreateWithFlags(&h->fork_event, cudaEventDisableTiming));
  for (int i = 1; i < Plan::kNumLanes; ++i)
    if (!h->lane_streams[i]) FILM_CUDA(cudaStreamCreateWithFlags(&h->lane_streams[i], cudaStreamNonBlocking));
  while ((int)h->token_events.size() < P->num_tokens) {
    cudaEvent_t e;
    FILM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    h->token_events.push_back(e);
  }
  auto lane_stream = [&](int lane) { return lane == 0 ? origin : h->lane_streams[lane]; };
  FILM_CUDA(cudaEventRecord(h->fork_event, origin));
  bool forked[Plan::kNumLanes] = {true};
  for (auto& op : P->ops) {
    cudaStream_t st = lane_stream(op.lane);
    if (!forked[op.lane]) {
      FILM_CUDA(cudaStreamWaitEvent(st, h->fork_event, 0));
      forked[op.lane] = true;
    }
    for (int t : op.waits) FILM_CUDA(cudaStreamWaitEvent(st, h->token_events[t], 0));
    FILM_CUDA(op.fn(st));
    for (int t : op.signals) FILM_CUDA(cudaEventRecord(h->token_events[t], st));
  }
  if (P->tok_end >= 0) FILM_CUDA(cudaStreamWaitEvent(origin, h->token_events[P->tok_end], 0));
}

// Frees every cached plan (graphs + activation arenas) once the handle's stream has drained.
static void drop_plans(film_handle* h) {
  cudaStreamSynchronize(h->stream);
  cudaDeviceSynchronize();
  (void)cudaGetLastError();
  h->last_plan = nullptr;
  h->dev_events_valid = false;
  h->plans.clear();
}

static Plan* get_plan(film_handle* h, int hh, int ww, int align) {
  {
    // checked before the cache lookup: a plan built while "any_size" was on must not serve a call made after it is off
    int H, W, oy, ox;
    padded_size(hh, ww, align, H, W, oy, ox);
    check_supported_size(H, W, h->any_size != 0);
  }
  char key[96];
  snprintf(key, sizeof(key), "%dx%d_a%d_i%d_v%d_l%d_p%d_h%d_m%x_d%d", hh, ww, align > 0 ? align : 0, h->conv_impl, h->conv3x3_v2,
           h->use_lanes, h->conv3x3_2cta, h->conv3x3_halo, h->onepass_mask, h->keep_debug * 256 + h->fuse_flow_head * 64 + h->arena_reuse * 32 + h->mma_straight * 16 + h->plane_skip * 8 + h->conv3x3_dual * 4 +
               h->fuse_rgb_head * 2 + h->fe_conv0_tc);
  auto it = h->plans.find(key);
  if (it != h->plans.end()) return it->second.get();
  std::unique_ptr<Plan> p;
  try {
    p = build_plan(*h->model, hh, ww, align, h->conv_impl, h->keep_debug != 0, h->conv3x3_v2, h->num_sms,
                   h->conv3x3_2cta, h->conv3x3_halo, h->onepass_mask, h->use_lanes != 0, h->fe_conv0_tc | (h->fuse_rgb_head ? 0 : 2) | (h->conv3x3_dual ? 4 : 0) | (h->plane_skip ? 0 : 8) |
                       (h->mma_straight ? 0 : 16) | (h->arena_reuse ? 0 : 32) | (h->fuse_flow_head ? 0 : 64) |
                       (h->fuse_flow_head >= 2 ? 128 : 0), h->any_size != 0);
  } catch (const Error& e0) {
    if (e0.code != FILM_ERR_CUDA) throw;  // only an allocation failure is worth a retry
    // Every cached shape keeps its activation arena (GBs at 1080p).  If a new shape does not fit next to
    // them, drop the cache and retry once before giving up.
    if (h->plans.empty()) throw;
    drop_plans(h);
    p = build_plan(*h->model, hh, ww, align, h->conv_impl, h->keep_debug != 0, h->conv3x3_v2, h->num_sms,
                   h->conv3x3_2cta, h->conv3x3_halo, h->onepass_mask, h->use_lanes != 0, h->fe_conv0_tc | (h->fuse_rgb_head ? 0 : 2) | (h->conv3x3_dual ? 4 : 0) | (h->plane_skip ? 0 : 8) |
                       (h->mma_straight ? 0 : 16) | (h->arena_reuse ? 0 : 32) | (h->fuse_flow_head ? 0 : 64) |
                       (h->fuse_flow_head >= 2 ? 128 : 0), h->any_size != 0);
  }
  if (h->use_graph) {
    cudaGraph_t g = nullptr;
    FILM_CUDA(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    try {
      enqueue_plan(h, p.get(), h->stream);
    } catch (const Error& err) {
      cudaStreamEndCapture(h->stream, &g);
      if (g) cudaGraphDestroy(g);
      (void)cudaGetLastError();
      throw Error{FILM_ERR_CUDA, "kernel launch failed during capture: " + err.msg};
    }
    FILM_CUDA(cudaStreamEndCapture(h->stream, &g));
    FILM_CUDA(cudaGraphInstantiate(&p->graph, g, 0));
    cudaGraphDestroy(g);
  }
  Plan* raw = p.get();
  h->plans[key] = std::move(p);
  return raw;
}

// runs the network of plan P on its xin -> xout (stream-ordered, not synchronised)
static void run_plan(film_handle* h, Plan* P, cudaStream_t st) {
  if (P->graph && !h->time_ops) {  // a captured graph can be replayed on any stream
    FILM_CUDA(cudaGraphLaunch(P->graph, st));
  } else {
    if (h->time_ops && st == h->stream) {
      // timed eager run: one event pair per op (bench.py's live per-kernel roofline numbers)
      const size_t n = P->ops.size();
      while (h->op_events.size() < n + 1) {
        cudaEvent_t e;
        FILM_CUDA(cudaEventCreate(&e));
        h->op_events.push_back(e);
      }
      FILM_CUDA(cudaEventRecord(h->op_events[0], st));
      for (size_t i = 0; i < n; ++i) {
        FILM_CUDA(P->ops[i].fn(st));
        FILM_CUDA(cudaEventRecord(h->op_events[i + 1], st));
      }
      FILM_CUDA(cudaStreamSynchronize(st));
      P->op_ms.assign(n, 0.f);
      for (size_t i = 0; i < n; ++i) FILM_CUDA(cudaEventElapsedTime(&P->op_ms[i], h->op_events[i], h->op_events[i + 1]));
    } else {
      enqueue_plan(h, P, st);
    }
  }
  h->last_plan = P;
}

extern "C" {

const char* film_version(void) {
  return "film_b200 0.2 sm_100a split=" FILM_SPLIT_NAME
         " mma=tcgen05.kind::f16, per-stage precision plan: 3-pass (hi*hi+hi*lo+lo*hi) or 1-pass (hi*hi)";
}

int film_create(film_handle** out, const char* weights_path, int device_ordinal) {
  if (!out || !weights_path) {
    g_create_error = "null argument";
    return FILM_ERR_ARG;
  }
  *out = nullptr;
  film_handle* h = nullptr;
  try {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
      throw Error{FILM_ERR_CUDA, "no CUDA device: the FILM B200 engine has no CPU fallback"};
    if (device_ordinal < 0 || device_ordinal >= ndev) throw Error{FILM_ERR_ARG, "bad device ordinal"};
    FILM_CUDA(cudaSetDevice(device_ordinal));
    cudaDeviceProp prop;
    FILM_CUDA(cudaGetDeviceProperties(&prop, device_ordinal));
    if (prop.major != 10)
      throw Error{FILM_ERR_CUDA, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                                     ", this engine is sm_100a-only (tcgen05/TMEM/TMA)"};
    h = new film_handle;
    h->device = device_ordinal;
    memset(&h->prof, 0, sizeof(h->prof));
    FILM_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    for (auto& e : h->ev) FILM_CUDA(cudaEventCreate(&e));
    FILM_CUDA(conv_tc_configure());
    FILM_CUDA(conv3x3_tc_configure());
    FILM_CUDA(conv3x3_tc2_configure());
    if (const char* e2 = getenv("FILM_2CTA")) h->conv3x3_2cta = atoi(e2);
    if (const char* e3 = getenv("FILM_HALO")) h->conv3x3_halo = atoi(e3);
    if (const char* e5 = getenv("FILM_FE0_TC")) h->fe_conv0_tc = atoi(e5) ? 1 : 0;
    if (const char* e6 = getenv("FILM_RGB_FUSE")) h->fuse_rgb_head = atoi(e6) ? 1 : 0;
    if (const char* e7 = getenv("FILM_DUAL")) h->conv3x3_dual = atoi(e7) ? 1 : 0;
    if (const char* e8 = getenv("FILM_PLANE_SKIP")) h->plane_skip = atoi(e8) ? 1 : 0;
    if (const char* e11 = getenv("FILM_FLOW_HEAD_FUSE")) h->fuse_flow_head = atoi(e11) < 0 ? 0 : (atoi(e11) > 2 ? 2 : atoi(e11));
    if (const char* e9 = getenv("FILM_STRAIGHT")) h->mma_straight = atoi(e9) ? 1 : 0;
    if (const char* e10 = getenv("FILM_ARENA_REUSE")) h->arena_reuse = atoi(e10) ? 1 : 0;
    if (const char* e4 = getenv("FILM_ONEPASS")) h->onepass_mask = (uint32_t)strtoul(e4, nullptr, 0);
    h->num_sms = prop.multiProcessorCount;
    WeightMap w = read_weight_file(weights_path);
    h->model.reset(new Model);
    h->model->load(w);
    *out = h;
    return FILM_OK;
  } catch (const Error& e) {
    fail(nullptr, e);
    if (h) film_destroy(h);
    return e.code;
  } catch (const std::exception& e) {
    fail(nullptr, Error{FILM_ERR_CUDA, std::string("internal error: ") + e.what()});
    if (h) film_destroy(h);
    return FILM_ERR_CUDA;
  } catch (...) {
    fail(nullptr, Error{FILM_ERR_CUDA, "unknown internal error"});
    if (h) film_destroy(h);
    return FILM_ERR_CUDA;
  }
}

void film_destroy(film_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  h->plans.clear();
  h->model.reset();
  for (auto& e : h->ev)
    if (e) cudaEventDestroy(e);
  for (auto& e : h->op_events) cudaEventDestroy(e);
  for (auto& e : h->token_events) cudaEventDestroy(e);
  for (int i = 0; i < 2; ++i) {
    if (h->stage_in[i]) cudaFree(h->stage_in[i]);
    if (h->stage_out[i]) cudaFree(h->stage_out[i]);
    for (cudaEvent_t e : {h->ev_in[i], h->ev_done[i], h->ev_free[i], h->ev_out[i]})
      if (e) cudaEventDestroy(e);
  }
  if (h->u8_stage) cudaFree(h->u8_stage);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->fork_event) cudaEventDestroy(h->fork_event);
  for (int i = 1; i < Plan::kNumLanes; ++i)
    if (h->lane_streams[i]) cudaStreamDestroy(h->lane_streams[i]);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

const char* film_last_error(film_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int film_set_option(film_handle* h, const char* name, int value) {
  if (!h || !name) return FILM_ERR_ARG;
  try {
  std::string n(name);
  if (n == "conv_impl") h->conv_impl = value;
  else if (n == "use_graph") h->use_graph = value;
  else if (n == "keep_debug") h->keep_debug = value;
  else if (n == "time_ops") h->time_ops = value;
  else if (n == "use_lanes") h->use_lanes = value;
  else if (n == "conv3x3_v2") h->conv3x3_v2 = value;
  else if (n == "conv3x3_2cta") h->conv3x3_2cta = value;
  else if (n == "conv3x3_halo") h->conv3x3_halo = value;
  else if (n == "onepass_mask") h->onepass_mask = (uint32_t)value & ((1u << ST_COUNT) - 1u);
  else if (n == "onepass_default") h->onepass_mask = kDefaultOnepassMask;
  else if (n == "fe_conv0_tc") h->fe_conv0_tc = value ? 1 : 0;
  else if (n == "fuse_rgb_head") h->fuse_rgb_head = value ? 1 : 0;
  else if (n == "conv3x3_dual") h->conv3x3_dual = value ? 1 : 0;
  else if (n == "plane_skip") h->plane_skip = value ? 1 : 0;
  else if (n == "fuse_flow_head") h->fuse_flow_head = value < 0 ? 0 : (value > 2 ? 2 : value);
  else if (n == "mma_straight") h->mma_straight = value ? 1 : 0;
  else if (n == "arena_reuse") h->arena_reuse = value ? 1 : 0;
  else if (n == "any_size") h->any_size = value ? 1 : 0;
  else if (n == "clear_plans") drop_plans(h);
  else {
    h->err = "unknown option " + n;
    return FILM_ERR_ARG;
  }
  return FILM_OK;
  }
  FILM_CATCH_ALL(h)
}

int film_stage_count(void) { return ST_COUNT; }

int film_stage_name(int stage, char* buf, int buf_size) {
  if (!buf || buf_size < 1 || stage < 0 || stage >= ST_COUNT) return FILM_ERR_ARG;
  try {
    const std::string n = stage_name(stage);
    snprintf(buf, (size_t)buf_size, "%s", n.c_str());
    return FILM_OK;
  } catch (...) {
    return FILM_ERR_CUDA;
  }
}

int film_get_option(film_handle* h, const char* name, int* value) {
  if (!h || !name || !value) return FILM_ERR_ARG;
  if (!strcmp(name, "onepass_mask")) *value = (int)h->onepass_mask;
  else if (!strcmp(name, "onepass_default")) *value = (int)kDefaultOnepassMask;
  else if (!strcmp(name, "conv3x3_halo")) *value = h->conv3x3_halo;
  else if (!strcmp(name, "conv3x3_2cta")) *value = h->conv3x3_2cta;
  else if (!strcmp(name, "keep_debug")) *value = h->keep_debug;
  else if (!strcmp(name, "any_size")) *value = h->any_size;
  else return FILM_ERR_ARG;
  return FILM_OK;
}

int film_synchronize(film_handle* h) {
  if (!h) return FILM_ERR_ARG;
  try {
    FILM_CUDA(cudaSetDevice(h->device));
    FILM_CUDA(cudaStreamSynchronize(h->stream));
    return FILM_OK;
  }
  FILM_CATCH_ALL(h)
}

extern "C++" {
// Double-buffered device staging for the multi-call paths (tiles, batches): [2 frames in] / [1 frame out]
static void ensure_staging(film_handle* h, size_t frame_bytes) {
  if (!h->copy_stream) FILM_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    if (!h->ev_in[i]) {
      FILM_CUDA(cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
      FILM_CUDA(cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
      FILM_CUDA(cudaEventCreateWithFlags(&h->ev_free[i], cudaEventDisableTiming));
      FILM_CUDA(cudaEventCreateWithFlags(&h->ev_out[i], cudaEventDisableTiming));
    }
  }
  if (h->stage_bytes >= frame_bytes) return;
  for (int i = 0; i < 2; ++i) {
    if (h->stage_in[i]) cudaFree(h->stage_in[i]);
    if (h->stage_out[i]) cudaFree(h->stage_out[i]);
    h->stage_in[i] = h->stage_out[i] = nullptr;
  }
  h->stage_bytes = 0;
  for (int i = 0; i < 2; ++i) {
    FILM_CUDA(cudaMalloc(&h->stage_in[i], 2 * frame_bytes));
    FILM_CUDA(cudaMalloc(&h->stage_out[i], frame_bytes));
  }
  h->stage_bytes = frame_bytes;
}

// Runs `n` independent network calls of plan P with copies overlapped: item i's inputs are fetched by
// `fetch(i, dst_x0, dst_x1, stream)` (host -> device staging) and its result is delivered by
// `deliver(i, src, stream)`; while item i computes on the handle's stream, item i+1 uploads and item
// i-1 downloads on the copy stream.
template <class Fetch, class Deliver>
static void run_pipelined(film_handle* h, Plan* P, int n, size_t frame_bytes, Fetch fetch, Deliver deliver) {
  ensure_staging(h, frame_bytes);
  cudaStream_t cs = h->copy_stream, ms = h->stream;
  FILM_CUDA(cudaStreamSynchronize(ms));
  FILM_CUDA(cudaStreamSynchronize(cs));
  for (int i = 0; i < n; ++i) {
    const int b = i & 1;
    // upload item i (its staging buffer was released by the compute of item i-2)
    if (i >= 2) FILM_CUDA(cudaStreamWaitEvent(cs, h->ev_free[b], 0));
    fetch(i, h->stage_in[b], (float*)((char*)h->stage_in[b] + frame_bytes), cs);
    FILM_CUDA(cudaEventRecord(h->ev_in[b], cs));
    // compute item i
    FILM_CUDA(cudaStreamWaitEvent(ms, h->ev_in[b], 0));
    FILM_CUDA(cudaMemcpyAsync(P->xin, h->stage_in[b], 2 * frame_bytes, cudaMemcpyDeviceToDevice, ms));
    FILM_CUDA(cudaEventRecord(h->ev_free[b], ms));
    run_plan(h, P, ms);
    if (i >= 2) FILM_CUDA(cudaStreamWaitEvent(ms, h->ev_out[b], 0));  // stage_out[b] drained by item i-2's download
    FILM_CUDA(cudaMemcpyAsync(h->stage_out[b], P->xout, frame_bytes, cudaMemcpyDeviceToDevice, ms));
    FILM_CUDA(cudaEventRecord(h->ev_done[b], ms));
    // download item i-1 (overlaps the compute of item i, already enqueued)
    if (i >= 1) {
      const int pb = (i - 1) & 1;
      FILM_CUDA(cudaStreamWaitEvent(cs, h->ev_done[pb], 0));
      deliver(i - 1, h->stage_out[pb], cs);
      FILM_CUDA(cudaEventRecord(h->ev_out[pb], cs));
    }
  }
  const int lb = (n - 1) & 1;
  FILM_CUDA(cudaStreamWaitEvent(cs, h->ev_done[lb], 0));
  deliver(n - 1, h->stage_out[lb], cs);
  FILM_CUDA(cudaStreamSynchronize(cs));
  FILM_CUDA(cudaStreamSynchronize(ms));
}

}  // extern "C++"

static void check_frame_args(const void* x0, const void* x1, const void* out, int B, int H, int W) {
  if (!x0 || !x1 || !out) throw Error{FILM_ERR_ARG, "null frame pointer"};
  if (B < 1 || H < 1 || W < 1) throw Error{FILM_ERR_ARG, "batch, height and width must be positive"};
}

static void fill_profile(film_handle* h, Plan* P, float ms_net, float ms_h2d, float ms_d2h) {
  film_profile_t& p = h->prof;
  p.last_call_ms = ms_net;
  p.last_h2d_ms = ms_h2d;
  p.last_d2h_ms = ms_d2h;
  p.conv_flops = P->conv_flops;
  p.mma_flops = P->mma_flops;
  p.warp_bytes = P->warp_bytes;
  p.kernel_launches = (int64_t)P->ops.size();
  p.arena_bytes = P->arena_bytes;
  p.padded_h = P->H;
  p.padded_w = P->W;
  p.used_graph = P->graph ? 1 : 0;
}

int film_interpolate(film_handle* h, const float* x0, const float* x1, const float* dt, int B, int H, int W,
                     int align, float* out) {
  if (!h) return FILM_ERR_ARG;
  (void)dt;  // ignored like the reference ignores `time` (models/film_net/interpolator.py:102,163)
  try {
    check_frame_args(x0, x1, out, B, H, W);
    FILM_CUDA(cudaSetDevice(h->device));
    (void)cudaGetLastError();
    Plan* P = get_plan(h, H, W, align);
    const size_t frame = (size_t)H * W * 3 * sizeof(float);
    float ms_net = 0, ms_h2d = 0, ms_d2h = 0;
    if (B > 1 && !h->time_ops) {
      // batch of pairs: uploads / downloads of neighbouring pairs overlap the network calls
      run_pipelined(h, P, B, frame,
                    [&](int b, float* d0, float* d1, cudaStream_t cs) {
                      FILM_CUDA(cudaMemcpyAsync(d0, (const char*)x0 + b * frame, frame, cudaMemcpyHostToDevice, cs));
                      FILM_CUDA(cudaMemcpyAsync(d1, (const char*)x1 + b * frame, frame, cudaMemcpyHostToDevice, cs));
                    },
                    [&](int b, const float* src, cudaStream_t cs) {
                      FILM_CUDA(cudaMemcpyAsync((char*)out + b * frame, src, frame, cudaMemcpyDeviceToHost, cs));
                    });
      fill_profile(h, P, 0.f, 0.f, 0.f);
      return FILM_OK;
    }
    for (int b = 0; b < B; ++b) {
      FILM_CUDA(cudaEventRecord(h->ev[0], h->stream));
      FILM_CUDA(cudaMemcpyAsync(P->xin, (const char*)x0 + b * frame, frame, cudaMemcpyHostToDevice, h->stream));
      FILM_CUDA(cudaMemcpyAsync((char*)P->xin + frame, (const char*)x1 + b * frame, frame, cudaMemcpyHostToDevice, h->stream));
      FILM_CUDA(cudaEventRecord(h->ev[1], h->stream));
      run_plan(h, P, h->stream);
      FILM_CUDA(cudaEventRecord(h->ev[2], h->stream));
      FILM_CUDA(cudaMemcpyAsync((char*)out + b * frame, P->xout, frame, cudaMemcpyDeviceToHost, h->stream));
      FILM_CUDA(cudaEventRecord(h->ev[3], h->stream));
      FILM_CUDA(cudaStreamSynchronize(h->stream));
      float t;
      FILM_CUDA(cudaEventElapsedTime(&t, h->ev[0], h->ev[1]));
      ms_h2d += t;
      FILM_CUDA(cudaEventElapsedTime(&t, h->ev[1], h->ev[2]));
      ms_net += t;
      FILM_CUDA(cudaEventElapsedTime(&t, h->ev[2], h->ev[3]));
      ms_d2h += t;
    }
    fill_profile(h, P, ms_net, ms_h2d, ms_d2h);
    return FILM_OK;
  }
  FILM_CATCH_ALL(h)
}

int film_interpolate_device(film_handle* h, const float* d_x0, const float* d_x1, int B, int H, int W,
                            int64_t in_pitch, int align, float* d_out, int64_t out_pitch, void* cuda_stream) {
  if (!h) return FILM_ERR_ARG;
  try {
    check_frame_args(d_x0, d_x1, d_out, B, H, W);
    if (in_pitch < (int64_t)W * 3 || out_pitch < (int64_t)W * 3) throw Error{FILM_ERR_ARG, "pitch smaller than a row"};
    FILM_CUDA(cudaSetDevice(h->device));
    (void)cudaGetLastError();
    Plan* P = get_plan(h, H, W, align);
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : h->stream;
    const size_t row = (size_t)W * 3 * sizeof(float);
    for (int b = 0; b < B; ++b) {
      // stage into the plan's fixed input buffers so the captured graph stays pointer-stable
      FILM_CUDA(cudaMemcpy2DAsync(P->xin, row, d_x0 + (int64_t)b * H * in_pitch, in_pitch * 4, row, H,
                                  cudaMemcpyDeviceToDevice, st));
      FILM_CUDA(cudaMemcpy2DAsync(P->xin + (int64_t)H * W * 3, row, d_x1 + (int64_t)b * H * in_pitch, in_pitch * 4, row, H,
                                  cudaMemcpyDeviceToDevice, st));
      FILM_CUDA(cudaEventRecord(h->ev[1], st));
      run_plan(h, P, st);
      FILM_CUDA(cudaEventRecord(h->ev[2], st));
      FILM_CUDA(cudaMemcpy2DAsync(d_out + (int64_t)b * H * out_pitch, out_pitch * 4, P->xout, row, row, H,
                                  cudaMemcpyDeviceToDevice, st));
    }
    fill_profile(h, P, -1.f, 0.f, 0.f);
    h->dev_events_valid = true;
    return FILM_OK;
  }
  FILM_CATCH_ALL(h)
}

int film_interpolate_tiled(film_handle* h, const float* x0, const float* x1, const float* dt, int H, int W, int align,
                           int block_h, int block_w, float* out) {
  if (!h) return FILM_ERR_ARG;
  (void)dt;
  try {
    check_frame_args(x0, x1, out, 1, H, W);
    if (block_h < 1 || block_w < 1) throw Error{FILM_ERR_ARG, "block shape must be positive"};
    // eval/interpolator.py:84-89
    if (H % block_h) throw Error{FILM_ERR_ARG, "block_height=" + std::to_string(block_h) + " should evenly divide height=" + std::to_string(H) + "."};
    if (W % block_w) throw Error{FILM_ERR_ARG, "block_width=" + std::to_string(block_w) + " should evenly divide width=" + std::to_string(W) + "."};
    FILM_CUDA(cudaSetDevice(h->device));
    const int ph = H / block_h, pw = W / block_w;
    Plan* P = get_plan(h, ph, pw, align);
    const size_t row = (size_t)pw * 3 * sizeof(float), full_row = (size_t)W * 3 * sizeof(float);
    float ms_net = 0, ms_h2d = 0, ms_d2h = 0;
    if (block_h * block_w > 1 && !h->time_ops) {
      // tiles in row-major order (eval/interpolator.py:199-202), each padded on its own; the strided
      // upload of tile t+1 and download of tile t-1 overlap the network call of tile t
      const size_t tile_bytes = (size_t)ph * pw * 3 * sizeof(float);
      auto tile_off = [&](int t) { return ((size_t)(t / block_w) * ph * W + (size_t)(t % block_w) * pw) * 3; };
      run_pipelined(h, P, block_h * block_w, tile_bytes,
                    [&](int t, float* d0, float* d1, cudaStream_t cs) {
                      FILM_CUDA(cudaMemcpy2DAsync(d0, row, x0 + tile_off(t), full_row, row, ph, cudaMemcpyHostToDevice, cs));
                      FILM_CUDA(cudaMemcpy2DAsync(d1, row, x1 + tile_off(t), full_row, row, ph, cudaMemcpyHostToDevice, cs));
                    },
                    [&](int t, const float* src, cudaStream_t cs) {
                      FILM_CUDA(cudaMemcpy2DAsync(out + tile_off(t), full_row, src, row, row, ph, cudaMemcpyDeviceToHost, cs));
                    });
      fill_profile(h, P, 0.f, 0.f, 0.f);
      return FILM_OK;
    }
    // tiles are processed in row-major order (eval/interpolator.py:199-202), each padded on its own
    for (int r = 0; r < block_h; ++r)
      for (int c = 0; c < block_w; ++c) {
        const size_t off = ((size_t)r * ph * W + (size_t)c * pw) * 3;
        FILM_CUDA(cudaEventRecord(h->ev[0], h->stream));
        FILM_CUDA(cudaMemcpy2DAsync(P->xin, row, x0 + off, full_row, row, ph, cudaMemcpyHostToDevice, h->stream));
        FILM_CUDA(cudaMemcpy2DAsync(P->xin + (size_t)ph * pw * 3, row, x1 + off, full_row, row, ph, cudaMemcpyHostToDevice, h->stream));
        FILM_CUDA(cudaEventRecord(h->ev[1], h->stream));
        run_plan(h, P, h->stream);
        FILM_CUDA(cudaEventRecord(h->ev[2], h->stream));
        FILM_CUDA(cudaMemcpy2DAsync(out + off, full_row, P->xout, row, row, ph, cudaMemcpyDeviceToHost, h->stream));
        FILM_CUDA(cudaEventRecord(h->ev[3], h->stream));
        FILM_CUDA(cudaStreamSynchronize(h->stream));
        float t;
        FILM_CUDA(cudaEventElapsedTime(&t, h->ev[0], h->ev[1]));
        ms_h2d += t;
        FILM_CUDA(cudaEventElapsedTime(&t, h->ev[1], h->ev[2]));
        ms_net += t;
        FILM_CUDA(cudaEventElapsedTime(&t, h->ev[2], h->ev[3]));
        ms_d2h += t;
      }
    fill_profile(h, P, ms_net, ms_h2d, ms_d2h);
    return FILM_OK;
  }
  FILM_CATCH_ALL(h)
}

extern "C++" {
// Shared body of film_interpolate_recursive / film_interpolate_recursive_u8.  `u8`: the two input frames and the
// 2^times + 1 output frames are 8-bit (eval/util.py:38-41 dequantisation on the way in, :51-52 quantisation on the
// way out, both on the device); the recursion itself always runs on the unquantised float32 mid-frames, like
// the reference (eval/util.py:85-91 passes the float mid-frame on, write_image quantises only what is saved).
static int recursive_impl(film_handle* h, const void* frame0, const void* frame1, int H, int W, int align,
                          int times_to_interpolate, void* out, bool u8) {
  if (!h) return FILM_ERR_ARG;
  try {
    check_frame_args(frame0, frame1, out, 1, H, W);
    if (times_to_interpolate < 0 || times_to_interpolate > 10) throw Error{FILM_ERR_ARG, "times_to_interpolate must be in [0, 10]"};
    FILM_CUDA(cudaSetDevice(h->device));
    (void)cudaGetLastError();
    Plan* P = get_plan(h, H, W, align);
    const int n = (1 << times_to_interpolate) + 1;
    const int64_t elems = (int64_t)H * W * 3;
    const size_t frame = (size_t)elems * sizeof(float);
    const size_t io_frame = u8 ? (size_t)elems : frame;   // bytes of one frame at the host boundary
    ensure_staging(h, 16);  // creates the copy stream
    std::vector<std::pair<int, cudaEvent_t>> frame_events;
    float* seq = nullptr;
    uint8_t* q = nullptr;   // u8 mode: [2 input frames][n output frames]
    FILM_CUDA(cudaMalloc(&seq, frame * n));
    if (u8 && cudaMalloc(&q, io_frame * (n + 2)) != cudaSuccess) {
      cudaFree(seq);
      throw Error{FILM_ERR_CUDA, "out of device memory for the 8-bit frame staging"};
    }
    cudaError_t e = cudaSuccess;
    auto slot = [&](int i) { return (float*)((char*)seq + frame * i); };
    auto qslot = [&](int i) { return q + io_frame * (size_t)(i + 2); };
    auto chk = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    chk(cudaEventRecord(h->ev[0], h->stream));
    if (u8) {
      chk(cudaMemcpyAsync(q, frame0, io_frame, cudaMemcpyHostToDevice, h->stream));
      chk(cudaMemcpyAsync(q + io_frame, frame1, io_frame, cudaMemcpyHostToDevice, h->stream));
      chk(launch_u8_to_f32(q, slot(0), elems, h->stream));
      chk(launch_u8_to_f32(q + io_frame, slot(n - 1), elems, h->stream));
    } else {
      chk(cudaMemcpyAsync(slot(0), frame0, frame, cudaMemcpyHostToDevice, h->stream));
      chk(cudaMemcpyAsync(slot(n - 1), frame1, frame, cudaMemcpyHostToDevice, h->stream));
    }
    chk(cudaEventRecord(h->ev[1], h->stream));
    // level-synchronous traversal of the binary tree of eval/util.py:62-91; every mid-frame stays in HBM
    for (int step = (n - 1) / 2; step >= 1 && e == cudaSuccess; step /= 2) {
      for (int i = step; i < n - 1 && e == cudaSuccess; i += 2 * step) {
        chk(cudaMemcpyAsync(P->xin, slot(i - step), frame, cudaMemcpyDeviceToDevice, h->stream));
        chk(cudaMemcpyAsync((char*)P->xin + frame, slot(i + step), frame, cudaMemcpyDeviceToDevice, h->stream));
        if (e == cudaSuccess) {
          try {
            run_plan(h, P, h->stream);
          } catch (...) {
            cudaStreamSynchronize(h->stream);
            for (auto& fe : frame_events) cudaEventDestroy(fe.second);
            cudaFree(seq);
            if (q) cudaFree(q);
            throw;
          }
        }
        chk(cudaMemcpyAsync(slot(i), P->xout, frame, cudaMemcpyDeviceToDevice, h->stream));
        if (u8) chk(launch_f32_to_u8(slot(i), qslot(i), elems, h->stream));
        if (e == cudaSuccess) {
          cudaEvent_t ev;
          chk(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
          chk(cudaEventRecord(ev, h->stream));
          frame_events.push_back({i, ev});
        }
      }
    }
    chk(cudaEventRecord(h->ev[2], h->stream));
    // everything is enqueued; download each mid-frame as soon as it exists (copy stream), while the
    // deeper recursion levels are still computing
    memcpy(out, frame0, io_frame);
    memcpy((char*)out + io_frame * (n - 1), frame1, io_frame);
    for (auto& fe : frame_events) {
      chk(cudaStreamWaitEvent(h->copy_stream, fe.second, 0));
      chk(cudaMemcpyAsync((char*)out + io_frame * fe.first, u8 ? (const void*)qslot(fe.first) : (const void*)slot(fe.first),
                          io_frame, cudaMemcpyDeviceToHost, h->copy_stream));
    }
    chk(cudaStreamSynchronize(h->copy_stream));
    chk(cudaEventRecord(h->ev[3], h->stream));
    chk(cudaStreamSynchronize(h->stream));
    for (auto& fe : frame_events) cudaEventDestroy(fe.second);
    float t_h2d = 0, t_net = 0, t_d2h = 0;
    if (e == cudaSuccess) {
      cudaEventElapsedTime(&t_h2d, h->ev[0], h->ev[1]);
      cudaEventElapsedTime(&t_net, h->ev[1], h->ev[2]);
      cudaEventElapsedTime(&t_d2h, h->ev[2], h->ev[3]);
    }
    cudaFree(seq);
    if (q) cudaFree(q);
    FILM_CUDA(e);
    fill_profile(h, P, t_net, t_h2d, t_d2h);
    h->prof.kernel_launches = (int64_t)P->ops.size() * (n - 2);
    return FILM_OK;
  }
  FILM_CATCH_ALL(h)
}
}  // extern "C++"

int film_interpolate_recursive(film_handle* h, const float* frame0, const float* frame1, int H, int W, int align,
                               int times_to_interpolate, float* out) {
  return recursive_impl(h, frame0, frame1, H, W, align, times_to_interpolate, out, false);
}

int film_interpolate_recursive_u8(film_handle* h, const uint8_t* frame0, const uint8_t* frame1, int H, int W, int align,
                                  int times_to_interpolate, uint8_t* out) {
  return recursive_impl(h, frame0, frame1, H, W, align, times_to_interpolate, out, true);
}

int film_interpolate_u8(film_handle* h, const uint8_t* x0, const uint8_t* x1, int B, int H, int W, int align,
                        uint8_t* out) {
  if (!h) return FILM_ERR_ARG;
  try {
    check_frame_args(x0, x1, out, B, H, W);
    FILM_CUDA(cudaSetDevice(h->device));
    (void)cudaGetLastError();
    Plan* P = get_plan(h, H, W, align);
    const int64_t elems = (int64_t)H * W * 3;
    if (h->u8_bytes < (size_t)elems * 3) {   // [x0][x1][out] 8-bit staging on the device
      if (h->u8_stage) cudaFree(h->u8_stage);
      h->u8_stage = nullptr;
      h->u8_bytes = 0;
      FILM_CUDA(cudaMalloc(&h->u8_stage, (size_t)elems * 3));
      h->u8_bytes = (size_t)elems * 3;
    }
    uint8_t* q = h->u8_stage;
    float ms_net = 0, ms_h2d = 0, ms_d2h = 0;
    for (int b = 0; b < B; ++b) {
      FILM_CUDA(cudaEventRecord(h->ev[0], h->stream));
      FILM_CUDA(cudaMemcpyAsync(q, x0 + (int64_t)b * elems, elems, cudaMemcpyHostToDevice, h->stream));
      FILM_CUDA(cudaMemcpyAsync(q + elems, x1 + (int64_t)b * elems, elems, cudaMemcpyHostToDevice, h->stream));
      FILM_CUDA(cudaEventRecord(h->ev[1], h->stream));
      FILM_CUDA(launch_u8_to_f32(q, P->xin, elems, h->stream));            // eval/util.py:38-41
      FILM_CUDA(launch_u8_to_f32(q + elems, P->xin + elems, elems, h->stream));
      run_plan(h, P, h->stream);
      FILM_CUDA(launch_f32_to_u8(P->xout, q + 2 * elems, elems, h->stream));  // eval/util.py:51-52
      FILM_CUDA(cudaEventRecord(h->ev[2], h->stream));
      FILM_CUDA(cudaMemcpyAsync(out + (int64_t)b * elems, q + 2 * elems, elems, cudaMemcpyDeviceToHost, h->stream));
      FILM_CUDA(cudaEventRecord(h->ev[3], h->stream));
      FILM_CUDA(cudaStreamSynchronize(h->stream));
      float t;
      FILM_CUDA(cudaEventElapsedTime(&t, h->ev[0], h->ev[1]));
      ms_h2d += t;
      FILM_CUDA(cudaEventElapsedTime(&t, h->ev[1], h->ev[2]));
      ms_net += t;
      FILM_CUDA(cudaEventElapsedTime(&t, h->ev[2], h->ev[3]));
      ms_d2h += t;
    }
    fill_profile(h, P, ms_net, ms_h2d, ms_d2h);
    return FILM_OK;
  }
  FILM_CATCH_ALL(h)
}

void* film_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 16, cudaHostAllocDefault) != cudaSuccess) {
    (void)cudaGetLastError();
    return nullptr;
  }
  return p;
}

void film_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

int film_profile(film_handle* h, film_profile_t* out) {
  if (!h || !out) return FILM_ERR_ARG;
  if (h->prof.last_call_ms < 0 && h->last_plan && h->dev_events_valid) {
    // device-pointer call: resolve the event pair lazily (blocks until that call finished)
    float t = 0;
    if (cudaEventSynchronize(h->ev[2]) == cudaSuccess && cudaEventElapsedTime(&t, h->ev[1], h->ev[2]) == cudaSuccess)
      h->prof.last_call_ms = t;
    else
      (void)cudaGetLastError();  // never leave a stale error for the next launch check
  }
  *out = h->prof;
  return FILM_OK;
}

int film_op_table(film_handle* h, char* buf, int64_t buf_size, int64_t* needed) {
  if (!h || !h->last_plan) return FILM_ERR_ARG;
  try {
  std::string out = "idx,category,name,ms,ref_flops,alg_bytes\n";
  Plan* P = h->last_plan;
  for (size_t i = 0; i < P->ops.size(); ++i) {
    char line[256];
    snprintf(line, sizeof(line), "%zu,%d,%s,%.6f,%.0f,%.0f\n", i, P->ops[i].category, P->ops[i].name.c_str(),
             i < P->op_ms.size() ? P->op_ms[i] : -1.f, P->ops[i].flops, P->ops[i].bytes);
    out += line;
  }
  if (needed) *needed = (int64_t)out.size() + 1;
  if (buf && buf_size > 0) {
    const size_t n = out.size() < (size_t)buf_size - 1 ? out.size() : (size_t)buf_size - 1;
    memcpy(buf, out.data(), n);
    buf[n] = 0;
  }
  return FILM_OK;
  }
  FILM_CATCH_ALL(h)
}

int film_debug_read(film_handle* h, const char* name, float* dst, int64_t* count) {
  if (!h || !name) return FILM_ERR_ARG;
  try {
    if (!h->last_plan) throw Error{FILM_ERR_ARG, "no call has been made yet"};
    auto it = h->last_plan->debug.find(name);
    if (it == h->last_plan->debug.end()) throw Error{FILM_ERR_ARG, std::string("unknown debug tensor ") + name};
    const DebugTensor& d = it->second;
    if (d.recycled)
      throw Error{FILM_ERR_ARG, std::string(name) + " lives in a recycled activation buffer: set option keep_debug = 1 "
                                                    "before the call to read intermediates"};
    const int64_t n = d.npix * d.Cn;
    if (count) *count = n;
    if (!dst) return FILM_OK;
    FILM_CUDA(cudaSetDevice(h->device));
    FILM_CUDA(cudaStreamSynchronize(h->stream));
    if (!d.split) {
      FILM_CUDA(cudaMemcpy(dst, d.p0, n * 4, cudaMemcpyDeviceToHost));
    } else {
      float* tmp;
      FILM_CUDA(cudaMalloc(&tmp, n * 4));
      cudaError_t e = launch_unsplit((const sp_t*)d.p0, (const sp_t*)d.p1, d.C, d.c_off, d.Cn, d.npix, tmp, h->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
      if (e == cudaSuccess) e = cudaMemcpy(dst, tmp, n * 4, cudaMemcpyDeviceToHost);
      cudaFree(tmp);
      FILM_CUDA(e);
    }
    return FILM_OK;
  }
  FILM_CATCH_ALL(h)
}

}  // extern "C"
