// svb_convnext.cu -- host side of the CoordinateRegressor forward: state-dict ingestion
// (timm ConvNeXt key scheme, SURVEY 8b), stem fold, 16-bit repack, TMA descriptors, launch plan.
//
// Replaces the device work of predict_ivd_locations' model(tensor)
// (spine_vision/datasets/classification/cropping.py:474-475) for the module built by
// load_localization_model (cropping.py:407-441).
#include "svb_convnext_kernels.cuh"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <algorithm>
#include <memory>
#include <string>
#include <thread>
#include <vector>

using namespace svb;

namespace svb {

static const double IMAGENET_MEAN[3] = {0.485, 0.456, 0.406};  // cropping.py:23
static const double IMAGENET_STD[3] = {0.229, 0.224, 0.225};   // cropping.py:24

struct BlockParams {
    float *wdw, *bdw, *lnw, *lnb, *b1, *b2, *gamma;
    float *grn_w = nullptr, *grn_b = nullptr;  // ConvNeXt-V2: GlobalResponseNorm weight / bias [4C]; gamma is all ones then
    float* s1 = nullptr;  // LayerNorm folded into fc1 (svb_model::ln_fold): s_n = sum_k r16(W1[n,k] g_k); b1 then holds t_n
    void *w1, *w2;  // 16-bit [4C][C], [C][4C]
    void* wdw16;    // depthwise taps as 16-bit [49][C] (the diagonal B operands of the tensor-core depthwise kernel)
    void* wtc = nullptr;  // dwconv_rawtc_kernel: [C/64][7 dy][112 = (dx, c')][64 k] 16-bit, zero except k % 16 == c' (see the kernel)
    CUtensorMap wdw_map, wdw16_map, w1_map, w2_map, wtc_map, wtc2_map;  // wtc2: 56-row boxes (each CTA of a pair stages half of a B matrix)
    CUtensorMap w1f_map, w2f_map;  // fused-MLP weight boxes: W1 {64, 32}, W2 {64, C/2} (each CTA of the pair stages half a tile)
};
struct DownParams {
    float *lnw, *lnb, *bias;
    void* w;  // 16-bit [Cout][4*Cin], k = (ky*2+kx)*Cin + ci
    CUtensorMap w_map;
};
struct ActPlan {  // tensor maps that depend on the workspace pointer and the micro-batch geometry
    const void* ws = nullptr;
    int nb = 0, H = 0, W = 0;
    CUtensorMap x_map[4];   // 4-D NHWC halo maps per stage
    CUtensorMap xr_map[4];  // the same for dwconv_raw_kernel (16-pixel-wide tiles: box {64, 22, 14, 1})
    CUtensorMap xr4_map[4]; // ... and its 4-row tiles (box {64, 22, 10, 1})
    CUtensorMap xtc_map[4]; // 4-D NHWC maps of the tensor-core depthwise kernel: box {64, W+6, rows, 1}, 128B swizzle
    int tc_rows[4] = {0, 0, 0, 0};  // rows per box; 0 = the stage runs the CUDA-core kernel
    CUtensorMap xtc2_map[4];         // dwconv_rawtc_kernel: box {64, W, 256 / W + 6, 1} (mode A) or {64, 32, 14, 1} (mode B), 128B swizzle
    int tc2[4] = {0, 0, 0, 0};       // 0 = the stage runs dwconv_raw_kernel; 1 = mode A; 2 = mode B
    CUtensorMap a_map[4];   // [M, C]   fc1 A operand
    CUtensorMap h_map[4];   // [M, 4C]  fc2 A operand
    CUtensorMap a2_map[4];  // [M/4, 4C_prev] downsample A operand (index = destination stage)
    CUtensorMap ox_map[4];  // [M, C]   32x32 epilogue boxes over the residual stream X (fc2 / downsample output, fc2 residual)
    CUtensorMap oh_map[4];  // [M, 4C]  32x32 epilogue boxes over the hidden buffer (fc1 output)
};

}  // namespace svb

struct svb_model {
    int dtype = SVB_BF16;
    int dims[4] = {0, 0, 0, 0};
    int depths[4] = {0, 0, 0, 0};
    int hid = 0, nout = 0;
    int device = 0;
    bool v2 = false;  // ConvNeXt-V2: GRN in every block's MLP, no layer scale
    int tc2_setting = 0x11, mlp_fused_setting = -1;  // SVB_DWCONV_TC2 / SVB_TC2_MODEB and SVB_MLP_FUSED as read at creation
    bool ln_fold = true;  // the block LayerNorm is folded into fc1 (dwconv_raw_kernel + GEMM_LNGELU); SVB_LN_FOLD=0 at creation: separate LN
    // two micro-batches in flight (svb_model_forward): odd micro-batches run on this stream with the second half of the
    // workspace, so that the ramp-up and tail of one chain's persistent kernels are back-filled by the other chain's CTAs
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t fork_ev = nullptr, join_ev = nullptr;
    void* slab = nullptr;
    size_t slab_bytes = 0;
    float *stem_w = nullptr, *stem_b = nullptr, *stem_lnw = nullptr, *stem_lnb = nullptr;
    float *stem_w3 = nullptr, *stem_b3 = nullptr;  // the un-folded stem [C0][3*4*4] + bias (svb_model_forward_f32: model(tensor) callers)
    std::vector<BlockParams> blocks[4];
    DownParams down[4];
    float *hn0w = nullptr, *hn0b = nullptr, *hn1w = nullptr, *hn1b = nullptr, *hw1 = nullptr, *hb1 = nullptr,
          *hw2 = nullptr, *hb2 = nullptr;
    ActPlan plans[4];  // (workspace half, micro-batch size) pairs in use: two chains x {full, tail} micro-batch
    int next_plan = 0;
    std::vector<cudaEvent_t> events;
    // every CUDA resource the handle owns goes here, so that an error return half-way through svb_model_create
    // (std::unique_ptr guard) releases the slab and the streams too
    ~svb_model() {
        for (auto e : events) cudaEventDestroy(e);
        if (aux_stream) { cudaStreamSynchronize(aux_stream); cudaStreamDestroy(aux_stream); }
        if (fork_ev) cudaEventDestroy(fork_ev);
        if (join_ev) cudaEventDestroy(join_ev);
        if (slab) cudaFree(slab);
    }
};

namespace svb {

static CUtensorMapDataType tmap_dtype(int dtype) {
    return dtype == SVB_FP16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
}
static uint16_t to16(float v, int dtype) {
    if (dtype == SVB_FP16) {
        float c = v > 65504.f ? 65504.f : (v < -65504.f ? -65504.f : v);
        __half h = __float2half_rn(c);
        uint16_t u;
        memcpy(&u, &h, 2);
        return u;
    }
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
}

// bulk fp32 -> 16-bit of the big MLP matrices (87 M of the 88 M parameters): bit arithmetic for bf16 (round to nearest even,
// NaN kept quiet) instead of a library call per element, spread over a few host threads -- model creation is what a short
// dataset run waits for
static void convert16_range(const float* src, uint16_t* dst, size_t n, int dtype) {
    if (dtype == SVB_FP16) {
        for (size_t i = 0; i < n; ++i) dst[i] = to16(src[i], dtype);
        return;
    }
    for (size_t i = 0; i < n; ++i) {
        uint32_t u;
        memcpy(&u, src + i, 4);
        if ((u & 0x7FFFFFFFu) > 0x7F800000u) { dst[i] = (uint16_t)((u >> 16) | 0x0040u); continue; }  // NaN
        u += 0x7FFFu + ((u >> 16) & 1u);
        dst[i] = (uint16_t)(u >> 16);
    }
}
static void convert16(const float* src, uint16_t* dst, size_t n, int dtype) {
    const size_t nt = n >= (1u << 20) ? 8 : 1;
    if (nt == 1) { convert16_range(src, dst, n, dtype); return; }
    std::vector<std::thread> th;
    const size_t per = (n + nt - 1) / nt;
    for (size_t t = 0; t < nt; ++t) {
        const size_t lo = t * per, hi = std::min(n, lo + per);
        if (lo < hi) th.emplace_back(convert16_range, src + lo, dst + lo, hi - lo, dtype);
    }
    for (auto& x : th) x.join();
}

// K-major 2-D operand map: rows x K, box {64, box_rows}, 128-byte swizzle
static int make_operand_map(CUtensorMap* map, int dtype, const void* base, uint64_t rows, uint64_t K, uint32_t box_rows) {
    const uint64_t dims[2] = {K, rows};
    const uint64_t strides[1] = {K * 2};
    const uint32_t box[2] = {64, box_rows};
    return encode_tmap(map, tmap_dtype(dtype), 2, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}
// epilogue box map: rows x N 16-bit row-major, box {32 columns, 32 rows}, 64-byte swizzle (gemm_kernel epilogue)
static int make_epilogue_map(CUtensorMap* map, int dtype, const void* base, uint64_t rows, uint64_t N) {
    const uint64_t dims[2] = {N, rows};
    const uint64_t strides[1] = {N * 2};
    const uint32_t box[2] = {32, 32};
    return encode_tmap(map, tmap_dtype(dtype), 2, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
}
// cudaFuncSetAttribute is a per-DEVICE setting: a process that drives a second GPU must opt in there too (the caches below are
// keyed by the current device; the flags only ever go from false to true, so a race costs a repeated call, nothing else)
constexpr int MAX_DEVICES = 64;
static int current_device_slot() {
    int d = 0;
    cudaGetDevice(&d);
    return (d >= 0 && d < MAX_DEVICES) ? d : 0;
}

static int gemm_bn(int N) { return (N % 256 == 0) ? 256 : 128; }
// CTA-pair (cta_group::2) tiles pay off when the K loop is long enough to hide the pair's tile hand-over
// (measured on B200, profiles/r01_gemm_shapes.txt): K >= 1024, or K >= 512 with at least two N tiles of 256.
// SVB_GEMM_CG=1|2 forces one kernel for A/B testing.
static int gemm_cg(int N, int K) {
    static int forced = -1;
    if (forced < 0) {
        const char* e = getenv("SVB_GEMM_CG");
        forced = (e && (e[0] == '1' || e[0] == '2')) ? (e[0] - '0') : 0;
    }
    if (forced) return forced;
    return (K >= 1024 || (K >= 512 && N >= 512)) ? 2 : 1;
}

// Co-resident ("half-SM") GEMM footprint, per stage: SVB_COEX is a string of four 0/1 flags (stage 0..3), e.g. "1110".
// A stage whose flag is set runs its fc1 / fc2 GEMMs as gemm_kernel<.., BN = 128, .., HALF = 1> (<= 113.5 KB of shared
// memory, 256 TMEM columns), so that the other micro-batch chain's depthwise-conv CTAs fit on the same SM.
static bool coex_stage(int s) {
    static int mask = -1;
    if (mask < 0) {
        mask = 0;
        const char* e = getenv("SVB_COEX");
        for (int i = 0; e && i < 4 && e[i]; ++i)
            if (e[i] == '1') mask |= 1 << i;
    }
    return s >= 0 && s < 4 && ((mask >> s) & 1);
}
// standalone svb_gemm: SVB_GEMM_HALF=1 selects the co-resident footprint (tests / experiments); read on every call
static bool gemm_half_env() {
    const char* e = getenv("SVB_GEMM_HALF");
    return e && e[0] == '1';
}
static int gemm_bn_for(int N, bool half) { return half ? 128 : gemm_bn(N); }
// SVB_LN_FOLD=0 (read when a model is created): keep the round-1 block -- dwconv_ln_kernel writes the NORMALISED fc1 operand,
// fc1 is a plain bias + GELU GEMM.  Default: folded (see dwconv_raw_kernel).
static bool ln_fold_env() {
    const char* e = getenv("SVB_LN_FOLD");
    return !(e && e[0] == '0');
}
// SVB_CARVEOUT=1: ask for the maximum shared-memory carve-out on the persistent kernels.  Two kernels whose preferred L1 /
// shared split differs cannot be resident on one SM at the same time (the split is an SM-wide setting), so a half-SM GEMM
// CTA and a depthwise CTA only ever share an SM when both ask for the same split.
static bool carveout_max() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("SVB_CARVEOUT");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v != 0;
}

// rows per depthwise tile: bounded by the 512 TMEM columns a CTA may hold (2 warps x TH pixels x NV values), see DwCfg
static int dw_th(int C) { return C >= 1536 ? 4 : (C >= 384 ? 8 : 16); }
// Programmatic dependent launch for the persistent kernels of the forward chain (depthwise conv + LN, GEMMs): the next
// kernel's CTAs are scheduled as SMs drain and run their set-up (barriers, TMEM allocation, descriptor prefetch) under the
// previous kernel's tail; griddepcontrol.wait in the kernels keeps the data dependence.  SVB_PDL=0 turns it off (A/B).
static bool pdl_enabled() {
    static int enabled = -1;
    if (enabled < 0) {
        const char* e = getenv("SVB_PDL");
        enabled = (e && e[0] == '0') ? 0 : 1;
    }
    return enabled != 0;
}
// fused fc1 -> GELU -> fc2 kernel (hidden activation kept on chip) for the widths whose accumulators fit TMEM:
// C = 128 / 256 (stages 0-1 of convnext_base).  Round 1 measured a tie with the un-fused pair and left it off; the reason turned
// out to be the MMA ISSUE path (its 32 / 64-clk MMAs each paid ~130 clk of ELECT / R2UR.BROADCAST latency).  With the warp-uniform
// issue loop: 644 -> 458 us at C = 128 and 402 -> 318 us at C = 256 per 64 images, against 596 / 335 us for the un-fused pair with
// the folded LayerNorm (profiles/r02w_fused_uniform.txt).  On by default for the LayerNorm-folded forward; SVB_MLP_FUSED=0 / 1
// forces it off / on (1 also in the un-folded forward).
// (read when a model is created and kept in the handle, like SVB_LN_FOLD / SVB_DWCONV_TC2: a test can create models under
// different settings in one process)
static int mlp_fused_env() {
    const char* e = getenv("SVB_MLP_FUSED");
    return e ? (e[0] == '1' ? 1 : 0) : -1;
}
static bool mlp_fused(int setting, int C) { return setting == 1 && (C == 128 || C == 256); }          // un-folded forward: opt-in
static bool mlp_fused_lnf(int setting, int C) { return setting != 0 && (C == 128 || C == 256); }      // folded forward: default
// Tensor-core depthwise kernel (shifted-view diagonal MMAs): C = 256 / 512 when one stage pair of halo tiles fits
// in shared memory.  SVB_DWCONV_TC=0 forces the CUDA-core kernel everywhere (A/B testing).
static int dw_tc_rows(int C, int W) {
    // Measured on B200 (profiles/r01_dwconv_tc.txt): correct, but 3x SLOWER than the FP32-pipe kernel -- every tap re-reads
    // its 128 x 16 operand slice from shared memory (16x redundant MMAs also mean 16x redundant operand traffic), so the
    // kernel is bound by the shared-memory operand feed, not the tensor pipe.  Kept as tested evidence; off by default.
    static int enabled = -1;
    if (enabled < 0) {
        const char* e = getenv("SVB_DWCONV_TC");
        enabled = (e && e[0] == '1') ? 1 : 0;
    }
    if (!enabled || (C != 256 && C != 512)) return 0;
    const int P = W + 6;
    const int NR = (2 * P + 132) / P + 6;
    if (P > 256 || NR > 256) return 0;
    const int smem = C == 512 ? DwTcCfg<512>::smem_bytes(P, NR) : DwTcCfg<256>::smem_bytes(P, NR);
    return smem <= 227 * 1024 ? NR : 0;
}

// dwconv_rawtc_kernel (the 7 x 7 taps as seven row-shifted tcgen05 MMAs with the stencil columns in N).  0 = the stage keeps
// dwconv_raw_kernel; 1 = mode A (W in {8, 16, 32}: units of whole image rows); 2 = mode B (32-lane windows with an x halo).
// SVB_DWCONV_TC2=0 switches it off, =2 also allows bf16 (8-bit tap mantissas; fp16 keeps 11).  SVB_TC2_MODEB=0 keeps mode B off.
static int dw_tc2_env() {  // bit 0..1: SVB_DWCONV_TC2 (default 1), bit 4: SVB_TC2_MODEB (default 1), bit 5: SVB_TC2_PAIR (default 0)
    const char* e = getenv("SVB_DWCONV_TC2");
    const char* b = getenv("SVB_TC2_MODEB");
    const char* p = getenv("SVB_TC2_PAIR");
    return ((e ? atoi(e) : 1) & 3) | (((b ? atoi(b) : 1) != 0) << 4) | (((p ? atoi(p) : 0) != 0) << 5);
}
static int dw_tc2_mode(int setting, int dtype, int C, int H, int W) {
    const int enabled = setting & 3, modeb = (setting >> 4) & 1;
    if (!enabled || (dtype != SVB_FP16 && enabled < 2)) return 0;
    if (C % 64 != 0 || C / 64 > num_sms() || H < 1 || W < 1) return 0;
    if (W == 8 || W == 16 || W == 32) return 1;
    return modeb ? 2 : 0;
}
// taps fp32 [49][C] -> B operands [C/64][7 dy][112 = dx * 16 + c'][64 = g * 16 + c] (16-bit): w[dy][dx][64 k + 16 g + c] where c == c'
static void pack_wtc(const float* taps, uint16_t* dst, int C, int dtype) {
    const int NCH = C / 64;
    memset(dst, 0, (size_t)NCH * 7 * 112 * 64 * 2);
    for (int k = 0; k < NCH; ++k)
        for (int dy = 0; dy < 7; ++dy)
            for (int dx = 0; dx < 7; ++dx)
                for (int g = 0; g < 4; ++g)
                    for (int c = 0; c < 16; ++c)
                        dst[(((size_t)k * 7 + dy) * 112 + dx * 16 + c) * 64 + g * 16 + c] = to16(taps[(size_t)(dy * 7 + dx) * C + k * 64 + g * 16 + c], dtype);
}
static int make_wtc_map(CUtensorMap* map, int dtype, const void* base, int C, int rows = 112) {
    const uint64_t dims[2] = {64, (uint64_t)(C / 64) * 7 * 112};
    const uint64_t strides[1] = {128};
    const uint32_t box[2] = {64, (uint32_t)rows};
    return encode_tmap(map, tmap_dtype(dtype), 2, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}
static int make_xtc2_map(CUtensorMap* map, int dtype, const void* base, int C, int nb, int H, int W, int mode) {
    const uint64_t uC = C;
    const uint64_t dims[4] = {uC, (uint64_t)W, (uint64_t)H, (uint64_t)nb};
    const uint64_t strides[3] = {uC * 2, (uint64_t)W * uC * 2, (uint64_t)H * W * uC * 2};
    const uint32_t box[4] = {64, (uint32_t)(mode == 1 ? W : 32), (uint32_t)(mode == 1 ? 256 / W + 6 : 14), 1};
    return encode_tmap(map, tmap_dtype(dtype), 4, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

struct HostWeights {
    std::map<std::string, const svb_weight_desc*> by_name;
    const svb_weight_desc* get(const std::string& n) const {
        auto it = by_name.find(n);
        return it == by_name.end() ? nullptr : it->second;
    }
};
static int64_t numel(const svb_weight_desc* w) {
    int64_t n = 1;
    for (int i = 0; i < w->ndim; ++i) n *= w->shape[i];
    return n;
}

// bump allocator over one device slab (two passes: size, then fill)
struct Slab {
    uint8_t* base = nullptr;
    size_t off = 0;
    std::vector<uint8_t> host;
    void* put(const void* src, size_t bytes) {
        off = align_up(off, 256);
        if (host.size() < off + bytes) host.resize(off + bytes);
        memcpy(host.data() + off, src, bytes);
        void* p = reinterpret_cast<void*>(off);  // offset now, rebased after upload
        off += bytes;
        return p;
    }
};
template <typename P> static void rebase(P*& p, uint8_t* base) { p = reinterpret_cast<P*>(base + reinterpret_cast<size_t>(p)); }

}  // namespace svb

extern "C" int svb_model_create(svb_model** out, const svb_weight_desc* weights, int n_weights, int dtype) {
    SVB_REQUIRE(out && weights && n_weights > 0, SVB_ERR_INVALID_ARG, "model_create: null/empty arguments");
    SVB_REQUIRE(dtype == SVB_BF16 || dtype == SVB_FP16, SVB_ERR_INVALID_ARG, "model_create: dtype %d", dtype);
    if (int rc = check_device_sm100()) return rc;
    *out = nullptr;
    HostWeights hwts;
    for (int i = 0; i < n_weights; ++i) {
        SVB_REQUIRE(weights[i].name && weights[i].data, SVB_ERR_INVALID_ARG, "model_create: weight %d has null name/data", i);
        hwts.by_name[weights[i].name] = &weights[i];
    }
    auto need = [&](const std::string& n, const svb_weight_desc** w) -> int {
        *w = hwts.get(n);
        SVB_REQUIRE(*w != nullptr, SVB_ERR_MISSING_WEIGHT, "model_create: state dict has no '%s'", n.c_str());
        return SVB_OK;
    };
#define NEED(var, name)                                   \
    const svb_weight_desc* var = nullptr;                 \
    if (int rc = need((name), &var)) return rc;

    svb_model* m = new svb_model();
    std::unique_ptr<svb_model> guard(m);
    m->dtype = dtype;
    SVB_CUDA_OK(cudaGetDevice(&m->device));

    // ---- geometry from the state dict -------------------------------------------------------
    NEED(stem_w, "backbone.stem.0.weight");
    SVB_REQUIRE(stem_w->ndim == 4 && stem_w->shape[1] == 3 && stem_w->shape[2] == 4 && stem_w->shape[3] == 4,
                SVB_ERR_UNSUPPORTED_MODEL, "stem conv must be [C0,3,4,4]");
    for (int s = 0; s < 4; ++s) {
        int d = 0;
        while (hwts.get("backbone.stages." + std::to_string(s) + ".blocks." + std::to_string(d) + ".conv_dw.weight")) ++d;
        SVB_REQUIRE(d > 0, SVB_ERR_MISSING_WEIGHT, "no blocks found for stage %d", s);
        m->depths[s] = d;
        const svb_weight_desc* g = hwts.get("backbone.stages." + std::to_string(s) + ".blocks.0.norm.weight");
        SVB_REQUIRE(g != nullptr, SVB_ERR_MISSING_WEIGHT, "model_create: state dict has no 'backbone.stages.%d.blocks.0.norm.weight'", s);
        m->dims[s] = (int)g->shape[0];
        SVB_REQUIRE(m->dims[s] % 32 == 0 && m->dims[s] >= 96 && m->dims[s] <= 2816, SVB_ERR_UNSUPPORTED_MODEL,
                    "stage %d width %d: this build supports the ConvNeXt widths (tiny / small 96..768, base 128..1024, "
                    "large 192..1536, xlarge 256..2048, v2_huge 352..2816)", s, m->dims[s]);
    }
    SVB_REQUIRE(m->dims[0] == (int)stem_w->shape[0], SVB_ERR_UNSUPPORTED_MODEL, "stem width != stage-0 width");
    m->v2 = hwts.get("backbone.stages.0.blocks.0.mlp.grn.weight") != nullptr;  // timm convnextv2_*: GRN instead of layer scale
    m->ln_fold = ln_fold_env();
    m->tc2_setting = dw_tc2_env();
    m->mlp_fused_setting = mlp_fused_env();
    SVB_REQUIRE(m->dims[0] == 96 || m->dims[0] == 128 || m->dims[0] == 192 || m->dims[0] == 256 || m->dims[0] == 352,
                SVB_ERR_UNSUPPORTED_MODEL, "stem width %d unsupported (supported: 96 tiny / small, 128 base, 192 large, 256 xlarge, "
                "352 v2_huge)", m->dims[0]);
    // the un-folded block (SVB_LN_FOLD=0) runs dwconv_ln_kernel, which parks all channels in TMEM and has no instance at the
    // convnextv2_huge widths: refuse such a model here rather than partway through a forward
    for (int s = 0; s < 4 && !m->ln_fold; ++s) {
        const int C = m->dims[s];
        SVB_REQUIRE(C == 96 || C == 128 || C == 192 || C == 256 || C == 384 || C == 512 || C == 768 || C == 1024 || C == 1536 || C == 2048,
                    SVB_ERR_UNSUPPORTED_MODEL, "stage %d width %d: SVB_LN_FOLD=0 (the un-folded LayerNorm block) does not support "
                    "this width; unset it to run v2_huge", s, C);
    }
    NEED(head_w1, "head.2.weight");
    NEED(head_w2, "head.5.weight");
    m->hid = (int)head_w1->shape[0];
    m->nout = (int)head_w2->shape[0];
    SVB_REQUIRE(head_w1->shape[1] == m->dims[3] && head_w2->shape[1] == m->hid && m->nout % 2 == 0,
                SVB_ERR_UNSUPPORTED_MODEL, "head shapes do not match generic.py:343-351");

    Slab slab;
    auto put_f32 = [&](const svb_weight_desc* w, int64_t expect) -> float* {
        if (numel(w) != expect) return nullptr;
        return static_cast<float*>(slab.put(w->data, (size_t)expect * 4));
    };
#define PUT_F32(dst, name, count)                                                                             \
    {                                                                                                         \
        NEED(_w, (name));                                                                                     \
        dst = put_f32(_w, (count));                                                                           \
        SVB_REQUIRE(numel(_w) == (int64_t)(count), SVB_ERR_UNSUPPORTED_MODEL, "'%s' has %lld elements, expected %lld", \
                    std::string(name).c_str(), (long long)numel(_w), (long long)(count));                     \
    }

    // ---- stem: fold /255, mean/std and the 3 identical input planes (SURVEY Appendix C) ------
    {
        const int C0 = m->dims[0];
        NEED(stem_b, "backbone.stem.0.bias");
        SVB_REQUIRE(numel(stem_b) == C0, SVB_ERR_UNSUPPORTED_MODEL, "stem bias size");
        std::vector<float> wf((size_t)C0 * 16), bf(C0);
        for (int co = 0; co < C0; ++co) {
            double bacc = stem_b->data[co];
            for (int p = 0; p < 16; ++p) {
                double acc = 0.0;
                for (int c = 0; c < 3; ++c) {
                    const double w = stem_w->data[((size_t)co * 3 + c) * 16 + p];
                    acc += w / (255.0 * IMAGENET_STD[c]);
                    bacc -= w * IMAGENET_MEAN[c] / IMAGENET_STD[c];
                }
                wf[(size_t)co * 16 + p] = (float)acc;
            }
            bf[co] = (float)bacc;
        }
        m->stem_w = static_cast<float*>(slab.put(wf.data(), wf.size() * 4));
        m->stem_b = static_cast<float*>(slab.put(bf.data(), bf.size() * 4));
        m->stem_w3 = static_cast<float*>(slab.put(stem_w->data, (size_t)C0 * 48 * 4));
        m->stem_b3 = static_cast<float*>(slab.put(stem_b->data, (size_t)C0 * 4));
        PUT_F32(m->stem_lnw, "backbone.stem.1.weight", C0);
        PUT_F32(m->stem_lnb, "backbone.stem.1.bias", C0);
    }
    // ---- stages ----------------------------------------------------------------------------
    std::vector<uint16_t> tmp16;
    for (int s = 0; s < 4; ++s) {
        const int C = m->dims[s];
        const std::string sp = "backbone.stages." + std::to_string(s) + ".";
        if (s > 0) {
            const int Cin = m->dims[s - 1];
            DownParams& d = m->down[s];
            PUT_F32(d.lnw, sp + "downsample.0.weight", Cin);
            PUT_F32(d.lnb, sp + "downsample.0.bias", Cin);
            PUT_F32(d.bias, sp + "downsample.1.bias", C);
            NEED(dw, sp + "downsample.1.weight");
            SVB_REQUIRE(numel(dw) == (int64_t)C * Cin * 4, SVB_ERR_UNSUPPORTED_MODEL, "downsample conv size (stage %d)", s);
            tmp16.resize((size_t)C * Cin * 4);
            for (int co = 0; co < C; ++co)
                for (int ci = 0; ci < Cin; ++ci)
                    for (int ky = 0; ky < 2; ++ky)
                        for (int kx = 0; kx < 2; ++kx)
                            tmp16[(size_t)co * 4 * Cin + (size_t)(ky * 2 + kx) * Cin + ci] =
                                to16(dw->data[(((size_t)co * Cin + ci) * 2 + ky) * 2 + kx], dtype);
            d.w = slab.put(tmp16.data(), tmp16.size() * 2);
        }
        m->blocks[s].resize(m->depths[s]);
        for (int j = 0; j < m->depths[s]; ++j) {
            BlockParams& bp = m->blocks[s][j];
            const std::string bn = sp + "blocks." + std::to_string(j) + ".";
            NEED(cw, bn + "conv_dw.weight");
            SVB_REQUIRE(numel(cw) == (int64_t)C * 49, SVB_ERR_UNSUPPORTED_MODEL, "conv_dw must be [C,1,7,7]");
            std::vector<float> taps((size_t)49 * C);  // [tap][C]
            for (int c = 0; c < C; ++c)
                for (int t = 0; t < 49; ++t) taps[(size_t)t * C + c] = cw->data[(size_t)c * 49 + t];
            bp.wdw = static_cast<float*>(slab.put(taps.data(), taps.size() * 4));
            tmp16.resize((size_t)49 * C);
            for (size_t i = 0; i < tmp16.size(); ++i) tmp16[i] = to16(taps[i], dtype);
            bp.wdw16 = slab.put(tmp16.data(), tmp16.size() * 2);
            if (C % 64 == 0) {  // B operands of dwconv_rawtc_kernel (98 KB per 64 channels)
                tmp16.resize((size_t)(C / 64) * 7 * 112 * 64);
                pack_wtc(taps.data(), tmp16.data(), C, dtype);
                bp.wtc = slab.put(tmp16.data(), tmp16.size() * 2);
            }
            PUT_F32(bp.bdw, bn + "conv_dw.bias", C);
            PUT_F32(bp.lnw, bn + "norm.weight", C);
            PUT_F32(bp.lnb, bn + "norm.bias", C);
            if (!m->ln_fold) PUT_F32(bp.b1, bn + "mlp.fc1.bias", 4 * C);
            PUT_F32(bp.b2, bn + "mlp.fc2.bias", C);
            if (m->v2) {
                std::vector<float> ones((size_t)C, 1.0f);
                bp.gamma = static_cast<float*>(slab.put(ones.data(), ones.size() * 4));
                PUT_F32(bp.grn_w, bn + "mlp.grn.weight", 4 * C);
                PUT_F32(bp.grn_b, bn + "mlp.grn.bias", 4 * C);
            } else {
                PUT_F32(bp.gamma, bn + "gamma", C);
            }
            NEED(w1, bn + "mlp.fc1.weight");
            NEED(w2, bn + "mlp.fc2.weight");
            SVB_REQUIRE(numel(w1) == (int64_t)4 * C * C && numel(w2) == (int64_t)4 * C * C, SVB_ERR_UNSUPPORTED_MODEL,
                        "mlp weights must be [4C,C] and [C,4C]");
            tmp16.resize((size_t)4 * C * C);
            if (m->ln_fold) {
                // fc1(LN(y)) = rstd * (W1 diag(g)) y - rstd mu * s + t:  W1g = r16(W1 * g) is the GEMM operand, s_n = sum_k W1g[n,k]
                // (of the ROUNDED values: what the tensor cores multiply), t_n = sum_k W1[n,k] lnb_k + b1_n (double -> float)
                NEED(lnw_w, bn + "norm.weight");
                NEED(lnb_w, bn + "norm.bias");
                NEED(b1_w, bn + "mlp.fc1.bias");
                SVB_REQUIRE(numel(b1_w) == (int64_t)4 * C, SVB_ERR_UNSUPPORTED_MODEL, "fc1 bias size");
                std::vector<float> wg((size_t)4 * C * C), sn((size_t)4 * C), tn((size_t)4 * C);
                const size_t rows = (size_t)4 * C;
                auto fold_rows = [&](size_t lo, size_t hi) {
                    for (size_t n = lo; n < hi; ++n) {
                        const float* wr = w1->data + n * C;
                        float* gr = wg.data() + n * C;
                        double t = b1_w->data[n];
                        for (int k = 0; k < C; ++k) { gr[k] = wr[k] * lnw_w->data[k]; t += (double)wr[k] * (double)lnb_w->data[k]; }
                        tn[n] = (float)t;
                    }
                };
                {
                    std::vector<std::thread> th;
                    const size_t nt = 8, per = (rows + nt - 1) / nt;
                    for (size_t q = 0; q < nt; ++q) { const size_t lo = q * per, hi = std::min(rows, lo + per); if (lo < hi) th.emplace_back(fold_rows, lo, hi); }
                    for (auto& x : th) x.join();
                }
                convert16(wg.data(), tmp16.data(), tmp16.size(), dtype);
                for (size_t n = 0; n < rows; ++n) {
                    double acc = 0.0;
                    for (int k = 0; k < C; ++k) {
                        const uint16_t u = tmp16[n * C + k];
                        float f;
                        if (dtype == SVB_FP16) { __half hh; memcpy(&hh, &u, 2); f = __half2float(hh); }
                        else { const uint32_t w32 = (uint32_t)u << 16; memcpy(&f, &w32, 4); }
                        acc += (double)f;
                    }
                    sn[n] = (float)acc;
                }
                bp.b1 = static_cast<float*>(slab.put(tn.data(), tn.size() * 4));
                bp.s1 = static_cast<float*>(slab.put(sn.data(), sn.size() * 4));
            } else {
                convert16(w1->data, tmp16.data(), tmp16.size(), dtype);
            }
            bp.w1 = slab.put(tmp16.data(), tmp16.size() * 2);
            convert16(w2->data, tmp16.data(), tmp16.size(), dtype);
            bp.w2 = slab.put(tmp16.data(), tmp16.size() * 2);
        }
    }
    // ---- head --------------------------------------------------------------------------------
    {
        const int C = m->dims[3];
        PUT_F32(m->hn0w, "backbone.head.norm.weight", C);
        PUT_F32(m->hn0b, "backbone.head.norm.bias", C);
        PUT_F32(m->hn1w, "head.0.weight", C);
        PUT_F32(m->hn1b, "head.0.bias", C);
        PUT_F32(m->hw1, "head.2.weight", (int64_t)m->hid * C);
        PUT_F32(m->hb1, "head.2.bias", m->hid);
        PUT_F32(m->hw2, "head.5.weight", (int64_t)m->nout * m->hid);
        PUT_F32(m->hb2, "head.5.bias", m->nout);
    }
    // ---- upload + rebase + weight tensor maps ------------------------------------------------
    m->slab_bytes = align_up(slab.off, 256);
    SVB_CUDA_OK(cudaMalloc(&m->slab, m->slab_bytes));
    SVB_CUDA_OK(cudaMemcpy(m->slab, slab.host.data(), slab.off, cudaMemcpyHostToDevice));
    uint8_t* base = static_cast<uint8_t*>(m->slab);
    rebase(m->stem_w, base); rebase(m->stem_b, base); rebase(m->stem_lnw, base); rebase(m->stem_lnb, base);
    rebase(m->stem_w3, base); rebase(m->stem_b3, base);
    rebase(m->hn0w, base); rebase(m->hn0b, base); rebase(m->hn1w, base); rebase(m->hn1b, base);
    rebase(m->hw1, base); rebase(m->hb1, base); rebase(m->hw2, base); rebase(m->hb2, base);
    for (int s = 0; s < 4; ++s) {
        const int C = m->dims[s];
        if (s > 0) {
            DownParams& d = m->down[s];
            rebase(d.lnw, base); rebase(d.lnb, base); rebase(d.bias, base);
            uint8_t* w = base + reinterpret_cast<size_t>(d.w);
            d.w = w;
            if (int rc = make_operand_map(&d.w_map, dtype, d.w, C, 4 * (uint64_t)m->dims[s - 1], gemm_bn(C) / gemm_cg(C, 4 * m->dims[s - 1]))) return rc;
        }
        for (auto& bp : m->blocks[s]) {
            rebase(bp.wdw, base); rebase(bp.bdw, base); rebase(bp.lnw, base); rebase(bp.lnb, base);
            rebase(bp.b1, base); rebase(bp.b2, base); rebase(bp.gamma, base);
            if (m->ln_fold) rebase(bp.s1, base);
            if (m->v2) { rebase(bp.grn_w, base); rebase(bp.grn_b, base); }
            bp.w1 = base + reinterpret_cast<size_t>(bp.w1);
            bp.w2 = base + reinterpret_cast<size_t>(bp.w2);
            bp.wdw16 = base + reinterpret_cast<size_t>(bp.wdw16);
            if (C % 64 == 0) {
                bp.wtc = base + reinterpret_cast<size_t>(bp.wtc);
                if (int rc = make_wtc_map(&bp.wtc_map, dtype, bp.wtc, C)) return rc;
                if (int rc = make_wtc_map(&bp.wtc2_map, dtype, bp.wtc, C, 56)) return rc;
            }
            {
                const uint64_t dims16[2] = {(uint64_t)C, 49};
                const uint64_t strides16[1] = {(uint64_t)C * 2};
                const uint32_t box16[2] = {64, 49};
                if (int rc = encode_tmap(&bp.wdw16_map, tmap_dtype(dtype), 2, bp.wdw16, dims16, strides16, box16,
                                         CU_TENSOR_MAP_SWIZZLE_NONE))
                    return rc;
            }
            if (int rc = make_operand_map(&bp.w1_map, dtype, bp.w1, 4 * (uint64_t)C, C, gemm_bn_for(4 * C, coex_stage(s)) / gemm_cg(4 * C, C))) return rc;
            if (int rc = make_operand_map(&bp.w2_map, dtype, bp.w2, C, 4 * (uint64_t)C, gemm_bn_for(C, coex_stage(s)) / gemm_cg(C, 4 * C))) return rc;
            if (C == 128 || C == 256) {
                if (int rc = make_operand_map(&bp.w1f_map, dtype, bp.w1, 4 * (uint64_t)C, C, 32)) return rc;
                if (int rc = make_operand_map(&bp.w2f_map, dtype, bp.w2, C, 4 * (uint64_t)C, C / 2)) return rc;
            }
            const uint64_t dims[2] = {(uint64_t)C, 49};
            const uint64_t strides[1] = {(uint64_t)C * 4};
            const uint32_t box[2] = {64, 49};
            if (int rc = encode_tmap(&bp.wdw_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, bp.wdw, dims, strides, box,
                                     CU_TENSOR_MAP_SWIZZLE_NONE))
                return rc;
        }
    }
    SVB_CUDA_OK(cudaStreamCreateWithFlags(&m->aux_stream, cudaStreamNonBlocking));
    SVB_CUDA_OK(cudaEventCreateWithFlags(&m->fork_ev, cudaEventDisableTiming));
    SVB_CUDA_OK(cudaEventCreateWithFlags(&m->join_ev, cudaEventDisableTiming));
    *out = guard.release();
    return SVB_OK;
#undef NEED
#undef PUT_F32
}

extern "C" int svb_model_destroy(svb_model* m) {
    if (!m) return SVB_OK;
    delete m;  // ~svb_model releases the streams, events and the weight slab
    return SVB_OK;
}

extern "C" int svb_model_info(const svb_model* m, int32_t out[10]) {
    SVB_REQUIRE(m && out, SVB_ERR_INVALID_ARG, "model_info: null argument");
    out[0] = m->nout / 2;
    out[1] = 2;
    for (int i = 0; i < 4; ++i) { out[2 + i] = m->dims[i]; out[6 + i] = m->depths[i]; }
    return SVB_OK;
}

namespace svb {

struct WsLayout {
    size_t x, a, h, stat, stat_part, grn_part, grn_scale, total;
};
static WsLayout ws_layout(const svb_model* m, int nb, int H, int W) {
    // stage 0 is the largest for every buffer (tokens/4, channels*2 per stage)
    const size_t t0 = (size_t)nb * (H / 4) * (W / 4);
    const size_t c0 = m->dims[0];
    WsLayout L;
    size_t o = 0;
    L.x = o; o += align_up(t0 * c0 * 2, 1024);
    L.a = o; o += align_up(t0 * c0 * 2, 1024);
    L.h = o; o += align_up(t0 * c0 * 4 * 2, 1024);
    L.stat = o; o += align_up(t0 * 8, 1024);  // (rstd, -mu rstd) per token: the folded LayerNorm of the current block
    // dwconv_rawtc_kernel's per-chunk partial (sum, sum of squares) [token][C / 64]: the largest stage (stage 0 for every
    // variant, but 352 / 64 floors to 5 chunks there, so it is not taken for granted)
    size_t part_words = 0;
    for (int s = 0, hs = H / 4, wsz = W / 4; s < 4; ++s, hs /= 2, wsz /= 2)
        part_words = std::max(part_words, (size_t)nb * hs * wsz * std::max<size_t>(1, (size_t)m->dims[s] / 64));
    L.stat_part = o; o += align_up(part_words * 8, 1024);
    L.grn_part = L.grn_scale = o;
    if (m->v2) {  // partial sums of squares [nb][ceil(tokens / GRN_ROWS)][4C] and scales [nb][4C]: the largest stage of each
        size_t part = 0, scale = 0;
        for (int s = 0, hs = H / 4, wsz = W / 4; s < 4; ++s, hs /= 2, wsz /= 2) {
            const size_t c4 = (size_t)m->dims[s] * 4;
            part = std::max(part, ceil_div<size_t>((size_t)hs * wsz, GRN_ROWS) * c4);
            scale = std::max(scale, c4);
        }
        L.grn_part = o; o += align_up((size_t)nb * part * 4, 1024);
        L.grn_scale = o; o += align_up((size_t)nb * scale * 4, 1024);
    }
    L.total = o;
    return L;
}

static int build_plan(svb_model* m, ActPlan* p, uint8_t* ws, int nb, int H, int W) {
    const WsLayout L = ws_layout(m, nb, H, W);
    int h = H / 4, w = W / 4;
    for (int s = 0; s < 4; ++s) {
        const uint64_t C = m->dims[s];
        const uint64_t M = (uint64_t)nb * h * w;
        {
            const uint64_t dims[4] = {C, (uint64_t)w, (uint64_t)h, (uint64_t)nb};
            const uint64_t strides[3] = {C * 2, (uint64_t)w * C * 2, (uint64_t)h * w * C * 2};
            const uint32_t box[4] = {64, 14, (uint32_t)(dw_th((int)C) + 6), 1};
            if (int rc = encode_tmap(&p->x_map[s], tmap_dtype(m->dtype), 4, ws + L.x, dims, strides, box,
                                     CU_TENSOR_MAP_SWIZZLE_NONE))
                return rc;
        }
        {
            const uint64_t dims[4] = {C, (uint64_t)w, (uint64_t)h, (uint64_t)nb};
            const uint64_t strides[3] = {C * 2, (uint64_t)w * C * 2, (uint64_t)h * w * C * 2};
            const uint32_t box[4] = {64, 22, 14, 1};  // DwRawCfg: TW + 6, TH + 6
            if (int rc = encode_tmap(&p->xr_map[s], tmap_dtype(m->dtype), 4, ws + L.x, dims, strides, box,
                                     CU_TENSOR_MAP_SWIZZLE_NONE))
                return rc;
            const uint32_t box4[4] = {64, 22, 10, 1};
            if (int rc = encode_tmap(&p->xr4_map[s], tmap_dtype(m->dtype), 4, ws + L.x, dims, strides, box4,
                                     CU_TENSOR_MAP_SWIZZLE_NONE))
                return rc;
        }
        p->tc_rows[s] = dw_tc_rows((int)C, w);
        if (p->tc_rows[s]) {
            const uint64_t dims[4] = {C, (uint64_t)w, (uint64_t)h, (uint64_t)nb};
            const uint64_t strides[3] = {C * 2, (uint64_t)w * C * 2, (uint64_t)h * w * C * 2};
            const uint32_t box[4] = {64, (uint32_t)(w + 6), (uint32_t)p->tc_rows[s], 1};
            if (int rc = encode_tmap(&p->xtc_map[s], tmap_dtype(m->dtype), 4, ws + L.x, dims, strides, box,
                                     CU_TENSOR_MAP_SWIZZLE_128B))
                return rc;
        }
        p->tc2[s] = m->ln_fold ? dw_tc2_mode(m->tc2_setting, m->dtype, (int)C, h, w) : 0;
        if (p->tc2[s]) {
            if (int rc = make_xtc2_map(&p->xtc2_map[s], m->dtype, ws + L.x, (int)C, nb, h, w, p->tc2[s])) return rc;
        }
        if (int rc = make_operand_map(&p->a_map[s], m->dtype, ws + L.a, M, C, 128)) return rc;
        if (int rc = make_operand_map(&p->h_map[s], m->dtype, ws + L.h, M, 4 * C, 128)) return rc;
        if (s > 0) {
            if (int rc = make_operand_map(&p->a2_map[s], m->dtype, ws + L.a, M, 4 * (uint64_t)m->dims[s - 1], 128)) return rc;
        }
        if (int rc = make_epilogue_map(&p->ox_map[s], m->dtype, ws + L.x, M, C)) return rc;
        if (int rc = make_epilogue_map(&p->oh_map[s], m->dtype, ws + L.h, M, 4 * C)) return rc;
        h /= 2;
        w /= 2;
    }
    p->ws = ws;
    p->nb = nb;
    p->H = H;
    p->W = W;
    return SVB_OK;
}

static int get_plan(svb_model* m, uint8_t* ws, int nb, int H, int W, ActPlan** out) {
    for (auto& p : m->plans)
        if (p.ws == ws && p.nb == nb && p.H == H && p.W == W) { *out = &p; return SVB_OK; }
    ActPlan* p = &m->plans[m->next_plan];
    m->next_plan = (m->next_plan + 1) & 3;
    if (int rc = build_plan(m, p, ws, nb, H, W)) { p->ws = nullptr; return rc; }
    *out = p;
    return SVB_OK;
}

// ---- launchers -------------------------------------------------------------------------------
template <typename T, int BN, int MODE, int CG, int HALF = 0>
static int launch_gemm_t(const CUtensorMap& a, const CUtensorMap& w, const CUtensorMap& out, const CUtensorMap& resid,
                         const float* bias, const float* gamma, int M, int N, int K, cudaStream_t st, const float2* rowstat = nullptr, int m0 = 0) {
    using Cfg = GemmCfg<BN, CG, HALF>;
    auto kern = gemm_kernel<T, BN, MODE, CG, HALF>;
    static bool attr_done[MAX_DEVICES] = {};
    const int dslot = current_device_slot();
    if (!attr_done[dslot]) {
        SVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        if (carveout_max()) SVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        attr_done[dslot] = true;
    }
    const int tiles = ceil_div(M - m0, 128 * CG) * ceil_div(N, BN);
    const int units = num_sms() / CG;  // CTAs, or CTA pairs
    const int grid = (tiles < units ? tiles : units) * CG;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(Cfg::NUM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    SVB_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, a, w, out, resid, bias, gamma, M, N, K, rowstat, m0));
    count_launch();
    return SVB_OK;
}
template <typename T>
static int launch_gemm(const CUtensorMap& a, const CUtensorMap& w, const CUtensorMap& out, const CUtensorMap& resid,
                       const float* bias, const float* gamma, int M, int N, int K, int mode, cudaStream_t st, bool half = false,
                       const float2* rowstat = nullptr, int m0 = 0) {
    SVB_REQUIRE(N % 32 == 0 && K % 8 == 0, SVB_ERR_INVALID_ARG, "gemm: N (%d) must be a multiple of 32, K (%d) of 8", N, K);
    SVB_REQUIRE(mode != GEMM_LNGELU || (rowstat && gamma && !half), SVB_ERR_INVALID_ARG, "gemm: the folded-LayerNorm mode needs rowstat and s_n");
    const int bn = gemm_bn_for(N, half);
    const int cg = gemm_cg(N, K);
    if (half) {
#define SVB_GEMM_HALF_CASE(MODE_, CG_)                                          \
    if (mode == MODE_ && cg == CG_)                                             \
        return launch_gemm_t<T, 128, MODE_, CG_, 1>(a, w, out, resid, bias, gamma, M, N, K, st, nullptr, m0);
        SVB_GEMM_HALF_CASE(GEMM_GELU, 2)
        SVB_GEMM_HALF_CASE(GEMM_RESID, 2)
        SVB_GEMM_HALF_CASE(GEMM_BIAS, 2)
        SVB_GEMM_HALF_CASE(GEMM_GELU, 1)
        SVB_GEMM_HALF_CASE(GEMM_RESID, 1)
        SVB_GEMM_HALF_CASE(GEMM_BIAS, 1)
#undef SVB_GEMM_HALF_CASE
        return set_error(SVB_ERR_INVALID_ARG, "gemm: unsupported mode %d", mode);
    }
#define SVB_GEMM_CASE(BN_, MODE_, CG_)                                          \
    if (bn == BN_ && mode == MODE_ && cg == CG_)                                \
        return launch_gemm_t<T, BN_, MODE_, CG_>(a, w, out, resid, bias, gamma, M, N, K, st, rowstat, m0);
    SVB_GEMM_CASE(256, GEMM_LNGELU, 2)
    SVB_GEMM_CASE(128, GEMM_LNGELU, 2)
    SVB_GEMM_CASE(256, GEMM_LNGELU, 1)
    SVB_GEMM_CASE(128, GEMM_LNGELU, 1)
    SVB_GEMM_CASE(256, GEMM_GELU, 2)
    SVB_GEMM_CASE(128, GEMM_GELU, 2)
    SVB_GEMM_CASE(256, GEMM_RESID, 2)
    SVB_GEMM_CASE(128, GEMM_RESID, 2)
    SVB_GEMM_CASE(256, GEMM_BIAS, 2)
    SVB_GEMM_CASE(128, GEMM_BIAS, 2)
    SVB_GEMM_CASE(256, GEMM_GELU, 1)
    SVB_GEMM_CASE(128, GEMM_GELU, 1)
    SVB_GEMM_CASE(256, GEMM_RESID, 1)
    SVB_GEMM_CASE(128, GEMM_RESID, 1)
    SVB_GEMM_CASE(256, GEMM_BIAS, 1)
    SVB_GEMM_CASE(128, GEMM_BIAS, 1)
#undef SVB_GEMM_CASE
    return set_error(SVB_ERR_INVALID_ARG, "gemm: unsupported mode %d", mode);
}

template <typename T, int C, bool LNF>
static int launch_mlp_fused_t(const CUtensorMap& a, const BlockParams& bp, const CUtensorMap& x, int M, cudaStream_t st, const float2* rowstat,
                              int stat_parts) {
    using Cfg = MlpCfg<C>;
    auto kern = mlp_fused_kernel<T, C, LNF>;
    static bool attr_done[MAX_DEVICES] = {};
    const int dslot = current_device_slot();
    if (!attr_done[dslot]) {
        SVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        attr_done[dslot] = true;
    }
    const int tiles = ceil_div(M, 256);
    const int pairs = num_sms() / 2;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((tiles < pairs ? tiles : pairs) * 2);
    cfg.blockDim = dim3(Cfg::NUM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    SVB_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, a, bp.w1f_map, bp.w2f_map, x, (const float*)bp.b1, (const float*)bp.b2,
                                   (const float*)bp.gamma, M, (const float*)bp.s1, rowstat, stat_parts));
    count_launch();
    return SVB_OK;
}
// rowstat != nullptr: the LayerNorm-folded form (bp.b1 = t_n, bp.s1 = s_n, a = the raw depthwise output); stat_parts > 0: rowstat is
// dwconv_rawtc_kernel's partial sums [M][stat_parts]
template <typename T>
static int launch_mlp_fused(const CUtensorMap& a, const BlockParams& bp, const CUtensorMap& x, int C, int M, cudaStream_t st,
                            const float2* rowstat = nullptr, int stat_parts = 0) {
    if (C == 128)
        return rowstat ? launch_mlp_fused_t<T, 128, true>(a, bp, x, M, st, rowstat, stat_parts) : launch_mlp_fused_t<T, 128, false>(a, bp, x, M, st, nullptr, 0);
    if (C == 256)
        return rowstat ? launch_mlp_fused_t<T, 256, true>(a, bp, x, M, st, rowstat, stat_parts) : launch_mlp_fused_t<T, 256, false>(a, bp, x, M, st, nullptr, 0);
    return set_error(SVB_ERR_UNSUPPORTED_MODEL, "fused MLP: unsupported width %d", C);
}

template <typename T, int C, int TH>
static int launch_dwconv_t(const CUtensorMap& x, const BlockParams& bp, void* out, int nb, int H, int W, cudaStream_t st) {
    using Cfg = DwCfg<C, TH>;
    auto kern = dwconv_ln_kernel<T, C, TH>;
    static bool attr_done[MAX_DEVICES] = {};
    const int dslot = current_device_slot();
    if (!attr_done[dslot]) {
        SVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        if (carveout_max()) SVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        attr_done[dslot] = true;
    }
    const int tx = ceil_div(W, Cfg::TW), ty = ceil_div(H, TH);
    const int tiles = nb * tx * ty;
    const int slots = num_sms() * Cfg::CTAS_PER_SM;  // persistent CTAs
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(tiles < slots ? tiles : slots);
    cfg.blockDim = dim3(Cfg::NUM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    SVB_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, x, bp.wdw_map, (const float*)bp.bdw, (const float*)bp.lnw, (const float*)bp.lnb,
                                   static_cast<T*>(out), H, W, tx, ty, tiles));
    count_launch();
    return SVB_OK;
}
template <typename T, int C, int TH>
static int launch_dwconv_raw_th(const CUtensorMap& x, const BlockParams& bp, void* out, float2* rowstat, int nb, int H, int W, cudaStream_t st, int b0) {
    using Cfg = DwRawCfg<C, TH>;
    auto kern = dwconv_raw_kernel<T, C, TH>;
    static bool attr_done[MAX_DEVICES] = {};
    const int dslot = current_device_slot();
    if (!attr_done[dslot]) {
        SVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        attr_done[dslot] = true;
    }
    const int tx = ceil_div(W, Cfg::TW), ty = ceil_div(H, TH);
    const int tiles = nb * tx * ty;
    const int slots = num_sms() * 2;  // persistent CTAs, two per SM
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(tiles < slots ? tiles : slots);
    cfg.blockDim = dim3(Cfg::NUM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    SVB_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, x, bp.wdw_map, (const float*)bp.bdw, static_cast<T*>(out), rowstat, H, W, tx, ty, tiles, b0));
    count_launch();
    return SVB_OK;
}
// images per sub-batch of stage s (see forward_chunk): SVB_SUB="a,b,c,d" overrides per stage (0 = the whole micro-batch).
// Default: as many images as keep the stage's hidden activation [tokens, 4C] x 16 bit near 32 MB per chain (two chains share L2),
// whole GEMM row tiles only.
static int sub_batch_images(int s, int nb, int tokens, int C) {
    static int forced[4] = {-1, -1, -1, -1};
    static bool parsed = false;
    if (!parsed) {
        parsed = true;
        const char* e = getenv("SVB_SUB");
        for (int i = 0; e && i < 4 && *e; ++i) {
            forced[i] = atoi(e);
            while (*e && *e != ',') ++e;
            if (*e == ',') ++e;
        }
    }
    int sub;
    if (forced[s] >= 0) sub = forced[s] == 0 ? nb : forced[s];
    else {
        // Measured on B200 (profiles/r02j_subbatch.txt, ms per 256 series): whole micro-batch 69.4; 8/32 images 70.5; 4/16 72.3;
        // 2/8 72.6; 1/4 75.8.  The hidden tensor does stay in L2, but launches of 8..64 tiles per SM lose more to their tails
        // and to the second chain's evictions than the HBM round trip costs: off unless SVB_SUB asks for it.
        (void)tokens; (void)C;
        return nb;
    }
    if (sub < 1) sub = 1;
    while (sub < nb && ((long long)sub * tokens) % 256 != 0) ++sub;  // whole 256-row tile pairs
    return sub < nb ? sub : nb;
}

template <typename T>
static int launch_dwconv_rawtc(const CUtensorMap& x, const BlockParams& bp, void* out, float2* rowstat, float2* stat_part, int C, int nb, int H,
                               int W, int mode, cudaStream_t st, int b0 = 0, bool finalize = true, bool pair = false) {
    // rowstat / stat_part address the micro-batch's first token; images [b0, b0 + nb) are written.  finalize = false: the consumer
    // (mlp_fused_kernel) adds the partial sums up itself.  pair: the cta_group::2 variant (two units at a time per CTA pair)
    using Cfg = DwTc2Cfg;
    static bool attr_done[MAX_DEVICES] = {};
    const int dslot = current_device_slot();
    if (!attr_done[dslot]) {
        SVB_CUDA_OK(cudaFuncSetAttribute(dwconv_rawtc_kernel<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        SVB_CUDA_OK(cudaFuncSetAttribute(dwconv_rawtc_kernel<T, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        attr_done[dslot] = true;
    }
    const int NCH = C / 64;
    const int rowpx = mode == 1 ? W : 32, nwin = mode == 1 ? 1 : ceil_div(W, 26);
    const int units_y = ceil_div(H, mode == 1 ? 256 / W : 8);
    const int num_units = nb * nwin * units_y;
    const int cg = pair ? 2 : 1;
    int per_chunk = num_sms() / cg / NCH;  // CTAs (or CTA pairs) per channel chunk
    if (per_chunk > ceil_div(num_units, cg)) per_chunk = ceil_div(num_units, cg);
    if (per_chunk < 1) return set_error(SVB_ERR_UNSUPPORTED_MODEL, "dwconv (tensor core): %d channel chunks do not fit %d SMs", NCH, num_sms());
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(NCH * per_chunk * cg));
    cfg.blockDim = dim3(Cfg::NUM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = 2;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.attrs = pdl_enabled() ? attr : attr + 1;
    cfg.numAttrs = (pdl_enabled() ? 1 : 0) + (pair ? 1 : 0);
    if (pair) {
        SVB_CUDA_OK(cudaLaunchKernelEx(&cfg, dwconv_rawtc_kernel<T, 2>, x, bp.wtc2_map, (const float*)bp.bdw, static_cast<T*>(out), stat_part, C, H, W, rowpx,
                                       nwin, units_y, num_units, b0));
    } else {
        SVB_CUDA_OK(cudaLaunchKernelEx(&cfg, dwconv_rawtc_kernel<T, 1>, x, bp.wtc_map, (const float*)bp.bdw, static_cast<T*>(out), stat_part, C, H, W, rowpx,
                                       nwin, units_y, num_units, b0));
    }
    count_launch();
    if (finalize) {
        const long long t0 = (long long)b0 * H * W, tokens = (long long)nb * H * W;
        cudaLaunchConfig_t fc{};
        fc.gridDim = dim3((unsigned)ceil_div<long long>(tokens, 256));
        fc.blockDim = dim3(256);
        fc.stream = st;
        fc.attrs = attr;
        fc.numAttrs = pdl_enabled() ? 1 : 0;
        SVB_CUDA_OK(cudaLaunchKernelEx(&fc, ln_stat_finalize_kernel, (const float2*)(stat_part + t0 * NCH), rowstat + t0, tokens, NCH, 1.0f / (float)C));
        count_launch();
    }
    return SVB_OK;
}

// rows per tile: 8, or 4 when 8-row tiles would leave most of the 2 x 148 CTA slots empty (the last stage: 16 x 16 tokens per image)
static int dw_raw_th(int nb, int H, int W) { return nb * ceil_div(W, 16) * ceil_div(H, 8) >= num_sms() * 3 / 2 ? 8 : 4; }
// 704, 1408 and 2816 channels (convnextv2_huge stages 1-3) take TH = 4 always: at TH = 8 they need more than the 128 registers of two CTAs
// per SM and spill (44 B of stores, 80 B of loads per thread under ptxas 12.9)
template <typename T, int C>
static int launch_dwconv_raw_t(const CUtensorMap& x8, const CUtensorMap& x4, const BlockParams& bp, void* out, float2* rowstat, int nb, int H, int W,
                               cudaStream_t st, int b0) {
    constexpr bool th8_spills = C == 704 || C == 1408 || C == 2816;
    if constexpr (!th8_spills)
        if (dw_raw_th(nb, H, W) == 8) return launch_dwconv_raw_th<T, C, 8>(x8, bp, out, rowstat, nb, H, W, st, b0);
    return launch_dwconv_raw_th<T, C, 4>(x4, bp, out, rowstat, nb, H, W, st, b0);
}
template <typename T>
static int launch_dwconv_raw(const CUtensorMap& x, const CUtensorMap& x4, const BlockParams& bp, void* out, float2* rowstat, int C, int nb, int H, int W, cudaStream_t st,
                             int b0 = 0) {
    switch (C) {
        case 128: return launch_dwconv_raw_t<T, 128>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 256: return launch_dwconv_raw_t<T, 256>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 512: return launch_dwconv_raw_t<T, 512>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 1024: return launch_dwconv_raw_t<T, 1024>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 2048: return launch_dwconv_raw_t<T, 2048>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 96: return launch_dwconv_raw_t<T, 96>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 192: return launch_dwconv_raw_t<T, 192>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 384: return launch_dwconv_raw_t<T, 384>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 768: return launch_dwconv_raw_t<T, 768>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 1536: return launch_dwconv_raw_t<T, 1536>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 352: return launch_dwconv_raw_t<T, 352>(x, x4, bp, out, rowstat, nb, H, W, st, b0);  // convnextv2_huge
        case 704: return launch_dwconv_raw_t<T, 704>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 1408: return launch_dwconv_raw_t<T, 1408>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
        case 2816: return launch_dwconv_raw_t<T, 2816>(x, x4, bp, out, rowstat, nb, H, W, st, b0);
    }
    return set_error(SVB_ERR_UNSUPPORTED_MODEL, "dwconv (raw): unsupported width %d", C);
}
template <typename T, int C>
static int launch_dwconv_tc_t(const CUtensorMap& xtc, const BlockParams& bp, void* out, int nb, int H, int W, int NR, cudaStream_t st) {
    using Cfg = DwTcCfg<C>;
    auto kern = dwconv_ln_tc_kernel<T, C>;
    const int P = W + 6;
    const int smem = Cfg::smem_bytes(P, NR);
    static int attr_smem[MAX_DEVICES] = {};
    const int dslot = current_device_slot();
    if (smem > attr_smem[dslot]) {
        SVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_smem[dslot] = smem;
    }
    const int tiles_per_img = ceil_div(H * P, 128);
    const int tiles = nb * tiles_per_img;
    const int grid = tiles < num_sms() ? tiles : num_sms();
    kern<<<grid, Cfg::NUM_THREADS, smem, st>>>(xtc, bp.wdw16_map, bp.bdw, bp.lnw, bp.lnb, static_cast<T*>(out), H, W, NR,
                                               Cfg::stage_bytes(P, NR), tiles_per_img, tiles);
    SVB_LAUNCHED();
    return SVB_OK;
}
template <typename T>
static int launch_dwconv_tc(const CUtensorMap& xtc, const BlockParams& bp, void* out, int C, int nb, int H, int W, int NR, cudaStream_t st) {
    if (C == 512) return launch_dwconv_tc_t<T, 512>(xtc, bp, out, nb, H, W, NR, st);
    if (C == 256) return launch_dwconv_tc_t<T, 256>(xtc, bp, out, nb, H, W, NR, st);
    return set_error(SVB_ERR_UNSUPPORTED_MODEL, "dwconv (tensor-core): unsupported width %d", C);
}
template <typename T>
static int launch_dwconv(const CUtensorMap& x, const BlockParams& bp, void* out, int C, int nb, int H, int W, cudaStream_t st) {
    switch (C) {
        case 128: return launch_dwconv_t<T, 128, 16>(x, bp, out, nb, H, W, st);
        case 256: return launch_dwconv_t<T, 256, 16>(x, bp, out, nb, H, W, st);
        case 512: return launch_dwconv_t<T, 512, 8>(x, bp, out, nb, H, W, st);
        case 1024: return launch_dwconv_t<T, 1024, 8>(x, bp, out, nb, H, W, st);
        case 2048: return launch_dwconv_t<T, 2048, 4>(x, bp, out, nb, H, W, st);  // convnext_xlarge stage 3
        case 96: return launch_dwconv_t<T, 96, 16>(x, bp, out, nb, H, W, st);     // convnext_tiny / small stage 0
        case 192: return launch_dwconv_t<T, 192, 16>(x, bp, out, nb, H, W, st);   // convnext_large (and tiny / small stage 1)
        case 384: return launch_dwconv_t<T, 384, 8>(x, bp, out, nb, H, W, st);
        case 768: return launch_dwconv_t<T, 768, 8>(x, bp, out, nb, H, W, st);
        case 1536: return launch_dwconv_t<T, 1536, 4>(x, bp, out, nb, H, W, st);
    }
    return set_error(SVB_ERR_UNSUPPORTED_MODEL, "dwconv: unsupported width %d", C);
}
template <typename T>
static int launch_ln_patchify(const void* x, const DownParams& d, void* a2, int Cin, int nb, int H, int W, cudaStream_t st) {
    const int pg = Cin <= 512 ? 4 : (Cin <= 1024 ? 2 : 1);  // LnPatchifyPG: x-adjacent tokens per warp iteration
    const long long groups = (long long)nb * H * ceil_div(W, pg);
    long long blocks = ceil_div<long long>(groups, 8);
    if (blocks > (long long)num_sms() * 8) blocks = (long long)num_sms() * 8;
    const T* xp = static_cast<const T*>(x);
    T* ap = static_cast<T*>(a2);
    switch (Cin) {
        case 128: ln_patchify_kernel<T, 128><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        case 256: ln_patchify_kernel<T, 256><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        case 512: ln_patchify_kernel<T, 512><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        case 1024: ln_patchify_kernel<T, 1024><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        case 96: ln_patchify_kernel<T, 96><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        case 192: ln_patchify_kernel<T, 192><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        case 384: ln_patchify_kernel<T, 384><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        case 768: ln_patchify_kernel<T, 768><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        case 352: ln_patchify_kernel<T, 352><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;  // convnextv2_huge
        case 704: ln_patchify_kernel<T, 704><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        case 1408: ln_patchify_kernel<T, 1408><<<(int)blocks, 256, 0, st>>>(xp, d.lnw, d.lnb, ap, nb, H, W); break;
        default: return set_error(SVB_ERR_UNSUPPORTED_MODEL, "ln_patchify: unsupported width %d", Cin);
    }
    SVB_LAUNCHED();
    return SVB_OK;
}

template <typename T>
static int launch_grn(T* hd, int nb, int tokens, int C4, const float* weight, const float* bias, float* part, float* scale, cudaStream_t st) {
    const int nchunk = ceil_div(tokens, GRN_ROWS);
    const dim3 grid(ceil_div(C4, 512), nchunk, nb);
    SVB_REQUIRE(nb <= 65535 && nchunk <= 65535 && C4 % 2 == 0 && (size_t)C4 * 4 <= 48 * 1024, SVB_ERR_UNSUPPORTED_MODEL,
                "grn: nb=%d tokens=%d C4=%d out of range", nb, tokens, C4);
    grn_sumsq_kernel<T><<<grid, 256, 0, st>>>(hd, tokens, C4, part);
    SVB_LAUNCHED();
    grn_finalize_kernel<<<nb, 256, (size_t)C4 * 4, st>>>(part, nchunk, C4, weight, scale);
    SVB_LAUNCHED();
    grn_apply_kernel<T><<<grid, 256, 0, st>>>(hd, tokens, C4, scale, bias);
    SVB_LAUNCHED();
    return SVB_OK;
}

template <typename T>
static int launch_head(const T* x, int nb, int tokens, int C, const float* n0w, const float* n0b, const float* n1w, const float* n1b,
                       const float* w1, const float* b1, int hid, const float* w2, const float* b2, int nout, float* coords,
                       cudaStream_t st) {
    // feat, hidden, reduction scratch, pool share, per-warp pools: 81 KB at C = 2048, 111 KB at C = 2816 (convnextv2_huge: one CTA
    // of the cluster per SM)
    const size_t smem = (size_t)(C + hid + 8 + C + 8 * C) * 4;
    SVB_REQUIRE(smem <= 227 * 1024, SVB_ERR_UNSUPPORTED_MODEL, "head: C=%d needs %zu bytes of shared memory", C, smem);
    auto kern = head_kernel<T>;
    static size_t attr_smem[MAX_DEVICES] = {};
    const int dslot = current_device_slot();
    if (smem > 48 * 1024 && smem > attr_smem[dslot]) {
        SVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_smem[dslot] = smem;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)nb * HEAD_CLUSTER);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = HEAD_CLUSTER;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SVB_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, x, tokens, C, n0w, n0b, n1w, n1b, w1, b1, hid, w2, b2, nout, coords));
    count_launch();
    return SVB_OK;
}

struct Timer {  // optional per-launch CUDA-event timing, accumulated per kernel class
    svb_model* m;
    cudaStream_t st;
    bool on;
    std::vector<int> classes;
    size_t used = 0;
    int begin(int cls) {
        if (!on) return SVB_OK;
        while (m->events.size() < used + 2) {
            cudaEvent_t e;
            SVB_CUDA_OK(cudaEventCreate(&e));
            m->events.push_back(e);
        }
        classes.push_back(cls);
        SVB_CUDA_OK(cudaEventRecord(m->events[used], st));
        return SVB_OK;
    }
    int end() {
        if (!on) return SVB_OK;
        SVB_CUDA_OK(cudaEventRecord(m->events[used + 1], st));
        used += 2;
        return SVB_OK;
    }
    int finish(float* times) {
        if (!on) return SVB_OK;
        SVB_CUDA_OK(cudaStreamSynchronize(st));
        for (size_t i = 0; i < classes.size(); ++i) {
            float ms = 0.f;
            SVB_CUDA_OK(cudaEventElapsedTime(&ms, m->events[2 * i], m->events[2 * i + 1]));
            times[classes[i]] += ms;
        }
        return SVB_OK;
    }
};

template <typename T>
static int forward_chunk(svb_model* m, const uint8_t* in, const float* in_f32, int nb, int H, int W, float* coords, uint8_t* ws,
                         cudaStream_t st, Timer& tm, void* const* stage_out, int n_stage_out) {
    ActPlan* plan = nullptr;
    if (int rc = get_plan(m, ws, nb, H, W, &plan)) return rc;
    const WsLayout L = ws_layout(m, nb, H, W);
    T* X = reinterpret_cast<T*>(ws + L.x);
    T* A = reinterpret_cast<T*>(ws + L.a);
    T* Hd = reinterpret_cast<T*>(ws + L.h);
    // svb_model_forward_stages: the residual stream after the last block of stage s, this micro-batch's images, on its own stream
    auto stage_done = [&](int s, int h, int w) -> int {
        if (s < n_stage_out)
            SVB_CUDA_OK(cudaMemcpyAsync(stage_out[s], X, (size_t)nb * h * w * m->dims[s] * sizeof(T), cudaMemcpyDeviceToDevice, st));
        return SVB_OK;
    };
#define RUN(cls, call)                             \
    {                                              \
        if (int rc = tm.begin(cls)) return rc;     \
        if (int rc = (call)) return rc;            \
        if (int rc = tm.end()) return rc;          \
    }
    // stem
    {
        const long long tokens = (long long)nb * (H / 4) * (W / 4);
        long long blocks = ceil_div<long long>(tokens, 8 * STEM_TPW * 4);
        if (blocks > (long long)num_sms() * 4) blocks = (long long)num_sms() * 4;  // stem_ln_kernel: 4 resident CTAs per SM
        if (blocks < 1) blocks = 1;
        if (int rc = tm.begin(SVB_KC_STEM)) return rc;
        if (in_f32 != nullptr && m->dims[0] <= 256)
            stem3_ln_kernel<T><<<(int)blocks, 256, 0, st>>>(in_f32, m->stem_w3, m->stem_b3, m->stem_lnw, m->stem_lnb, X, nb, H, W, m->dims[0]);
        else if (in_f32 != nullptr)  // 352 channels (convnextv2_huge): 11 per lane
            stem3_ln_kernel<T, 11><<<(int)blocks, 256, 0, st>>>(in_f32, m->stem_w3, m->stem_b3, m->stem_lnw, m->stem_lnb, X, nb, H, W, m->dims[0]);
        else if (m->dims[0] == 128)
            stem_ln_kernel<T, 4><<<(int)blocks, 256, 0, st>>>(in, m->stem_w, m->stem_b, m->stem_lnw, m->stem_lnb, X, nb, H, W);
        else if (m->dims[0] == 192)
            stem_ln_kernel<T, 6><<<(int)blocks, 256, 0, st>>>(in, m->stem_w, m->stem_b, m->stem_lnw, m->stem_lnb, X, nb, H, W);
        else if (m->dims[0] == 96)
            stem_ln_kernel<T, 4, 96><<<(int)blocks, 256, 0, st>>>(in, m->stem_w, m->stem_b, m->stem_lnw, m->stem_lnb, X, nb, H, W);
        else if (m->dims[0] == 352)
            stem_ln_kernel<T, 12, 352><<<(int)blocks, 256, 0, st>>>(in, m->stem_w, m->stem_b, m->stem_lnw, m->stem_lnb, X, nb, H, W);
        else
            stem_ln_kernel<T, 8><<<(int)blocks, 256, 0, st>>>(in, m->stem_w, m->stem_b, m->stem_lnw, m->stem_lnb, X, nb, H, W);
        SVB_LAUNCHED();
        if (int rc = tm.end()) return rc;
    }
    int h = H / 4, w = W / 4;
    for (int s = 0; s < 4; ++s) {
        const int C = m->dims[s];
        if (s > 0) {
            const int Cin = m->dims[s - 1];
            RUN(SVB_KC_LN_PATCHIFY, launch_ln_patchify<T>(X, m->down[s], A, Cin, nb, h, w, st));
            h /= 2;
            w /= 2;
            const int M2 = nb * h * w;
            RUN(SVB_KC_GEMM, launch_gemm<T>(plan->a2_map[s], m->down[s].w_map, plan->ox_map[s], plan->ox_map[s], m->down[s].bias,
                                            nullptr, M2, C, 4 * Cin, GEMM_BIAS, st));
        }
        const int M = nb * h * w;
        float2* rowstat = reinterpret_cast<float2*>(ws + L.stat);
        if (m->ln_fold) {
            // Depth-first over SUB-BATCHES of the micro-batch in the stages whose hidden activation is far larger than L2: the
            // [tokens, 4C] tensor fc1 writes is read back by fc2 while it is still in the 126 MB L2 (and the depthwise kernel
            // finds the residual stream fc2 just wrote there), instead of making the round trip through HBM.  A sub-batch is a
            // whole number of GEMM row tiles, so the tensor maps of the micro-batch serve every sub-batch (row / image offset).
            const int tok = h * w;
            int sub = sub_batch_images(s, nb, tok, C);
            for (int b0 = 0; b0 < nb; b0 += sub) {
                const int ns = (nb - b0) < sub ? (nb - b0) : sub;
                const int m0 = b0 * tok, m1 = (b0 + ns) * tok;
                for (const BlockParams& bp : m->blocks[s]) {
                    const bool fused = mlp_fused_lnf(m->mlp_fused_setting, C) && !m->v2 && ns == nb;
                    float2* stat_part = reinterpret_cast<float2*>(ws + L.stat_part);
                    if (plan->tc2[s]) {
                        RUN(SVB_KC_DWCONV_LN, launch_dwconv_rawtc<T>(plan->xtc2_map[s], bp, A, rowstat, stat_part, C, ns, h, w, plan->tc2[s], st, b0, !fused,
                                                                     (m->tc2_setting >> 5) & 1));
                    } else {
                        RUN(SVB_KC_DWCONV_LN, launch_dwconv_raw<T>(plan->xr_map[s], plan->xr4_map[s], bp, A, rowstat, C, ns, h, w, st, b0));
                    }
                    if (fused) {
                        if (plan->tc2[s]) { RUN(SVB_KC_MLP_FUSED, launch_mlp_fused<T>(plan->a_map[s], bp, plan->ox_map[s], C, M, st, stat_part, C / 64)); }
                        else { RUN(SVB_KC_MLP_FUSED, launch_mlp_fused<T>(plan->a_map[s], bp, plan->ox_map[s], C, M, st, rowstat, 0)); }
                        continue;
                    }
                    RUN(SVB_KC_GEMM, launch_gemm<T>(plan->a_map[s], bp.w1_map, plan->oh_map[s], plan->oh_map[s], bp.b1, bp.s1, m1, 4 * C, C,
                                                    GEMM_LNGELU, st, false, rowstat, m0));
                    if (m->v2) RUN(SVB_KC_GEMM, launch_grn<T>(Hd + (size_t)m0 * 4 * C, ns, tok, 4 * C, bp.grn_w, bp.grn_b,
                                                              reinterpret_cast<float*>(ws + L.grn_part), reinterpret_cast<float*>(ws + L.grn_scale), st));
                    RUN(SVB_KC_GEMM, launch_gemm<T>(plan->h_map[s], bp.w2_map, plan->ox_map[s], plan->ox_map[s], bp.b2, bp.gamma, m1, C, 4 * C,
                                                    GEMM_RESID, st, false, nullptr, m0));
                }
            }
            if (int rc = stage_done(s, h, w)) return rc;
            continue;
        }
        for (const BlockParams& bp : m->blocks[s]) {
            if (plan->tc_rows[s]) {
                RUN(SVB_KC_DWCONV_LN, launch_dwconv_tc<T>(plan->xtc_map[s], bp, A, C, nb, h, w, plan->tc_rows[s], st));
            } else {
                RUN(SVB_KC_DWCONV_LN, launch_dwconv<T>(plan->x_map[s], bp, A, C, nb, h, w, st));
            }
            if (mlp_fused(m->mlp_fused_setting, C) && !m->v2) {
                RUN(SVB_KC_MLP_FUSED, launch_mlp_fused<T>(plan->a_map[s], bp, plan->ox_map[s], C, M, st));
            } else {
                RUN(SVB_KC_GEMM, launch_gemm<T>(plan->a_map[s], bp.w1_map, plan->oh_map[s], plan->oh_map[s], bp.b1, nullptr, M, 4 * C, C,
                                                GEMM_GELU, st, coex_stage(s)));
                if (m->v2) RUN(SVB_KC_GEMM, launch_grn<T>(Hd, nb, h * w, 4 * C, bp.grn_w, bp.grn_b, reinterpret_cast<float*>(ws + L.grn_part),
                                                          reinterpret_cast<float*>(ws + L.grn_scale), st));
                RUN(SVB_KC_GEMM, launch_gemm<T>(plan->h_map[s], bp.w2_map, plan->ox_map[s], plan->ox_map[s], bp.b2, bp.gamma, M, C, 4 * C,
                                                GEMM_RESID, st, coex_stage(s)));
            }
        }
        if (int rc = stage_done(s, h, w)) return rc;
    }
    {
        const int C = m->dims[3];
        if (int rc = tm.begin(SVB_KC_HEAD)) return rc;
        if (int rc = launch_head<T>(X, nb, h * w, C, m->hn0w, m->hn0b, m->hn1w, m->hn1b, m->hw1, m->hb1, m->hid, m->hw2, m->hb2,
                                    m->nout, coords, st))
            return rc;
        if (int rc = tm.end()) return rc;
    }
#undef RUN
    return SVB_OK;
}

}  // namespace svb

// SVB_DUAL_CHAIN=0 keeps one micro-batch in flight (A/B testing; also what a workspace of the single size selects)
static bool dual_chain_enabled() {
    static int enabled = -1;
    if (enabled < 0) {
        const char* e = getenv("SVB_DUAL_CHAIN");
        enabled = (e && e[0] == '0') ? 0 : 1;
    }
    return enabled != 0;
}

extern "C" size_t svb_model_workspace_bytes(const svb_model* m, int micro_batch, int H, int W) {
    if (!m || micro_batch <= 0 || H <= 0 || W <= 0) return 0;
    const size_t one = align_up(ws_layout(m, micro_batch, H, W).total, 1024);
    return dual_chain_enabled() ? 2 * one : one;
}

static int model_forward_any(svb_model* m, const uint8_t* d_in_u8, const float* d_in_f32, int B, int H, int W, float* d_coords,
                             int micro_batch, void* d_ws, size_t ws_bytes, void* stream_, float* times_ms,
                             void* const* stage_out = nullptr, int n_stage_out = 0) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    SVB_REQUIRE(m && (d_in_u8 || d_in_f32) && d_coords && d_ws, SVB_ERR_INVALID_ARG, "model_forward: null argument");
    SVB_REQUIRE(B >= 0 && micro_batch > 0, SVB_ERR_INVALID_ARG, "model_forward: B=%d micro_batch=%d", B, micro_batch);
    SVB_REQUIRE(H > 0 && W > 0 && H % 32 == 0 && W % 32 == 0, SVB_ERR_INVALID_ARG,
                "model_forward: input %dx%d must be a positive multiple of 32 (ConvNeXt stride)", H, W);
    if (micro_batch > B && B > 0) micro_batch = B;
    const size_t need = ws_layout(m, micro_batch, H, W).total;
    SVB_REQUIRE(ws_bytes >= need, SVB_ERR_WORKSPACE_TOO_SMALL, "model_forward: workspace %zu < %zu bytes", ws_bytes, need);
    SVB_REQUIRE((reinterpret_cast<uintptr_t>(d_ws) & 1023) == 0, SVB_ERR_INVALID_ARG, "model_forward: workspace must be 1024-byte aligned");
    Timer tm{m, st, times_ms != nullptr};
    const size_t one = align_up(need, 1024);
    const bool dual = dual_chain_enabled() && times_ms == nullptr && B > micro_batch && ws_bytes >= 2 * one && m->aux_stream != nullptr;
    if (dual) {
        SVB_CUDA_OK(cudaEventRecord(m->fork_ev, st));
        SVB_CUDA_OK(cudaStreamWaitEvent(m->aux_stream, m->fork_ev, 0));
    }
    int chunk = 0;
    for (int b0 = 0; b0 < B; b0 += micro_batch, ++chunk) {
        const int nb = (B - b0) < micro_batch ? (B - b0) : micro_batch;
        const bool odd = dual && (chunk & 1);
        cudaStream_t cs = odd ? m->aux_stream : st;
        uint8_t* ws = static_cast<uint8_t*>(d_ws) + (odd ? one : 0);
        int rc;
        const uint8_t* in8 = d_in_u8 ? d_in_u8 + (size_t)b0 * H * W : nullptr;
        const float* in32 = d_in_f32 ? d_in_f32 + (size_t)b0 * 3 * H * W : nullptr;
        void* so[4] = {};
        for (int s = 0; s < n_stage_out; ++s)  // [B, H / 2^(s+2), W / 2^(s+2), C_s], 16-bit: this chunk starts at image b0
            so[s] = static_cast<uint8_t*>(stage_out[s]) + (size_t)b0 * (H >> (s + 2)) * (W >> (s + 2)) * m->dims[s] * 2;
        if (m->dtype == SVB_FP16)
            rc = forward_chunk<__half>(m, in8, in32, nb, H, W, d_coords + (size_t)b0 * m->nout, ws, cs, tm, so, n_stage_out);
        else
            rc = forward_chunk<__nv_bfloat16>(m, in8, in32, nb, H, W, d_coords + (size_t)b0 * m->nout, ws, cs, tm, so, n_stage_out);
        if (rc) return rc;
    }
    if (dual) {
        SVB_CUDA_OK(cudaEventRecord(m->join_ev, m->aux_stream));
        SVB_CUDA_OK(cudaStreamWaitEvent(st, m->join_ev, 0));
    }
    return tm.finish(times_ms);
}

extern "C" int svb_model_forward(svb_model* m, const uint8_t* d_in_u8, int B, int H, int W, float* d_coords,
                                 int micro_batch, void* d_ws, size_t ws_bytes, void* stream_, float* times_ms) {
    SVB_REQUIRE(d_in_u8, SVB_ERR_INVALID_ARG, "model_forward: null argument");
    return model_forward_any(m, d_in_u8, nullptr, B, H, W, d_coords, micro_batch, d_ws, ws_bytes, stream_, times_ms);
}

extern "C" int svb_model_forward_stages(svb_model* m, const uint8_t* d_in_u8, int B, int H, int W, float* d_coords, int micro_batch,
                                        void* d_ws, size_t ws_bytes, void* stream_, void* const* d_stage_out, int n_stage_out) {
    SVB_REQUIRE(d_in_u8 && d_stage_out, SVB_ERR_INVALID_ARG, "model_forward_stages: null argument");
    SVB_REQUIRE(n_stage_out >= 1 && n_stage_out <= 4, SVB_ERR_INVALID_ARG, "model_forward_stages: %d stage buffers (1..4)", n_stage_out);
    for (int s = 0; s < n_stage_out; ++s)
        SVB_REQUIRE(d_stage_out[s], SVB_ERR_INVALID_ARG, "model_forward_stages: stage buffer %d is null", s);
    return model_forward_any(m, d_in_u8, nullptr, B, H, W, d_coords, micro_batch, d_ws, ws_bytes, stream_, nullptr, d_stage_out, n_stage_out);
}

extern "C" int svb_model_forward_f32(svb_model* m, const float* d_in_nchw, int B, int H, int W, float* d_coords,
                                     int micro_batch, void* d_ws, size_t ws_bytes, void* stream_, float* times_ms) {
    SVB_REQUIRE(d_in_nchw, SVB_ERR_INVALID_ARG, "model_forward_f32: null argument");
    SVB_REQUIRE(!m || m->dims[0] <= 352, SVB_ERR_UNSUPPORTED_MODEL, "model_forward_f32: stem width %d > 352", m ? m->dims[0] : 0);
    return model_forward_any(m, nullptr, d_in_nchw, B, H, W, d_coords, micro_batch, d_ws, ws_bytes, stream_, times_ms);
}

extern "C" int svb_model_cost(const svb_model* m, int B, int H, int W, double* gemm_flops, int64_t* launches) {
    SVB_REQUIRE(m, SVB_ERR_INVALID_ARG, "model_cost: null model");
    double fl = 0.0;
    int64_t n = 1;  // stem
    int h = H / 4, w = W / 4;
    for (int s = 0; s < 4; ++s) {
        const double C = m->dims[s];
        if (s > 0) {
            h /= 2;
            w /= 2;
            fl += 2.0 * B * h * w * C * 4.0 * m->dims[s - 1];
            n += 2;
        }
        fl += (double)m->depths[s] * 2.0 * (2.0 * B * h * w * C * 4.0 * C);
        n += (m->v2 ? 6 : 3) * (int64_t)m->depths[s];
    }
    n += 1;  // head
    if (gemm_flops) *gemm_flops = fl;
    if (launches) *launches = n;
    return SVB_OK;
}

extern "C" int svb_gemm(const void* d_a, const void* d_w, void* d_out, const void* d_resid, const float* d_bias,
                        const float* d_gamma, int M, int N, int K, int mode, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_a && d_w && d_out && d_bias, SVB_ERR_INVALID_ARG, "gemm: null argument");
    SVB_REQUIRE(mode != GEMM_RESID || (d_resid && d_gamma), SVB_ERR_INVALID_ARG, "gemm: residual mode needs resid and gamma");
    SVB_REQUIRE(mode != GEMM_LNGELU || (d_resid && d_gamma), SVB_ERR_INVALID_ARG, "gemm: folded-LayerNorm mode needs the row statistics (d_resid) and s_n (d_gamma)");
    SVB_REQUIRE(M > 0 && N > 0 && K > 0, SVB_ERR_INVALID_ARG, "gemm: bad shape");
    CUtensorMap a_map, w_map, out_map, resid_map;
    if (int rc = make_operand_map(&a_map, dtype, d_a, M, K, 128)) return rc;
    const bool half = gemm_half_env() && N % 128 == 0 && mode != GEMM_LNGELU;
    const float2* rowstat = mode == GEMM_LNGELU ? static_cast<const float2*>(d_resid) : nullptr;
    if (int rc = make_operand_map(&w_map, dtype, d_w, N, K, gemm_bn_for(N, half) / gemm_cg(N, K))) return rc;
    if (int rc = make_epilogue_map(&out_map, dtype, d_out, M, N)) return rc;
    if (int rc = make_epilogue_map(&resid_map, dtype, mode == GEMM_RESID ? d_resid : d_out, M, N)) return rc;
    if (dtype == SVB_FP16) return launch_gemm<__half>(a_map, w_map, out_map, resid_map, d_bias, d_gamma, M, N, K, mode, st, half, rowstat);
    return launch_gemm<__nv_bfloat16>(a_map, w_map, out_map, resid_map, d_bias, d_gamma, M, N, K, mode, st, half, rowstat);
}

extern "C" int svb_mlp_fused(const void* d_a, const void* d_w1, const float* d_b1, const void* d_w2, const float* d_b2,
                             const float* d_gamma, void* d_x, int M, int C, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_a && d_w1 && d_b1 && d_w2 && d_b2 && d_gamma && d_x && M > 0, SVB_ERR_INVALID_ARG, "mlp_fused: bad arguments");
    SVB_REQUIRE(C == 128 || C == 256, SVB_ERR_UNSUPPORTED_MODEL, "mlp_fused: width %d (supported: 128, 256)", C);
    BlockParams bp{};
    bp.b1 = const_cast<float*>(d_b1);
    bp.b2 = const_cast<float*>(d_b2);
    bp.gamma = const_cast<float*>(d_gamma);
    CUtensorMap a_map, x_map;
    if (int rc = make_operand_map(&a_map, dtype, d_a, M, C, 128)) return rc;
    if (int rc = make_operand_map(&bp.w1f_map, dtype, d_w1, 4 * (uint64_t)C, C, 32)) return rc;
    if (int rc = make_operand_map(&bp.w2f_map, dtype, d_w2, C, 4 * (uint64_t)C, C / 2)) return rc;
    if (int rc = make_epilogue_map(&x_map, dtype, d_x, M, C)) return rc;
    if (dtype == SVB_FP16) return launch_mlp_fused<__half>(a_map, bp, x_map, C, M, st);
    return launch_mlp_fused<__nv_bfloat16>(a_map, bp, x_map, C, M, st);
}

extern "C" int svb_mlp_fused_ln(const void* d_a, const void* d_w1g, const float* d_t, const float* d_s, const float* d_rowstat, const void* d_w2,
                                const float* d_b2, const float* d_gamma, void* d_x, int M, int C, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_a && d_w1g && d_t && d_s && d_rowstat && d_w2 && d_b2 && d_gamma && d_x && M > 0, SVB_ERR_INVALID_ARG, "mlp_fused_ln: bad arguments");
    SVB_REQUIRE(C == 128 || C == 256, SVB_ERR_UNSUPPORTED_MODEL, "mlp_fused_ln: width %d (supported: 128, 256)", C);
    BlockParams bp{};
    bp.b1 = const_cast<float*>(d_t);
    bp.s1 = const_cast<float*>(d_s);
    bp.b2 = const_cast<float*>(d_b2);
    bp.gamma = const_cast<float*>(d_gamma);
    CUtensorMap a_map, x_map;
    if (int rc = make_operand_map(&a_map, dtype, d_a, M, C, 128)) return rc;
    if (int rc = make_operand_map(&bp.w1f_map, dtype, d_w1g, 4 * (uint64_t)C, C, 32)) return rc;
    if (int rc = make_operand_map(&bp.w2f_map, dtype, d_w2, C, 4 * (uint64_t)C, C / 2)) return rc;
    if (int rc = make_epilogue_map(&x_map, dtype, d_x, M, C)) return rc;
    const float2* rs = reinterpret_cast<const float2*>(d_rowstat);
    if (dtype == SVB_FP16) return launch_mlp_fused<__half>(a_map, bp, x_map, C, M, st, rs);
    return launch_mlp_fused<__nv_bfloat16>(a_map, bp, x_map, C, M, st, rs);
}

// ---------------------------------------------------------------------------------------------
// standalone layer entries (tests / profiling): the same kernels, tensor maps built per call
template <typename T>
static int stem_entry(const uint8_t* in, const float* wf, const float* bf, const float* lnw, const float* lnb, void* out,
                      int B, int H, int W, int C0, cudaStream_t st) {
    const long long tokens = (long long)B * (H / 4) * (W / 4);
    long long blocks = ceil_div<long long>(tokens, 8 * STEM_TPW * 4);
    if (blocks > (long long)num_sms() * 4) blocks = (long long)num_sms() * 4;  // stem_ln_kernel: 4 resident CTAs per SM
    if (blocks < 1) blocks = 1;
    if (C0 == 128) stem_ln_kernel<T, 4><<<(int)blocks, 256, 0, st>>>(in, wf, bf, lnw, lnb, static_cast<T*>(out), B, H, W);
    else if (C0 == 192) stem_ln_kernel<T, 6><<<(int)blocks, 256, 0, st>>>(in, wf, bf, lnw, lnb, static_cast<T*>(out), B, H, W);
    else if (C0 == 96) stem_ln_kernel<T, 4, 96><<<(int)blocks, 256, 0, st>>>(in, wf, bf, lnw, lnb, static_cast<T*>(out), B, H, W);
    else if (C0 == 256) stem_ln_kernel<T, 8><<<(int)blocks, 256, 0, st>>>(in, wf, bf, lnw, lnb, static_cast<T*>(out), B, H, W);
    else if (C0 == 352) stem_ln_kernel<T, 12, 352><<<(int)blocks, 256, 0, st>>>(in, wf, bf, lnw, lnb, static_cast<T*>(out), B, H, W);
    else return set_error(SVB_ERR_UNSUPPORTED_MODEL, "stem: width %d unsupported", C0);
    SVB_LAUNCHED();
    return SVB_OK;
}

extern "C" int svb_stem_ln(const uint8_t* d_in, const float* d_wf, const float* d_bf, const float* d_lnw, const float* d_lnb,
                           void* d_out, int B, int H, int W, int C0, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_in && d_wf && d_bf && d_lnw && d_lnb && d_out && B > 0 && H % 4 == 0 && W % 4 == 0, SVB_ERR_INVALID_ARG,
                "stem_ln: bad arguments");
    if (dtype == SVB_FP16) return stem_entry<__half>(d_in, d_wf, d_bf, d_lnw, d_lnb, d_out, B, H, W, C0, st);
    return stem_entry<__nv_bfloat16>(d_in, d_wf, d_bf, d_lnw, d_lnb, d_out, B, H, W, C0, st);
}

extern "C" int svb_dwconv_ln(const void* d_x, const float* d_taps, const float* d_bias, const float* d_lnw,
                             const float* d_lnb, void* d_out, int B, int H, int W, int C, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_x && d_taps && d_bias && d_lnw && d_lnb && d_out && B > 0 && H > 0 && W > 0, SVB_ERR_INVALID_ARG,
                "dwconv_ln: bad arguments");
    BlockParams bp{};
    bp.wdw = const_cast<float*>(d_taps);
    bp.bdw = const_cast<float*>(d_bias);
    bp.lnw = const_cast<float*>(d_lnw);
    bp.lnb = const_cast<float*>(d_lnb);
    {
        const uint64_t dims[2] = {(uint64_t)C, 49};
        const uint64_t strides[1] = {(uint64_t)C * 4};
        const uint32_t box[2] = {64, 49};
        if (int rc = encode_tmap(&bp.wdw_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, d_taps, dims, strides, box,
                                 CU_TENSOR_MAP_SWIZZLE_NONE))
            return rc;
    }
    CUtensorMap x_map;
    {
        const uint64_t uC = C;
        const uint64_t dims[4] = {uC, (uint64_t)W, (uint64_t)H, (uint64_t)B};
        const uint64_t strides[3] = {uC * 2, (uint64_t)W * uC * 2, (uint64_t)H * W * uC * 2};
        const uint32_t box[4] = {64, 14, (uint32_t)(dw_th(C) + 6), 1};
        if (int rc = encode_tmap(&x_map, tmap_dtype(dtype), 4, d_x, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE)) return rc;
    }
    if (dtype == SVB_FP16) return launch_dwconv<__half>(x_map, bp, d_out, C, B, H, W, st);
    return launch_dwconv<__nv_bfloat16>(x_map, bp, d_out, C, B, H, W, st);
}

extern "C" int svb_dwconv_raw(const void* d_x, const float* d_taps, const float* d_bias, void* d_out, float* d_rowstat, int B, int H,
                              int W, int C, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_x && d_taps && d_bias && d_out && d_rowstat && B > 0 && H > 0 && W > 0, SVB_ERR_INVALID_ARG, "dwconv_raw: bad arguments");
    BlockParams bp{};
    bp.wdw = const_cast<float*>(d_taps);
    bp.bdw = const_cast<float*>(d_bias);
    {
        const uint64_t dims[2] = {(uint64_t)C, 49};
        const uint64_t strides[1] = {(uint64_t)C * 4};
        const uint32_t box[2] = {64, 49};
        if (int rc = encode_tmap(&bp.wdw_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, d_taps, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE))
            return rc;
    }
    CUtensorMap x_map, x4_map;
    {
        const uint64_t uC = C;
        const uint64_t dims[4] = {uC, (uint64_t)W, (uint64_t)H, (uint64_t)B};
        const uint64_t strides[3] = {uC * 2, (uint64_t)W * uC * 2, (uint64_t)H * W * uC * 2};
        const uint32_t box[4] = {64, 22, 14, 1};
        if (int rc = encode_tmap(&x_map, tmap_dtype(dtype), 4, d_x, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE)) return rc;
        const uint32_t box4[4] = {64, 22, 10, 1};
        if (int rc = encode_tmap(&x4_map, tmap_dtype(dtype), 4, d_x, dims, strides, box4, CU_TENSOR_MAP_SWIZZLE_NONE)) return rc;
    }
    float2* rs = reinterpret_cast<float2*>(d_rowstat);
    if (dtype == SVB_FP16) return launch_dwconv_raw<__half>(x_map, x4_map, bp, d_out, rs, C, B, H, W, st);
    return launch_dwconv_raw<__nv_bfloat16>(x_map, x4_map, bp, d_out, rs, C, B, H, W, st);
}

extern "C" int svb_dwconv_tc_pack(const float* h_taps, void* h_wtc, int C, int dtype) {
    SVB_REQUIRE(h_taps && h_wtc && C > 0 && C % 64 == 0, SVB_ERR_INVALID_ARG, "dwconv_tc_pack: C (%d) must be a positive multiple of 64", C);
    SVB_REQUIRE(dtype == SVB_BF16 || dtype == SVB_FP16, SVB_ERR_INVALID_ARG, "dwconv_tc_pack: dtype %d", dtype);
    pack_wtc(h_taps, static_cast<uint16_t*>(h_wtc), C, dtype);
    return SVB_OK;
}

extern "C" int svb_dwconv_raw_tc(const void* d_x, const void* d_wtc, const float* d_bias, void* d_out, float* d_rowstat, float* d_stat_part,
                                 int B, int H, int W, int C, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_x && d_wtc && d_bias && d_out && d_rowstat && d_stat_part && B > 0 && H > 0 && W > 0, SVB_ERR_INVALID_ARG,
                "dwconv_raw_tc: bad arguments");
    SVB_REQUIRE(C % 64 == 0 && C / 64 <= num_sms(), SVB_ERR_UNSUPPORTED_MODEL, "dwconv_raw_tc: C (%d) must be a multiple of 64", C);
    const int mode = (W == 8 || W == 16 || W == 32) ? 1 : 2;
    BlockParams bp{};
    bp.bdw = const_cast<float*>(d_bias);
    if (int rc = make_wtc_map(&bp.wtc_map, dtype, d_wtc, C)) return rc;
    CUtensorMap x_map;
    if (int rc = make_xtc2_map(&x_map, dtype, d_x, C, B, H, W, mode)) return rc;
    float2* rs = reinterpret_cast<float2*>(d_rowstat);
    float2* sp = reinterpret_cast<float2*>(d_stat_part);
    if (int rc = make_wtc_map(&bp.wtc2_map, dtype, d_wtc, C, 56)) return rc;
    const bool pair = (dw_tc2_env() >> 5) & 1;  // SVB_TC2_PAIR=1: the cta_group::2 variant (read per call: tests compare both)
    if (dtype == SVB_FP16) return launch_dwconv_rawtc<__half>(x_map, bp, d_out, rs, sp, C, B, H, W, mode, st, 0, true, pair);
    return launch_dwconv_rawtc<__nv_bfloat16>(x_map, bp, d_out, rs, sp, C, B, H, W, mode, st, 0, true, pair);
}

extern "C" int svb_dwconv_ln_tc(const void* d_x, const void* d_taps16, const float* d_bias, const float* d_lnw,
                                const float* d_lnb, void* d_out, int B, int H, int W, int C, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_x && d_taps16 && d_bias && d_lnw && d_lnb && d_out && B > 0 && H > 0 && W > 0, SVB_ERR_INVALID_ARG,
                "dwconv_ln_tc: bad arguments");
    const int P = W + 6;
    const int NR = (C == 256 || C == 512) ? (2 * P + 132) / P + 6 : 0;
    SVB_REQUIRE(NR > 0 && (C == 512 ? DwTcCfg<512>::smem_bytes(P, NR) : DwTcCfg<256>::smem_bytes(P, NR)) <= 227 * 1024,
                SVB_ERR_UNSUPPORTED_MODEL, "dwconv_ln_tc: C=%d W=%d is outside the tensor-core kernel's range", C, W);
    BlockParams bp{};
    bp.bdw = const_cast<float*>(d_bias);
    bp.lnw = const_cast<float*>(d_lnw);
    bp.lnb = const_cast<float*>(d_lnb);
    {
        const uint64_t dims[2] = {(uint64_t)C, 49};
        const uint64_t strides[1] = {(uint64_t)C * 2};
        const uint32_t box[2] = {64, 49};
        if (int rc = encode_tmap(&bp.wdw16_map, tmap_dtype(dtype), 2, d_taps16, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE))
            return rc;
    }
    CUtensorMap x_map;
    {
        const uint64_t uC = C;
        const uint64_t dims[4] = {uC, (uint64_t)W, (uint64_t)H, (uint64_t)B};
        const uint64_t strides[3] = {uC * 2, (uint64_t)W * uC * 2, (uint64_t)H * W * uC * 2};
        const uint32_t box[4] = {64, (uint32_t)(W + 6), (uint32_t)NR, 1};
        if (int rc = encode_tmap(&x_map, tmap_dtype(dtype), 4, d_x, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    if (dtype == SVB_FP16) return launch_dwconv_tc<__half>(x_map, bp, d_out, C, B, H, W, NR, st);
    return launch_dwconv_tc<__nv_bfloat16>(x_map, bp, d_out, C, B, H, W, NR, st);
}

extern "C" int svb_ln_patchify(const void* d_x, const float* d_lnw, const float* d_lnb, void* d_out, int B, int H, int W,
                               int C, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_x && d_lnw && d_lnb && d_out && B > 0 && H % 2 == 0 && W % 2 == 0, SVB_ERR_INVALID_ARG,
                "ln_patchify: bad arguments");
    DownParams d{};
    d.lnw = const_cast<float*>(d_lnw);
    d.lnb = const_cast<float*>(d_lnb);
    if (dtype == SVB_FP16) return launch_ln_patchify<__half>(d_x, d, d_out, C, B, H, W, st);
    return launch_ln_patchify<__nv_bfloat16>(d_x, d, d_out, C, B, H, W, st);
}

extern "C" int svb_head(const void* d_x, int B, int tokens, int C, const float* n0w, const float* n0b, const float* n1w,
                        const float* n1b, const float* w1, const float* b1, int HID, const float* w2, const float* b2,
                        int NOUT, float* d_coords, int dtype, void* stream_) {
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (int rc = check_device_sm100()) return rc;
    SVB_REQUIRE(d_x && d_coords && B > 0 && tokens > 0 && C % 8 == 0, SVB_ERR_INVALID_ARG, "head: bad arguments (C must be a multiple of 8)");
    if (dtype == SVB_FP16)
        return launch_head<__half>(static_cast<const __half*>(d_x), B, tokens, C, n0w, n0b, n1w, n1b, w1, b1, HID, w2, b2, NOUT, d_coords, st);
    return launch_head<__nv_bfloat16>(static_cast<const __nv_bfloat16*>(d_x), B, tokens, C, n0w, n0b, n1w, n1b, w1, b1, HID, w2, b2, NOUT,
                                      d_coords, st);
}
