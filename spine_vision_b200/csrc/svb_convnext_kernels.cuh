// svb_convnext_kernels.cuh -- sm_100a device kernels of the CoordinateRegressor forward
// (spine_vision/training/models/generic.py:389-391 over a timm ConvNeXt backbone).
//
// Activations are NHWC ("token-major": [B*H*W, C]) 16-bit (bf16 or fp16), so every pointwise
// layer is a K-major GEMM operand as stored.  Kernels:
//   stem_ln_kernel      conv4x4 s4 (1 folded input channel) + LayerNorm2d         CUDA cores, HBM-bound
//   dwconv_ln_kernel    depthwise 7x7 + bias + LayerNorm(C)                       TMA halo tiles, warp-shuffle LN
//   gemm_kernel         D = epilogue(A * W^T): fc1+GELU / fc2*gamma+residual / downsample conv
//                       tcgen05.mma (kind::f16) with TMEM accumulators, TMA operand pipeline
//   ln_patchify_kernel  LayerNorm2d + 2x2/s2 patch gather (A operand of the downsample GEMM)
//   head_kernel         avg-pool + LayerNorm2d + LayerNorm + Linear + GELU + Linear + sigmoid
#pragma once
#include "svb_common.cuh"

namespace svb {

constexpr float LN_EPS_BACKBONE = 1e-6f;  // timm ConvNeXt LayerNorm / LayerNorm2d
constexpr float LN_EPS_HEAD = 1e-5f;      // nn.LayerNorm default (generic.py:344)
// depthwise conv: the 7 kx steps stay a rolled loop so that each step is one clean run of FFMA2s
// (operand-reuse friendly) behind its own batch of shared-memory loads
constexpr int DW_KX_UNROLL = 1;

// --------------------------------------------------------------------------------------------
// GELU(x) = x * Phi(x) with Phi through erfc(|x|/sqrt2) ~= exp2(poly5(|x|)), |x| clamped at 4*sqrt2.
// Max |erfc error| 6.8e-7 (fit in scripts/fit_gelu.py), i.e. far below 16-bit output rounding.
// 10 FP32 ops + 1 MUFU per element: the fc1 epilogue has a budget of ~16 issue slots per element
// at C=128 before it, not the tensor pipe, bounds the kernel.
__device__ __forceinline__ float gelu_fast(float x) {
    const float u = fminf(fabsf(x), 5.65685425f);
    float r = -5.20460508e-04f;            // c5 / 2^(5/2)
    r = fmaf(r, u, 7.39751849e-03f);       // c4 / 4
    r = fmaf(r, u, -5.25612477e-02f);      // c3 / 2^(3/2)
    r = fmaf(r, u, -4.59254682e-01f);      // c2 / 2
    r = fmaf(r, u, -1.15109138e+00f);      // c1 / sqrt2
    r *= u;
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(r));
    const float h = (0.5f * x) * e;
    return fmaxf(x, 0.0f) - fabsf(h);
}
__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

// ============================================================================ stem
// in  u8 [B,H,W] (K1 output, one plane); /255, ImageNet mean/std and the RGB replication of
// cropping.py:463-472 are folded into wf/bf (SURVEY Appendix C).  out [B,H/4,W/4,C0].
// One warp = STEM_TPW tokens per iteration (independent load / FMA / shuffle chains in flight: the
// kernel is latency-bound otherwise), lane = CPL consecutive output channels as packed fp32 pairs.
constexpr int STEM_TPW = 4;  // the 128-bit pixel-row load below assumes 4

template <typename T, int CPL, int C0 = 32 * CPL>
__global__ void __launch_bounds__(256, (CPL <= 4) ? 4 : 2) stem_ln_kernel(const uint8_t* __restrict__ in, const float* __restrict__ wf /*[C0][16]*/,
                                                         const float* __restrict__ bf, const float* __restrict__ lnw,
                                                         const float* __restrict__ lnb, T* __restrict__ out, int B, int H,
                                                         int W) {
    static_assert(CPL % 2 == 0, "stem packs channel pairs");
    // C0 < 32 * CPL (96 channels with CPL = 4, convnext_tiny / small): the lanes past C0 / CPL carry zero weights, stay out of
    // the LayerNorm sums and do not store.  RAGGED (C0 % CPL != 0; 352 channels with CPL = 12, convnextv2_huge): one lane is
    // only part-filled, so the same three things are done per channel pair (the off pairs of that lane are masked).  CPL = 12
    // rather than 11 channels per lane because the FMAs work on packed pairs; 29 lanes of 12 + one of 4 keep the 2 CTAs per SM
    // of the CPL = 8 (256-wide) stem.
    constexpr int NP = CPL / 2, TPW = STEM_TPW;
    constexpr bool RAGGED = C0 % CPL != 0;
    static_assert(C0 % 2 == 0 && C0 <= 32 * CPL, "stem width");
    // folded weights as packed channel pairs in shared memory, [tap][pair j][lane]: a warp's read of one (tap, j) is 256
    // contiguous bytes.  (In registers they cost 32 * NP registers per thread and held the kernel at 16 warps per SM, where
    // it is latency-bound; from shared memory each value is read once per TPW tokens.)
    __shared__ uint64_t s_w[16][NP][32];
    const int lane = threadIdx.x & 31;
    const bool lane_on = lane * CPL < C0;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int Ho = H >> 2, Wo = W >> 2;
    const long long tokens = (long long)B * Ho * Wo;

    for (int i = threadIdx.x; i < 16 * NP * 32; i += blockDim.x) {
        const int l = i & 31, j = (i >> 5) % NP, p = i / (32 * NP);
        const int c = l * CPL + 2 * j;
        s_w[p][j][l] = c < C0 ? pk2(wf[c * 16 + p], wf[(c + 1) * 16 + p]) : pk2(0.f, 0.f);
    }
    uint64_t bias2[NP];
    float g[CPL], be[CPL];
#pragma unroll
    for (int j = 0; j < NP; ++j) {
        const int c = lane * CPL + 2 * j;
        if constexpr (RAGGED) bias2[j] = c < C0 ? pk2(bf[c], bf[c + 1]) : pk2(0.f, 0.f);
        else bias2[j] = lane_on ? pk2(bf[c], bf[c + 1]) : pk2(0.f, 0.f);
    }
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
        if constexpr (RAGGED) {
            const int c = lane * CPL + j;
            g[j] = c < C0 ? lnw[c] : 0.f;
            be[j] = c < C0 ? lnb[c] : 0.f;
        } else {
            g[j] = lane_on ? lnw[lane * CPL + j] : 0.f; be[j] = lane_on ? lnb[lane * CPL + j] : 0.f;
        }
    }
    __syncthreads();

    const bool row_quad = (Wo % TPW) == 0;  // the TPW tokens of an iteration are x-adjacent: one 128-bit load per pixel row
    for (long long t0 = warp * TPW; t0 < tokens; t0 += nwarps * TPW) {
        uint32_t px[TPW][4];
        if (row_quad) {
            const int b = (int)(t0 / (Ho * Wo));
            const int rem = (int)(t0 - (long long)b * Ho * Wo);
            const int ty = rem / Wo, tx = rem - ty * Wo;
            const uint8_t* p = in + ((size_t)b * H + (size_t)ty * 4) * W + (size_t)tx * 4;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(p + (size_t)r * W));
                px[0][r] = v.x; px[1][r] = v.y; px[2][r] = v.z; px[3][r] = v.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < TPW; ++k) {
                const long long t = t0 + k < tokens ? t0 + k : tokens - 1;  // clamp: the store below is masked
                const int b = (int)(t / (Ho * Wo));
                const int rem = (int)(t - (long long)b * Ho * Wo);
                const int ty = rem / Wo, tx = rem - ty * Wo;
                const uint8_t* p = in + ((size_t)b * H + (size_t)ty * 4) * W + (size_t)tx * 4;
#pragma unroll
                for (int r = 0; r < 4; ++r) px[k][r] = __ldg(reinterpret_cast<const uint32_t*>(p + (size_t)r * W));
            }
        }
        uint64_t acc[TPW][NP];
        float s[TPW];
#pragma unroll
        for (int k = 0; k < TPW; ++k)
#pragma unroll
            for (int j = 0; j < NP; ++j) acc[k][j] = bias2[j];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            uint64_t wq[NP];
#pragma unroll
            for (int j = 0; j < NP; ++j) wq[j] = s_w[q][j][lane];
#pragma unroll
            for (int k = 0; k < TPW; ++k) {
                // u8 -> f32 without the conversion unit (I2F runs on the XU pipe at 16 lanes/clk/SM):
                // PRMT drops the byte into the mantissa of 2^23, one FADD removes the 2^23 -- exact for 0..255
                const float f = __uint_as_float(__byte_perm(px[k][q >> 2], 0x4B000000u, 0x7650u | (uint32_t)(q & 3))) - 8388608.0f;
                const uint64_t f2 = pk2(f, f);
#pragma unroll
                for (int j = 0; j < NP; ++j) acc[k][j] = fma2(f2, wq[j], acc[k][j]);
            }
        }
#pragma unroll
        for (int k = 0; k < TPW; ++k) {
            float a = 0.f;
#pragma unroll
            for (int j = 0; j < NP; ++j) { float lo, hi; upk2(acc[k][j], lo, hi); a += lo + hi; }
            s[k] = a;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int k = 0; k < TPW; ++k) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
        }
        float mean[TPW], v2[TPW];
#pragma unroll
        for (int k = 0; k < TPW; ++k) {
            mean[k] = s[k] * (1.0f / C0);
            float q = 0.f;
#pragma unroll
            for (int j = 0; j < NP; ++j) {
                float lo, hi;
                upk2(acc[k][j], lo, hi);
                lo -= mean[k]; hi -= mean[k];
                if constexpr (RAGGED)
                    if (lane * CPL + 2 * j >= C0) continue;
                q = fmaf(lo, lo, q);
                q = fmaf(hi, hi, q);
            }
            v2[k] = lane_on ? q : 0.f;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int k = 0; k < TPW; ++k) v2[k] += __shfl_xor_sync(0xffffffffu, v2[k], o);
        }
#pragma unroll
        for (int k = 0; k < TPW; ++k) {
            if (t0 + k >= tokens) break;
            const float rstd = 1.0f / sqrtf(v2[k] * (1.0f / C0) + LN_EPS_BACKBONE);
            uint32_t o[NP];
#pragma unroll
            for (int j = 0; j < NP; ++j) {
                float lo, hi;
                upk2(acc[k][j], lo, hi);
                o[j] = Cvt<T>::pack2(fmaf((lo - mean[k]) * rstd, g[2 * j], be[2 * j]),
                                     fmaf((hi - mean[k]) * rstd, g[2 * j + 1], be[2 * j + 1]));
            }
            if (!lane_on) continue;
            uint32_t* op = reinterpret_cast<uint32_t*>(out + (size_t)(t0 + k) * C0 + lane * CPL);
            if (NP == 2) *reinterpret_cast<uint2*>(op) = make_uint2(o[0], o[1]);
            else if (NP == 4) *reinterpret_cast<uint4*>(op) = make_uint4(o[0], o[1], o[NP > 2 ? 2 : 0], o[NP > 3 ? 3 : 0]);
            else {
#pragma unroll
                for (int j = 0; j < NP; ++j) {
                    if constexpr (RAGGED)
                        if (lane * CPL + 2 * j >= C0) continue;  // the part-filled lane: its pairs past C0
                    op[j] = o[j];
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------- stem, un-folded (compatibility path)
// in float32 NCHW [B,3,H,W] -- the tensor predict_ivd_locations builds (ToTensor + Normalize, cropping.py:463-472) and
// hands to model(tensor) (generic.py:389-391).  Any caller that runs the module on its own tensor (notebooks,
// BaseModel.test_inference) lands here; the dataset path uses the folded one-plane stem above.  One warp per token, lane =
// C0 / 32 (rounded up) consecutive channels; the 48 inputs of the patch are read once per token and broadcast.
// MAXC: channels per lane, C0 <= 32 * MAXC (8 up to 256 channels, 11 for convnextv2_huge's 352).
template <typename T, int MAXC = 8>
__global__ void __launch_bounds__(256) stem3_ln_kernel(const float* __restrict__ in, const float* __restrict__ w /*[C0][48] = [co][ci][ky][kx]*/,
                                                      const float* __restrict__ bias, const float* __restrict__ lnw,
                                                      const float* __restrict__ lnb, T* __restrict__ out, int B, int H, int W, int C0) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int Ho = H >> 2, Wo = W >> 2;
    const long long tokens = (long long)B * Ho * Wo;
    const int cpl = (C0 + 31) / 32;
    for (long long t = warp; t < tokens; t += nwarps) {
        const int b = (int)(t / (Ho * Wo));
        const int rem = (int)(t - (long long)b * Ho * Wo);
        const int ty = rem / Wo, tx = rem - ty * Wo;
        // lane l < 48 holds input (ci, ky, kx) = (l / 16, (l % 16) / 4, l % 4); lanes 0..15 also hold 32..47
        float x0 = 0.f, x1 = 0.f;
        {
            const int q = lane, ci = q >> 4, ky = (q >> 2) & 3, kx = q & 3;
            x0 = __ldg(in + (((size_t)b * 3 + ci) * H + (size_t)ty * 4 + ky) * W + (size_t)tx * 4 + kx);
            if (lane < 16) {
                const int q2 = 32 + lane, ci2 = q2 >> 4, ky2 = (q2 >> 2) & 3, kx2 = q2 & 3;
                x1 = __ldg(in + (((size_t)b * 3 + ci2) * H + (size_t)ty * 4 + ky2) * W + (size_t)tx * 4 + kx2);
            }
        }
        float acc[MAXC];
#pragma unroll
        for (int j = 0; j < MAXC; ++j) {
            const int c = lane * cpl + j;
            acc[j] = (j < cpl && c < C0) ? bias[c] : 0.f;
        }
        for (int q = 0; q < 48; ++q) {
            const float xv = __shfl_sync(0xffffffffu, q < 32 ? x0 : x1, q & 31);
#pragma unroll
            for (int j = 0; j < MAXC; ++j) {
                const int c = lane * cpl + j;
                if (j < cpl && c < C0) acc[j] = fmaf(xv, __ldg(w + (size_t)c * 48 + q), acc[j]);
            }
        }
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < MAXC; ++j) s += acc[j];
        const float mean = warp_sum(s) * (1.0f / C0);
        float v2 = 0.f;
#pragma unroll
        for (int j = 0; j < MAXC; ++j) {
            const int c = lane * cpl + j;
            if (j < cpl && c < C0) { const float d = acc[j] - mean; v2 = fmaf(d, d, v2); }
        }
        const float rstd = 1.0f / sqrtf(warp_sum(v2) * (1.0f / C0) + LN_EPS_BACKBONE);
#pragma unroll
        for (int j = 0; j < MAXC; ++j) {
            const int c = lane * cpl + j;
            if (j < cpl && c < C0) out[(size_t)t * C0 + c] = Cvt<T>::from_f(fmaf((acc[j] - mean) * rstd, lnw[c], lnb[c]));
        }
    }
}

// ============================================================================ depthwise 7x7 + LayerNorm
// One CTA = TH x 8 output pixels x all C channels; 8 consumer warps (one pixel column each, lane =
// channel pair) + 1 TMA producer warp.  Per 64-channel chunk the (TH+6) x 14 x 64 halo tile (4-D
// tensor map over NHWC, out-of-bounds = zero padding) and the chunk's [49][64] fp32 taps arrive in
// a STAGES-deep mbarrier ring.  Each thread slides a TH-row window down its column with packed
// FFMA2 (both channels of the pair per instruction; every halo value and tap is read from shared
// memory once per chunk).  The fp32 conv results of all chunks are parked in TENSOR MEMORY
// (tcgen05.st, the warp's own 32 lanes x 2*NCH*TH columns) instead of shared memory, so the ring
// can be deep and two CTAs fit per SM; LayerNorm then reads a pixel's C channels back with one
// tcgen05.ld per pixel, reduces with warp shuffles and writes the 16-bit K-major fc1 operand.
template <int C, int TH>
struct DwCfg {
    static constexpr int np2(int v) { int p = 1; while (p < v) p <<= 1; return p; }
    // NV = fp32 values a lane parks per pixel (2 per 64-channel chunk), padded to the next power of two: tcgen05.ld comes in
    // power-of-two column counts, and widths such as 192 / 384 / 768 / 1536 (convnext_large) have 6 / 12 / 24 / 48 values
    // NCH counts a trailing half chunk too (96 channels = 1.5 chunks, convnext_tiny / small): TMA zero-fills the channels past
    // C, the LayerNorm masks them
    static constexpr int TW = 8, CC = 64, NCH = (C + CC - 1) / CC, NV = np2(2 * NCH);
    static constexpr bool RAGGED = (C % CC) != 0;
    static constexpr int HALO_H = TH + 6, HALO_W = TW + 6;
    static constexpr int HALO_BYTES = HALO_H * HALO_W * CC * 2;
    static constexpr int W_BYTES = 49 * CC * 4;
    static constexpr int STAGE_BYTES = ((HALO_BYTES + W_BYTES + 127) / 128) * 128;
    static constexpr int COLS_PER_WARP = NV * TH;           // fp32 columns of TMEM per warp
    static constexpr int TMEM_COLS = 2 * COLS_PER_WARP;     // two warps share a lane quarter
    static constexpr int CTAS_PER_SM = TMEM_COLS <= 256 ? 2 : 1;
    static constexpr int STAGES_WANT = ((CTAS_PER_SM == 2 ? 110 * 1024 : 216 * 1024) - 2 * C * 4) / STAGE_BYTES;
    static constexpr int STAGES = STAGES_WANT < NCH ? STAGES_WANT : NCH;
    static constexpr int NUM_THREADS = 32 * (TW + 1);
    static constexpr int LN_BYTES = 2 * C * 4;             // LayerNorm weight + bias, fp32
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + LN_BYTES + 256 + 1024;  // + barriers + align slack
    static_assert(C % 32 == 0, "C must be a multiple of 32");
    static_assert(HALO_BYTES % 128 == 0, "halo stage must keep the tap buffer 128B aligned");
    static_assert(TMEM_COLS >= 32 && TMEM_COLS <= 512 && (TMEM_COLS & (TMEM_COLS - 1)) == 0, "TMEM columns: power of two <= 512");
    static_assert(STAGES >= 1, "at least one stage");
};

template <int N> struct TmemLd;  // 32 lanes x N consecutive fp32 columns: thread i gets lane (base+i)
template <> struct TmemLd<4> {
    static __device__ __forceinline__ void ld(uint32_t taddr, float* v) {
        uint32_t* r = reinterpret_cast<uint32_t*>(v);
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                     : "r"(taddr)
                     : "memory");
    }
};
template <> struct TmemLd<8> {
    static __device__ __forceinline__ void ld(uint32_t taddr, float* v) {
        uint32_t* r = reinterpret_cast<uint32_t*>(v);
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                     : "r"(taddr)
                     : "memory");
    }
};
template <> struct TmemLd<16> {
    static __device__ __forceinline__ void ld(uint32_t taddr, float* v) {
        uint32_t* r = reinterpret_cast<uint32_t*>(v);
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                     : "r"(taddr)
                     : "memory");
    }
};
template <> struct TmemLd<32> {
    static __device__ __forceinline__ void ld(uint32_t taddr, float* v) {
        uint32_t* r = reinterpret_cast<uint32_t*>(v);
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                     : "r"(taddr)
                     : "memory");
    }
};

template <> struct TmemLd<64> {  // two 32-column loads (ConvNeXt-xlarge stage 3: 2048 channels = 64 values per lane)
    static __device__ __forceinline__ void ld(uint32_t taddr, float* v) {
        TmemLd<32>::ld(taddr, v);
        TmemLd<32>::ld(taddr + 32u, v + 32);
    }
};

// thread i of the warp -> TMEM lane (base + i), two consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_x2(uint32_t taddr, uint64_t v) {
    float lo, hi;
    upk2(v, lo, hi);
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(__float_as_uint(lo)),
                 "r"(__float_as_uint(hi))
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

template <typename T> __device__ __forceinline__ uint64_t unpack2_pk(uint32_t u);
template <> __device__ __forceinline__ uint64_t unpack2_pk<__nv_bfloat16>(uint32_t u) {
    return (static_cast<uint64_t>(u & 0xFFFF0000u) << 32) | static_cast<uint64_t>(u << 16);
}
template <> __device__ __forceinline__ uint64_t unpack2_pk<__half>(uint32_t u) {
    const float2 f = Cvt<__half>::unpack2(u);
    return pk2(f.x, f.y);
}

// sum of PG=4 per-lane values over the 32 lanes, every lane receiving all 4 totals: recursive halving
// (10 shuffles) instead of 4 butterflies (20 shuffles).
__device__ __forceinline__ void warp_sum4(float (&a)[4], int lane) {
    const bool hi4 = (lane & 16) != 0, hi3 = (lane & 8) != 0;
    const float t0 = __shfl_xor_sync(0xffffffffu, hi4 ? a[0] : a[2], 16);
    const float t1 = __shfl_xor_sync(0xffffffffu, hi4 ? a[1] : a[3], 16);
    const float b0 = (hi4 ? a[2] : a[0]) + t0;  // lanes 0-15: pixel 0 / 1, lanes 16-31: pixel 2 / 3
    const float b1 = (hi4 ? a[3] : a[1]) + t1;
    float c = (hi3 ? b1 : b0) + __shfl_xor_sync(0xffffffffu, hi3 ? b0 : b1, 8);
    c += __shfl_xor_sync(0xffffffffu, c, 4);
    c += __shfl_xor_sync(0xffffffffu, c, 2);
    c += __shfl_xor_sync(0xffffffffu, c, 1);
    // lane group (bit4, bit3) now holds the total of pixel 2*bit4 + bit3
    a[0] = __shfl_sync(0xffffffffu, c, 0);
    a[1] = __shfl_sync(0xffffffffu, c, 8);
    a[2] = __shfl_sync(0xffffffffu, c, 16);
    a[3] = __shfl_sync(0xffffffffu, c, 24);
}

template <typename T, int C, int TH>
__global__ void __launch_bounds__(DwCfg<C, TH>::NUM_THREADS, DwCfg<C, TH>::CTAS_PER_SM)
dwconv_ln_kernel(const __grid_constant__ CUtensorMap x_map, const __grid_constant__ CUtensorMap w_map,
                 const float* __restrict__ bdw, const float* __restrict__ lnw, const float* __restrict__ lnb,
                 T* __restrict__ out, int H, int W, int tiles_x, int tiles_y, int num_tiles) {
    using Cfg = DwCfg<C, TH>;
    constexpr int TW = Cfg::TW, CC = Cfg::CC, STAGES = Cfg::STAGES, HALO_W = Cfg::HALO_W, NCH = Cfg::NCH, NV = Cfg::NV;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // pointer arithmetic keeps the shared address space
    uint8_t* s_stage = smem;
    float* s_ln = reinterpret_cast<float*>(smem + STAGES * Cfg::STAGE_BYTES);  // [C] weight, [C] bias
    uint64_t* s_full = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES + Cfg::LN_BYTES);
    uint64_t* s_empty = s_full + STAGES;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_empty + STAGES);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;

    if (tid == 0) {
        tma_prefetch_desc(&x_map);
        tma_prefetch_desc(&w_map);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], TW); }
        mbar_fence_init();
    }
    if (wid == TW) tmem_alloc<1>(s_tmem, Cfg::TMEM_COLS);
    for (int c = tid; c < C; c += Cfg::NUM_THREADS) { s_ln[c] = lnw[c]; s_ln[C + c] = lnb[c]; }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    pdl_launch_dependents();  // PDL: see svb_common.cuh; the waits sit in front of the first activation access

    // persistent CTA: tiles blockIdx.x, +gridDim.x, ...; the stage ring runs on across tiles, so the
    // producer is already fetching the next tile while the consumers normalise this one
    if (wid == TW) {
        // ---- TMA producer
        if (lane == 0) {
            pdl_wait();
            int it = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                int t = tile;
                const int tx = t % tiles_x; t /= tiles_x;
                const int ty = t % tiles_y;
                const int b = t / tiles_y;
                for (int k = 0; k < NCH; ++k, ++it) {
                    const int stage = it % STAGES;
                    if (it >= STAGES) mbar_wait(&s_empty[stage], ((it / STAGES) - 1) & 1);
                    uint8_t* dst = s_stage + stage * Cfg::STAGE_BYTES;
                    mbar_expect_tx(&s_full[stage], Cfg::HALO_BYTES + Cfg::W_BYTES);
                    tma_load_4d(dst, &x_map, &s_full[stage], k * CC, tx * TW - 3, ty * TH - 3, b);
                    tma_load_2d(dst + Cfg::HALO_BYTES, &w_map, &s_full[stage], k * CC, 0);
                }
            }
        }
    } else {
        // ---- consumers: warp = pixel column x0 + wid, lane = channel pair
        const uint32_t tcol0 = tmem_base + ((uint32_t)((wid & 3) * 32) << 16) + (uint32_t)((wid >> 2) * Cfg::COLS_PER_WARP);
        const uint64_t* s_gw = reinterpret_cast<const uint64_t*>(s_ln) + lane;       // channel pair (2*lane, 2*lane+1) of chunk kk at [kk*32]
        const uint64_t* s_gb = reinterpret_cast<const uint64_t*>(s_ln + C) + lane;
        int it = 0;
        pdl_wait();
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            int t = tile;
            const int tx = t % tiles_x; t /= tiles_x;
            const int ty = t % tiles_y;
            const int b = t / tiles_y;
            const int x = tx * TW + wid, y0 = ty * TH;
            auto ch_ok = [&](int kk) { return !Cfg::RAGGED || kk * CC + 2 * lane < C; };  // this lane's channel pair of chunk kk exists
            float2 bias_next = ch_ok(0) ? __ldg(reinterpret_cast<const float2*>(bdw + 2 * lane)) : make_float2(0.f, 0.f);
            for (int k = 0; k < NCH; ++k, ++it) {
                const int stage = it % STAGES;
                const float2 bias = bias_next;  // loaded one chunk ahead: no global-load latency in front of the FMAs
                if (k + 1 < NCH) bias_next = ch_ok(k + 1) ? __ldg(reinterpret_cast<const float2*>(bdw + (k + 1) * CC + 2 * lane)) : make_float2(0.f, 0.f);
                mbar_wait(&s_full[stage], (it / STAGES) & 1);
                const uint32_t* halo = reinterpret_cast<const uint32_t*>(s_stage + stage * Cfg::STAGE_BYTES) + wid * 32 + lane;  // [HALO_H][HALO_W][32] ch pairs
                const uint64_t* taps = reinterpret_cast<const uint64_t*>(s_stage + stage * Cfg::STAGE_BYTES + Cfg::HALO_BYTES) + lane;  // [49][32] fp32 pairs
                uint64_t acc[TH];
#pragma unroll
                for (int i = 0; i < TH; ++i) acc[i] = pk2(bias.x, bias.y);
#pragma unroll DW_KX_UNROLL
                for (int kx = 0; kx < 7; ++kx) {
                    uint64_t col[TH + 6], wv[7];
#pragma unroll
                    for (int r = 0; r < TH + 6; ++r) col[r] = unpack2_pk<T>(halo[(r * HALO_W + kx) * 32]);
#pragma unroll
                    for (int ky = 0; ky < 7; ++ky) wv[ky] = taps[(ky * 7 + kx) * 32];
#pragma unroll
                    for (int ky = 0; ky < 7; ++ky) {
#pragma unroll
                        for (int i = 0; i < TH; ++i) acc[i] = fma2(col[i + ky], wv[ky], acc[i]);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive_relaxed(&s_empty[stage]);  // this warp is done with the stage (all of it is in registers)
                // park the chunk's results: pixel i of the column -> columns [i*NV + 2k, +2)
#pragma unroll
                for (int i = 0; i < TH; ++i) tmem_st_x2(tcol0 + (uint32_t)(i * NV + 2 * k), acc[i]);
            }
            tmem_st_wait();

            // ---- LayerNorm over C: one tcgen05.ld per pixel gives the lane its 2 channels of every chunk
            constexpr int PG = NV <= 32 ? 4 : 1;  // pixels in flight (one at 2048 channels: 64 values per lane already)
            static_assert(TH % PG == 0, "TH must be a multiple of the pixel group");
#pragma unroll 1
            for (int p0 = 0; p0 < TH; p0 += PG) {
                float v[PG][NV];
#pragma unroll
                for (int g = 0; g < PG; ++g) TmemLd<NV>::ld(tcol0 + (uint32_t)((p0 + g) * NV), v[g]);
                tmem_ld_wait();
                float s[PG], q[PG];
#pragma unroll
                for (int g = 0; g < PG; ++g) {
                    uint64_t a2 = pk2(v[g][0], v[g][1]);
#pragma unroll
                    for (int kk = 1; kk < NCH; ++kk) a2 = add2(a2, pk2(v[g][2 * kk], v[g][2 * kk + 1]));
                    float lo, hi;
                    upk2(a2, lo, hi);
                    s[g] = lo + hi;
                }
                if constexpr (PG == 4) warp_sum4(s, lane);
                else {
#pragma unroll
                    for (int g = 0; g < PG; ++g) s[g] = warp_sum(s[g]);
                }
                uint64_t d[PG][NCH];
#pragma unroll
                for (int g = 0; g < PG; ++g) {
                    const float nm = -s[g] * (1.0f / C);
                    const uint64_t nm2 = pk2(nm, nm);
                    uint64_t a2 = pk2(0.f, 0.f);
#pragma unroll
                    for (int kk = 0; kk < NCH; ++kk) {
                        d[g][kk] = add2(pk2(v[g][2 * kk], v[g][2 * kk + 1]), nm2);
                        if (ch_ok(kk)) a2 = fma2(d[g][kk], d[g][kk], a2);  // channels past C (zero-filled) stay out of the variance
                    }
                    float lo, hi;
                    upk2(a2, lo, hi);
                    q[g] = lo + hi;
                }
                if constexpr (PG == 4) warp_sum4(q, lane);
                else {
#pragma unroll
                    for (int g = 0; g < PG; ++g) q[g] = warp_sum(q[g]);
                }
#pragma unroll
                for (int g = 0; g < PG; ++g) {
                    const int y = y0 + p0 + g;
                    if (y < H && x < W) {  // warp-uniform
                        const float rstd = 1.0f / sqrtf(q[g] * (1.0f / C) + LN_EPS_BACKBONE);
                        const uint64_t r2 = pk2(rstd, rstd);
                        uint32_t* op = reinterpret_cast<uint32_t*>(out + (((size_t)b * H + y) * W + x) * C) + lane;
#pragma unroll
                        for (int kk = 0; kk < NCH; ++kk) {
                            float lo, hi;
                            upk2(fma2(mul2(d[g][kk], r2), s_gw[kk * 32], s_gb[kk * 32]), lo, hi);
                            if (ch_ok(kk)) op[kk * (CC / 2)] = Cvt<T>::pack2(lo, hi);
                        }
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (wid == TW) tmem_dealloc<1>(tmem_base, Cfg::TMEM_COLS);
}

// ============================================================================ depthwise 7x7, LayerNorm folded into fc1
// The LayerNorm that follows the depthwise convolution is an affine map PER TOKEN; composed with fc1 it is
//     fc1(LN(y))[m, n] = rstd_m * (sum_k W1[n,k] g_k y[m,k]) - rstd_m mu_m * (sum_k W1[n,k] g_k) + (sum_k W1[n,k] b_k + b1[n])
// so this kernel writes the RAW convolution y (16-bit, the fc1 A operand) plus two numbers per token (rstd_m, -mu_m rstd_m) and
// the fc1 GEMM applies them in its epilogue (GEMM_LNGELU: acc over W1 * diag(g), column constants s_n and t_n).  What that buys:
//   * no parking of a tile's fp32 results for a second (LayerNorm) pass: no TMEM capacity limit on the tile, so a warp owns TWO
//     pixel columns (every halo value feeds both; the loop reaches 83 instead of 70 FMA / clk / SM, scripts/ubench/convloop2.cu)
//   * the LayerNorm pass itself (a fifth of the old kernel's instructions) shrinks to two accumulations per value
//   * the A operand is not rounded a second time after normalisation: predicted AND measured coordinate error goes DOWN
//     (scripts/emulate_precision.py: fp16 trained-like 0.176 -> 0.119 px)
// The statistics are taken from the fp32 results before rounding (mean of the rounded values differs by the MEAN rounding error,
// 2^-12 |y| / sqrt(C): far below one element's rounding).  One pass: var = E[y^2] - mu^2 in fp32 over C <= 2816 values
// (convnextv2_huge's last stage; each lane adds C / 64 values per pixel, the 32 lane sums meet in a shuffle tree).
// Per thread 16 pixels x packed (sum, sum of squares) pairs have to live across the channel chunks; 64 more registers next to
// the convolution's 88 would spill, so between chunks they are parked in TENSOR MEMORY (two tcgen05.st / .ld pairs per chunk,
// against 784 FFMA2) -- the epilogue of a chunk is then one F2FP, one STG and two packed FMA-pipe operations per pixel.
template <int C, int TH>
struct DwRawCfg {
    static constexpr int NC = 2, WARPS = 8, TW = WARPS * NC, CC = 64, NCH = (C + CC - 1) / CC;
    static constexpr bool RAGGED = (C % CC) != 0;
    static constexpr int HALO_H = TH + 6, HALO_W = TW + 6;
    static constexpr int HALO_BYTES = HALO_H * HALO_W * CC * 2;
    static constexpr int W_BYTES = 49 * CC * 4;
    static constexpr int STAGE_BYTES = ((HALO_BYTES + W_BYTES + 127) / 128) * 128;
    static constexpr int STAGES = NCH < 2 ? NCH : 2;
    static constexpr int ST = 4 * NC * TH;  // statistics words per thread: (sum lo, sum hi, sumsq lo, sumsq hi) per pixel
    static constexpr int TMEM_COLS = 2 * ST < 32 ? 32 : 2 * ST;  // two warps per lane quarter
    static_assert(ST == 32 || ST == 64, "TH = 4 or 8");
    // eight warps, no separate producer warp: a ninth warp makes 18 warps per SM = 5 on one scheduler, which caps every thread
    // at 96 registers (the loop needs ~110); lane 0 of warp 0 issues the TMA loads between its own chunks instead
    static constexpr int NUM_THREADS = 32 * WARPS;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 256 + 1024;  // + barriers + align slack
    static_assert(C % 32 == 0, "C must be a multiple of 32");
    static_assert(HALO_BYTES % 128 == 0, "halo stage must keep the tap buffer 128B aligned");
    static_assert(2 * SMEM_BYTES <= 227 * 1024, "two CTAs per SM");
};

__device__ __forceinline__ void tmem_st_32(uint32_t taddr, const float (&v)[32]) {
    const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
        "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
        "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
        "r"(r[31])
        : "memory");
}

template <typename T, int C, int TH>
__global__ void __launch_bounds__(DwRawCfg<C, TH>::NUM_THREADS, 2)
dwconv_raw_kernel(const __grid_constant__ CUtensorMap x_map, const __grid_constant__ CUtensorMap w_map,
                  const float* __restrict__ bdw, T* __restrict__ out, float2* __restrict__ rowstat, int H, int W, int tiles_x,
                  int tiles_y, int num_tiles, int b0) {
    // images [b0, b0 + num_tiles / (tiles_x * tiles_y)) of the micro-batch the tensor map describes
    using Cfg = DwRawCfg<C, TH>;
    constexpr int TW = Cfg::TW, CC = Cfg::CC, STAGES = Cfg::STAGES, HALO_W = Cfg::HALO_W, NCH = Cfg::NCH, WARPS = Cfg::WARPS;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* s_stage = smem;
    uint64_t* s_full = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
    uint64_t* s_empty = s_full + STAGES;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_empty + STAGES);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) {
        tma_prefetch_desc(&x_map);
        tma_prefetch_desc(&w_map);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], WARPS); }
        mbar_fence_init();
    }
    if (wid == 0) tmem_alloc<1>(s_tmem, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    pdl_launch_dependents();

    {
        // ---- warp = pixel columns x0, x0 + 1; lane = channel pair of the chunk.  Lane 0 of warp 0 is also the TMA producer:
        // before it starts iteration `it` it issues the load of iteration it + STAGES - 1 (the stage iteration it - 1 used; every
        // warp has arrived on its "empty" barrier by the time the slowest of them finished it), so a load has one whole chunk of
        // arithmetic to land.  The ring runs on across tiles.
        const int my_tiles = blockIdx.x < num_tiles ? (num_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
        const int total_it = my_tiles * NCH;
        int pj = 0;  // next iteration whose load has not been issued (producer lane only)
        auto produce_to = [&](int last) {
            for (; pj <= last && pj < total_it; ++pj) {
                const int stage = pj % STAGES;
                if (pj >= STAGES) mbar_wait(&s_empty[stage], ((pj / STAGES) - 1) & 1);
                int t = (int)blockIdx.x + (pj / NCH) * (int)gridDim.x;
                const int k = pj % NCH;
                const int tx = t % tiles_x; t /= tiles_x;
                const int ty = t % tiles_y;
                const int b = b0 + t / tiles_y;
                uint8_t* dst = s_stage + stage * Cfg::STAGE_BYTES;
                mbar_expect_tx(&s_full[stage], Cfg::HALO_BYTES + Cfg::W_BYTES);
                tma_load_4d(dst, &x_map, &s_full[stage], k * CC, tx * TW - 3, ty * TH - 3, b);
                tma_load_2d(dst + Cfg::HALO_BYTES, &w_map, &s_full[stage], k * CC, 0);
            }
        };
        const bool producer = wid == 0 && lane == 0;
        const uint32_t tcol0 = tmem_base + ((uint32_t)((wid & 3) * 32) << 16) + (uint32_t)((wid >> 2) * Cfg::ST);
        int it = 0;
        pdl_wait();
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            int t = tile;
            const int tx = t % tiles_x; t /= tiles_x;
            const int ty = t % tiles_y;
            const int b = b0 + t / tiles_y;
            const int x0 = tx * TW + 2 * wid, y0 = ty * TH;
            auto ch_ok = [&](int kk) { return !Cfg::RAGGED || kk * CC + 2 * lane < C; };
            float2 bias_next = ch_ok(0) ? __ldg(reinterpret_cast<const float2*>(bdw + 2 * lane)) : make_float2(0.f, 0.f);
            // per pixel p = c * TH + i: st[4p .. 4p+1] = packed sum, st[4p+2 .. 4p+3] = packed sum of squares of this lane's two
            // channels over the chunks so far
            float st[Cfg::ST];
            const int nrow = min(TH, H - y0);  // rows of the tile inside the image
            uint32_t* const orow0 = reinterpret_cast<uint32_t*>(out + (((size_t)b * H + y0) * W + x0) * C) + lane;
            const size_t row_pitch = (size_t)W * (C / 2);
            for (int k = 0; k < NCH; ++k, ++it) {
                const int stage = it % STAGES;
                const float2 bias = bias_next;
                if (k + 1 < NCH) bias_next = ch_ok(k + 1) ? __ldg(reinterpret_cast<const float2*>(bdw + (k + 1) * CC + 2 * lane)) : make_float2(0.f, 0.f);
                if (producer) produce_to(it + STAGES - 1);
                __syncwarp();
                mbar_wait(&s_full[stage], (it / STAGES) & 1);
                const uint32_t* halo = reinterpret_cast<const uint32_t*>(s_stage + stage * Cfg::STAGE_BYTES) + (2 * wid) * 32 + lane;  // [HALO_H][HALO_W][32] pairs
                const uint64_t* taps = reinterpret_cast<const uint64_t*>(s_stage + stage * Cfg::STAGE_BYTES + Cfg::HALO_BYTES) + lane;  // [49][32] fp32 pairs
                uint64_t acc0[TH], acc1[TH];
#pragma unroll
                for (int i = 0; i < TH; ++i) acc0[i] = acc1[i] = pk2(bias.x, bias.y);
                // input column j of the 8 the two outputs read: tap kx = j for output column 0, kx = j - 1 for column 1
                {
                    uint64_t col[TH + 6], w0[7];
#pragma unroll
                    for (int r = 0; r < TH + 6; ++r) col[r] = unpack2_pk<T>(halo[(r * HALO_W + 0) * 32]);
#pragma unroll
                    for (int ky = 0; ky < 7; ++ky) w0[ky] = taps[(ky * 7 + 0) * 32];
#pragma unroll
                    for (int ky = 0; ky < 7; ++ky)
#pragma unroll
                        for (int i = 0; i < TH; ++i) acc0[i] = fma2(col[i + ky], w0[ky], acc0[i]);
                }
#pragma unroll 1
                for (int j = 1; j < 7; ++j) {
                    uint64_t col[TH + 6], w0[7], w1[7];
#pragma unroll
                    for (int r = 0; r < TH + 6; ++r) col[r] = unpack2_pk<T>(halo[(r * HALO_W + j) * 32]);
#pragma unroll
                    for (int ky = 0; ky < 7; ++ky) { w0[ky] = taps[(ky * 7 + j) * 32]; w1[ky] = taps[(ky * 7 + j - 1) * 32]; }
#pragma unroll
                    for (int ky = 0; ky < 7; ++ky)
#pragma unroll
                        for (int i = 0; i < TH; ++i) { acc0[i] = fma2(col[i + ky], w0[ky], acc0[i]); acc1[i] = fma2(col[i + ky], w1[ky], acc1[i]); }
                }
                {
                    uint64_t col[TH + 6], w1[7];
#pragma unroll
                    for (int r = 0; r < TH + 6; ++r) col[r] = unpack2_pk<T>(halo[(r * HALO_W + 7) * 32]);
#pragma unroll
                    for (int ky = 0; ky < 7; ++ky) w1[ky] = taps[(ky * 7 + 6) * 32];
#pragma unroll
                    for (int ky = 0; ky < 7; ++ky)
#pragma unroll
                        for (int i = 0; i < TH; ++i) acc1[i] = fma2(col[i + ky], w1[ky], acc1[i]);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive_relaxed(&s_empty[stage]);  // the stage is in registers
                // ---- round to 16 bits and store the fc1 operand; fold the fp32 values into the token statistics
                if (k > 0) {
                    TmemLd<32>::ld(tcol0, st);
                    if constexpr (Cfg::ST == 64) TmemLd<32>::ld(tcol0 + 32u, st + 32);
                    tmem_ld_wait();
                } else {
#pragma unroll
                    for (int q = 0; q < Cfg::ST; ++q) st[q] = 0.f;
                }
                const bool okc = ch_ok(k);
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const bool okx = okc && x0 + c < W;
                    uint32_t* op = orow0 + c * (C / 2) + k * (CC / 2);
#pragma unroll
                    for (int i = 0; i < TH; ++i) {
                        const uint64_t v = c == 0 ? acc0[i] : acc1[i];
                        float lo, hi;
                        upk2(v, lo, hi);
                        const int p = c * TH + i;
                        uint64_t s2 = pk2(st[4 * p], st[4 * p + 1]), q2 = pk2(st[4 * p + 2], st[4 * p + 3]);
                        s2 = add2(s2, v);
                        q2 = fma2(v, v, q2);
                        upk2(s2, st[4 * p], st[4 * p + 1]);
                        upk2(q2, st[4 * p + 2], st[4 * p + 3]);
                        if (okx && i < nrow) *op = Cvt<T>::pack2(lo, hi);
                        op += row_pitch;
                    }
                }
                if (k + 1 < NCH) {
                    if constexpr (Cfg::ST == 64) {
                        tmem_st_32(tcol0, *reinterpret_cast<const float(*)[32]>(st));
                        tmem_st_32(tcol0 + 32u, *reinterpret_cast<const float(*)[32]>(st + 32));
                    } else {
                        tmem_st_32(tcol0, *reinterpret_cast<const float(*)[32]>(st));
                    }
                    tmem_st_wait();
                }
            }
            // ---- token statistics: sum over the 32 lanes (every channel of the pixel), then (rstd, -mu * rstd)
#pragma unroll
            for (int g4 = 0; g4 < (2 * TH) / 4; ++g4) {
                float s4[4], q4[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int p = 4 * g4 + j;
                    s4[j] = st[4 * p] + st[4 * p + 1];
                    q4[j] = st[4 * p + 2] + st[4 * p + 3];
                }
                warp_sum4(s4, lane);
                warp_sum4(q4, lane);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int p = 4 * g4 + j;
                    const int x = x0 + p / TH, y = y0 + p % TH;
                    if (lane == p && x < W && y < H) {
                        const float mu = s4[j] * (1.0f / C);
                        const float var = fmaxf(fmaf(-mu, mu, q4[j] * (1.0f / C)), 0.0f);
                        const float rstd = 1.0f / sqrtf(var + LN_EPS_BACKBONE);
                        rowstat[((size_t)b * H + y) * W + x] = make_float2(rstd, -mu * rstd);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (wid == 0) tmem_dealloc<1>(tmem_base, Cfg::TMEM_COLS);
}

// ============================================================================ tcgen05 GEMM
// D[M,N] = epilogue(A[M,K] * Wt[N,K]^T); A, Wt K-major 16-bit; fp32 accumulation in TMEM.
// Persistent CTAs, BK = 64 (one 128-byte swizzle atom), warp roles:
//   warp 0      TMA producer (one elected lane)
//   warp 1      TMEM allocator + tcgen05.mma issuer (one lane; the pair leader only when CG == 2)
//   warps 2..17 epilogue: tcgen05.ld -> bias / GELU / gamma*+residual -> 16-bit, staged through a
//               per-warp 32x32 swizzled shared-memory box and written (residual: also read) by TMA,
//               so global traffic is whole 64-byte row segments instead of 32 scattered rows per store.
// Two TMEM accumulator stages (2 x BN columns) let the epilogue of tile i overlap the MMAs of tile i+1.
//
// CG == 2 (cta_group::2): a cluster of two CTAs computes a 256 x BN tile.  Each CTA stages its own
// 128 rows of A and HALF of the W tile (BN/2 rows), so the W traffic from L2 per output element is
// halved; the leader issues tcgen05.mma.cta_group::2 for both and multicasts the commits.
// GEMM_LNGELU: fc1 with the block's LayerNorm folded in (see dwconv_raw_kernel): GELU(rstd_m * acc + (-mu_m rstd_m) * s_n + t_n),
// (rstd_m, -mu_m rstd_m) = rowstat[m], s_n passed as `gamma`, t_n as `bias`
enum GemmMode { GEMM_GELU = 0, GEMM_RESID = 1, GEMM_BIAS = 2, GEMM_LNGELU = 3 };

template <int BN, int CG>
struct GemmCfg {
    static constexpr int BM = 128, BK = 64;
    static constexpr int B_ROWS = BN / CG;             // rows of W this CTA stages
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = B_ROWS * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int STAGES = (192 * 1024) / STAGE_BYTES;  // 4 (48 KB), 6 (32 KB) or 8 (24 KB)
    static constexpr int EPI_WARPS = 16;                       // 4 per TMEM lane quarter: the epilogue is latency-bound per warp
    static constexpr int EPI_BUF_BYTES = 32 * 32 * 2;          // one 32x32 16-bit box per warp
    static constexpr int EPI_BYTES = EPI_WARPS * EPI_BUF_BYTES;
    static constexpr int NUM_BARS = 2 * STAGES + 4 + EPI_WARPS;
    static constexpr int TMEM_COLS = 2 * BN;  // 256 or 512: power of two
    static constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + 512 + 1024;
    static_assert(NUM_BARS * 8 + 8 <= 512, "barrier area");
    static_assert(B_BYTES % 1024 == 0, "B stage must keep 1024-byte (swizzle atom) alignment");
};

template <typename T> struct UmmaFmt;
template <> struct UmmaFmt<__nv_bfloat16> { static constexpr uint32_t v = 1; };
template <> struct UmmaFmt<__half> { static constexpr uint32_t v = 0; };

// GELU of a packed pair, 16-bit output: relu(x) - |x| * E(|x|), E(u) = erfc(u / sqrt2) / 2 = exp2(u * p(u) - 1) with a
// cubic p fitted for min-max |GELU error| (8.6e-6 on the whole real line, scripts/fit_gelu.py; the output is rounded to
// 16 bits, ulp >= 1.5e-5 wherever that matters).  Written in v = -min(|x|, 12) (one FMNMX with |.| and - modifiers), so
// the product v * E is already the negative correction; beyond |x| = 12 the exponent is < -74 and the result is relu(x).
// FMA-pipe cost per pair: 1 (bias, at the caller) + 4 (exponent) + 1 + 1 = 7 packed ops; the epilogues that call this
// are bound by exactly that pipe (FFMA2 issues at ~2.4 clk on B200).
template <typename T>
__device__ __forceinline__ uint32_t gelu_pack2(uint64_t x) {
    float x0, x1;
    upk2(x, x0, x1);
    const uint64_t v = pk2(fmaxf(-fabsf(x0), -12.0f), fmaxf(-fabsf(x1), -12.0f));
    uint64_t r = pk2(4.16166e-03f, 4.16166e-03f);
    r = fma2(r, v, pk2(4.573539e-02f, 4.573539e-02f));
    r = fma2(r, v, pk2(-4.6493057e-01f, -4.6493057e-01f));
    r = fma2(r, v, pk2(1.14956693e+00f, 1.14956693e+00f));
    r = fma2(r, v, pk2(-1.0f, -1.0f));
    float r0, r1, e0, e1;
    upk2(r, r0, r1);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(r0));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(r1));
    const uint64_t y = fma2(v, pk2(e0, e1), pk2(fmaxf(x0, 0.0f), fmaxf(x1, 0.0f)));
    float y0, y1;
    upk2(y, y0, y1);
    return Cvt<T>::pack2(y0, y1);
}

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <typename T, int BN, int MODE, int CG>
__global__ void __launch_bounds__(GemmCfg<BN, CG>::NUM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap a_map, const __grid_constant__ CUtensorMap w_map,
            const __grid_constant__ CUtensorMap out_map, const __grid_constant__ CUtensorMap resid_map,
            const float* __restrict__ bias, const float* __restrict__ gamma, int M, int N, int K,
            const float2* __restrict__ rowstat, int m0) {
    // rows [m0, M) of the operands the tensor maps describe (m0 a multiple of the tile height: a sub-batch of a micro-batch)
    using Cfg = GemmCfg<BN, CG>;
    constexpr int STAGES = Cfg::STAGES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // pointer arithmetic keeps the shared address space
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES * Cfg::A_BYTES;
    uint8_t* sEpi = smem + STAGES * Cfg::STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sEpi + Cfg::EPI_BYTES);
    uint64_t* full = bars;                 // [STAGES] TMA -> MMA   (the leader's copy is the live one when CG == 2)
    uint64_t* empty = bars + STAGES;       // [STAGES] MMA -> TMA   (multicast to both CTAs)
    uint64_t* tfull = bars + 2 * STAGES;   // [2] MMA -> epilogue   (multicast to both CTAs)
    uint64_t* tempty = tfull + 2;          // [2] epilogue -> MMA   (leader's copy; both CTAs' epilogue warps arrive)
    uint64_t* rfull = tempty + 2;          // [EPI_WARPS] residual box landed
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + Cfg::NUM_BARS);

    // the warp index through a shuffle: provably warp-uniform, so the role branches are uniform branches
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const uint32_t rank = CG == 2 ? cluster_ctarank() : 0u;
    const int tiles_n = (N + BN - 1) / BN;
    const int tiles_m = (M - m0 + Cfg::BM * CG - 1) / (Cfg::BM * CG);
    const int num_tiles = tiles_m * tiles_n;
    const int num_kb = (K + Cfg::BK - 1) / Cfg::BK;
    const int tile0 = (int)blockIdx.x / CG, tile_step = (int)gridDim.x / CG;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&a_map);
        tma_prefetch_desc(&w_map);
        tma_prefetch_desc(&out_map);
        if (MODE == GEMM_RESID) tma_prefetch_desc(&resid_map);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], Cfg::EPI_WARPS * CG); }
        for (int s = 0; s < Cfg::EPI_WARPS; ++s) mbar_init(&rfull[s], 1);
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc<CG>(tmem_ptr, Cfg::TMEM_COLS);
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    // PDL: the set-up above overlapped the previous kernel's tail; every thread that touches activations waits here
    pdl_launch_dependents();

    if (warp == 0) {
        if (lane == 0) {
            pdl_wait();
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = tile0; tile < num_tiles; tile += tile_step) {
                const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
                const int row_a = m0 + (m_blk * CG + (int)rank) * Cfg::BM;
                const int row_b = n_blk * BN + (int)rank * Cfg::B_ROWS;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    if (CG == 1) {
                        mbar_expect_tx(&full[stage], Cfg::STAGE_BYTES);
                        tma_load_2d(sA + stage * Cfg::A_BYTES, &a_map, &full[stage], kb * Cfg::BK, row_a);
                        tma_load_2d(sB + stage * Cfg::B_BYTES, &w_map, &full[stage], kb * Cfg::BK, row_b);
                    } else {
                        // both CTAs' bytes are counted on the leader's barrier; only the leader arrives
                        if (rank == 0) mbar_expect_tx(&full[stage], 2 * Cfg::STAGE_BYTES);
                        const uint32_t lbar = mapa_shared(smem_u32(&full[stage]), 0);
                        tma_load_2d_pair(sA + stage * Cfg::A_BYTES, &a_map, lbar, kb * Cfg::BK, row_a);
                        tma_load_2d_pair(sB + stage * Cfg::B_BYTES, &w_map, lbar, kb * Cfg::BK, row_b);
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (rank == 0) {
            // The WHOLE warp runs this loop and one elected lane issues (predicated instructions, no branch around them): the
            // descriptors then stay in uniform registers.  With `if (lane == 0)` around the loop every MMA operand went through an
            // ELECT / R2UR.BROADCAST / BRA.U.ANY sequence, ~130 clk of issue latency per MMA (measured in dwconv_rawtc_kernel) --
            // as long as the 128 clk of tensor work of a 128 x 256 x 16 MMA.
            // instruction descriptor: D=f32, A/B = T, both K-major, M = 128*CG, N = BN
            constexpr uint32_t idesc = (1u << 4) | (UmmaFmt<T>::v << 7) | (UmmaFmt<T>::v << 10) |
                                       ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((Cfg::BM * CG) >> 4) << 24);
            const uint32_t lead = elect_one() ? 1u : 0u;
            const uint32_t tm0 = __shfl_sync(0xffffffffu, tmem_base, 0);
            const uint64_t a00 = make_sw128_kmajor_desc(smem_u32(sA)), b00 = make_sw128_kmajor_desc(smem_u32(sB));
            int stage = 0;
            uint32_t phase = 0;
            int as = 0;
            uint32_t aphase = 0;
            for (int tile = tile0; tile < num_tiles; tile += tile_step) {
                mbar_wait(&tempty[as], aphase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tm0 + (uint32_t)(as * BN);
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint64_t adesc = a00 + (uint64_t)(stage * (Cfg::A_BYTES >> 4));
                    const uint64_t bdesc = b00 + (uint64_t)(stage * (Cfg::B_BYTES >> 4));
#pragma unroll
                    for (int k = 0; k < Cfg::BK / 16; ++k)  // +32 B per UMMA_K inside the swizzle atom
                        tc_mma_f16_if<CG>(lead, d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
                    tc_commit_if<CG>(lead, &empty[stage]);  // frees the smem slot (in both CTAs) once these MMAs retire
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                tc_commit_if<CG>(lead, &tfull[as]);  // accumulator complete -> epilogue (both CTAs)
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else {
        const int ew = warp - 2;
        const int q = warp & 3;             // TMEM lane quarter this warp may access
        const int slice = ew >> 2;          // which quarter of the BN columns
        constexpr int CW = BN / (Cfg::EPI_WARPS / 4);  // columns per warp: 64 or 32
        constexpr int CH = CW / 32;         // 32-column chunks per warp
        uint8_t* ebuf_p = sEpi + ew * Cfg::EPI_BUF_BYTES;
        const uint32_t ebuf = smem_u32(ebuf_p);
        uint64_t* rf = rfull + ew;
        // 64-byte rows, SWIZZLE_64B: 16-byte piece i of row r lives at r*64 + ((i ^ ((r >> 1) & 3)) << 4)
        const uint32_t row_off = ebuf + (uint32_t)lane * 64u;
        const uint32_t swz = ((uint32_t)lane >> 1) & 3u;
        uint32_t rph = 0;
        int as = 0;
        uint32_t aphase = 0;
        pdl_wait();
        for (int tile = tile0; tile < num_tiles; tile += tile_step) {
            const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
            const int row0 = m0 + (m_blk * CG + (int)rank) * Cfg::BM + q * 32;
            const int colw = n_blk * BN + slice * CW;
            const bool active = colw < N && row0 < M;  // warp-uniform
            uint64_t ra2 = 0, rb2 = 0;  // GEMM_LNGELU: this thread's row (token): (rstd, rstd) and (-mu rstd, -mu rstd)
            if (MODE == GEMM_LNGELU) {
                const float2 rs = (active && row0 + lane < M) ? __ldg(rowstat + row0 + lane) : make_float2(0.f, 0.f);
                ra2 = pk2(rs.x, rs.x);
                rb2 = pk2(rs.y, rs.y);
            }
            if (MODE == GEMM_RESID && active && lane == 0) {
                // the first residual box of the tile arrives while the MMAs are still running
                bulk_wait_read<0>();
                mbar_expect_tx(rf, Cfg::EPI_BUF_BYTES);
                tma_load_2d(ebuf_p, &resid_map, rf, colw, row0);
            }
            mbar_wait(&tfull[as], aphase);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < CH; ++c) {
                const int col = colw + c * 32;
                if (!active || col >= N) break;
                uint32_t r[32];
                tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN + slice * CW + c * 32), r);
                if (MODE == GEMM_RESID) {
                    if (c > 0 && lane == 0) {
                        bulk_wait_read<0>();
                        mbar_expect_tx(rf, Cfg::EPI_BUF_BYTES);
                        tma_load_2d(ebuf_p, &resid_map, rf, col, row0);
                    }
                } else {
                    if (lane == 0) bulk_wait_read<0>();  // the previous store has left the buffer
                    __syncwarp();
                }
                tmem_ld_wait();
                if (MODE == GEMM_RESID) {
                    mbar_wait(rf, rph);
                    rph ^= 1u;
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t addr = row_off + ((((uint32_t)i) ^ swz) << 4);
                    const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + col) + 2 * i);
                    const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + col) + 2 * i + 1);
                    uint64_t v01, v23, v45, v67;
                    if (MODE == GEMM_LNGELU) {
                        const float4 s0 = __ldg(reinterpret_cast<const float4*>(gamma + col) + 2 * i);
                        const float4 s1 = __ldg(reinterpret_cast<const float4*>(gamma + col) + 2 * i + 1);
                        v01 = fma2(ra2, pk2(__uint_as_float(r[8 * i + 0]), __uint_as_float(r[8 * i + 1])), fma2(rb2, pk2(s0.x, s0.y), pk2(b0.x, b0.y)));
                        v23 = fma2(ra2, pk2(__uint_as_float(r[8 * i + 2]), __uint_as_float(r[8 * i + 3])), fma2(rb2, pk2(s0.z, s0.w), pk2(b0.z, b0.w)));
                        v45 = fma2(ra2, pk2(__uint_as_float(r[8 * i + 4]), __uint_as_float(r[8 * i + 5])), fma2(rb2, pk2(s1.x, s1.y), pk2(b1.x, b1.y)));
                        v67 = fma2(ra2, pk2(__uint_as_float(r[8 * i + 6]), __uint_as_float(r[8 * i + 7])), fma2(rb2, pk2(s1.z, s1.w), pk2(b1.z, b1.w)));
                    } else {
                        v01 = add2(pk2(__uint_as_float(r[8 * i + 0]), __uint_as_float(r[8 * i + 1])), pk2(b0.x, b0.y));
                        v23 = add2(pk2(__uint_as_float(r[8 * i + 2]), __uint_as_float(r[8 * i + 3])), pk2(b0.z, b0.w));
                        v45 = add2(pk2(__uint_as_float(r[8 * i + 4]), __uint_as_float(r[8 * i + 5])), pk2(b1.x, b1.y));
                        v67 = add2(pk2(__uint_as_float(r[8 * i + 6]), __uint_as_float(r[8 * i + 7])), pk2(b1.z, b1.w));
                    }
                    uint4 o;
                    if (MODE == GEMM_GELU || MODE == GEMM_LNGELU) {
                        o = make_uint4(gelu_pack2<T>(v01), gelu_pack2<T>(v23), gelu_pack2<T>(v45), gelu_pack2<T>(v67));
                    } else {
                        if (MODE == GEMM_RESID) {
                            const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + col) + 2 * i);
                            const float4 g1 = __ldg(reinterpret_cast<const float4*>(gamma + col) + 2 * i + 1);
                            const uint4 rv = lds128(addr);
                            const float2 x01 = Cvt<T>::unpack2(rv.x), x23 = Cvt<T>::unpack2(rv.y);
                            const float2 x45 = Cvt<T>::unpack2(rv.z), x67 = Cvt<T>::unpack2(rv.w);
                            v01 = fma2(pk2(g0.x, g0.y), v01, pk2(x01.x, x01.y));
                            v23 = fma2(pk2(g0.z, g0.w), v23, pk2(x23.x, x23.y));
                            v45 = fma2(pk2(g1.x, g1.y), v45, pk2(x45.x, x45.y));
                            v67 = fma2(pk2(g1.z, g1.w), v67, pk2(x67.x, x67.y));
                        }
                        float f0, f1, f2, f3, f4, f5, f6, f7;
                        upk2(v01, f0, f1); upk2(v23, f2, f3); upk2(v45, f4, f5); upk2(v67, f6, f7);
                        o = make_uint4(Cvt<T>::pack2(f0, f1), Cvt<T>::pack2(f2, f3), Cvt<T>::pack2(f4, f5), Cvt<T>::pack2(f6, f7));
                    }
                    sts128(addr, o);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    tma_store_2d(&out_map, ebuf_p, col, row0);
                    bulk_commit();
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                // the accumulator stage is in registers (tcgen05.wait::ld above): nothing to release, so no fence
                if (CG == 1 || rank == 0) mbar_arrive_relaxed(&tempty[as]);
                else mbar_arrive_cluster_relaxed(mapa_shared(smem_u32(&tempty[as]), 0));
            }
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
        if (lane == 0) bulk_wait_all();  // shared memory must outlive the last TMA stores
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 1) tmem_dealloc<CG>(tmem_base, Cfg::TMEM_COLS);
}

// ============================================================================ fused ConvNeXt MLP (CTA pair)
// x <- x + gamma * (fc2(GELU(fc1(a) + b1)) + b2) for one block in ONE kernel: the 4C-wide hidden activation never
// leaves the SM.  A cluster of two CTAs owns 256 tokens (128 each, cta_group::2); the hidden dimension is walked in
// chunks of 64:
//     Hacc[128 tok, 64]   = A[128 tok, C] * W1[chunk]^T            (tcgen05, accumulator in TMEM, NB-fold buffered)
//     Hs  [128 tok, 64]   = bf16(GELU(Hacc + b1))                   (16 epilogue warps -> swizzled K-major smem operand)
//     Y   [128 tok, C  ] += Hs * W2[:, chunk]^T                     (tcgen05, accumulator in TMEM for the whole tile)
// and fc1 of chunks j+1 .. j+NB-1 is issued before fc2 of chunk j, so the GELU of chunk j runs under later MMAs.
// Both weight matrices stream through a ring of 8/16 KB slots (each CTA stages HALF of every weight tile; the pair's MMA
// reads both halves), so a weight byte is fetched from L2 once per 256 tokens.  TMEM: Y (C columns) + NB x 64 (Hacc).
//   warp 0       TMA producer (A tile, weight ring)
//   warp 1       leader: MMA issuer.  peer: relay -- it waits on the peer's LOCAL "epilogue done" barriers and forwards
//                ONE cluster-scope arrive to the leader (a release.cluster arrive from each of 16 epilogue warps costs a
//                cluster fence apiece: 30 % of all stall samples in the first version, profiles/r01_mlp_fused.txt)
//   warps 2..17  epilogue: GELU chunks, then the residual epilogue of the tile (residual in / result out by TMA)
template <int C>
struct MlpCfg {
    static constexpr int HC = 64;                     // hidden chunk: small, so that many chunks are in flight (the
                                                      // fc1 -> GELU -> fc2 chain of ONE chunk is ~3 k cycles long)
    static constexpr int NJ = 4 * C / HC;             // chunks per tile
    static constexpr int NB = (512 - C) / HC;         // hidden accumulators / smem operand buffers in flight: 6 / 4
    static constexpr int KB_A = C / 64;               // 64-wide k-blocks of the fc1 reduction
    static constexpr int A_BYTES = KB_A * 16384;      // this CTA's 128 tokens x C
    static constexpr int H_BYTES = 16384;             // one hidden chunk: 128 tokens x 64 (one k-block)
    static constexpr int W1_KB_BYTES = 32 * 128;      // this CTA's 32 of the chunk's 64 W1 rows, one k-block
    static constexpr int SLOT = KB_A * W1_KB_BYTES;   // = (C/2 rows) x 128 B of W2 as well: 8 KB / 16 KB
    static constexpr int W_SLOTS = C == 128 ? 7 : 5;  // one slot fewer than would fit: the epilogue's vectors live in shared memory
    static constexpr int VEC_BYTES = (4 * C + 4 * C + C + C) * 4;  // t_n / b1 [4C], s_n [4C], b2 [C], gamma [C] as fp32: with ~224 KB of
                                                      // shared memory taken, L1 is ~4 KB and every __ldg of them was an L2 round trip
                                                      // (long scoreboard: 34 % of the epilogue warps' stall samples)
    static constexpr int EPI_WARPS = 16;
    static constexpr int CH = C / 4 / 32;             // 32x32 output boxes per epilogue warp
    static constexpr bool STAGE_IN_H = C == 256;      // C=256: the output boxes are staged inside the (idle) hidden buffers
    static constexpr int STAGE_BYTES = STAGE_IN_H ? 0 : EPI_WARPS * CH * 2048;
    static constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;
    static constexpr int NUM_BARS = 2 * W_SLOTS + 2 + 6 * NB + 4 + EPI_WARPS;
    static constexpr int SMEM_BYTES = A_BYTES + NB * H_BYTES + STAGE_BYTES + W_SLOTS * SLOT + VEC_BYTES + NUM_BARS * 8 + 64 + 1024;
    static constexpr int TMEM_COLS = 512;
    static_assert(C == 128 || C == 256, "Y (C columns) + NB 64-column hidden accumulators must fit 512 TMEM columns");
    static_assert(C + NB * HC <= 512, "TMEM budget");
    static_assert(SLOT == (C / 2) * 128, "W1 and W2 chunk halves are the same size");
    static_assert(!STAGE_IN_H || NB * H_BYTES >= EPI_WARPS * CH * 2048, "staging must fit the hidden buffers");
    static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

// LNF: the block's LayerNorm folded into fc1 as in GEMM_LNGELU (a = the RAW depthwise output, W1 pre-multiplied by the LayerNorm
// weight): hidden = GELU(rstd_m * acc + (-mu_m rstd_m) * s_n + t_n) with (rstd_m, -mu_m rstd_m) = rowstat[m], s_n = `s1`, t_n = `b1`.
// A thread's token is the same for all 4C / 64 chunks of a tile, so the statistics cost one load per tile.
template <typename T, int C, bool LNF>
__global__ void __launch_bounds__(MlpCfg<C>::NUM_THREADS, 1)
mlp_fused_kernel(const __grid_constant__ CUtensorMap a_map, const __grid_constant__ CUtensorMap w1_map,
                 const __grid_constant__ CUtensorMap w2_map, const __grid_constant__ CUtensorMap x_map,
                 const float* __restrict__ b1, const float* __restrict__ b2, const float* __restrict__ gamma, int M,
                 const float* __restrict__ s1, const float2* __restrict__ rowstat, int stat_parts) {
    // stat_parts > 0: rowstat = dwconv_rawtc_kernel's per-chunk partial sums [M][stat_parts] (sum, sum of squares), finished here
    // (one or two 16-byte loads per thread and TILE; no ln_stat_finalize_kernel launch in front of this kernel)
    using Cfg = MlpCfg<C>;
    constexpr int NJ = Cfg::NJ, S = Cfg::W_SLOTS, NB = Cfg::NB, CH = Cfg::CH;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* sA = smem;
    uint8_t* sH = sA + Cfg::A_BYTES;                   // [NB][2 k-blocks][128 rows x 128 B]
    uint8_t* sStage = sH + NB * Cfg::H_BYTES;          // per-warp 32x32 output boxes (C=128); C=256 reuses sH
    uint8_t* sW = sStage + Cfg::STAGE_BYTES;
    float* sB1 = reinterpret_cast<float*>(sW + S * Cfg::SLOT);  // [4C] fc1 bias (t_n when LNF)
    float* sS1 = sB1 + 4 * C;                                   // [4C] s_n (LNF)
    float* sB2 = sS1 + 4 * C;                                   // [C]
    float* sGm = sB2 + C;                                       // [C]
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sB1) + Cfg::VEC_BYTES);
    uint64_t* wfull = bars;                 // [S]  leader's copy counts both CTAs' bytes
    uint64_t* wempty = wfull + S;           // [S]  multicast commit
    uint64_t* afull = wempty + S;           // leader
    uint64_t* aempty = afull + 1;           // multicast commit
    uint64_t* hacc_full = aempty + 1;       // [NB] multicast commit: fc1 of a chunk finished
    uint64_t* hacc_free_l = hacc_full + NB; // [NB] local: this CTA's 16 epilogue warps have read the accumulator
    uint64_t* hacc_free_p = hacc_free_l + NB;  // [NB] leader: the peer's relay says the same for the peer
    uint64_t* hs_full_l = hacc_free_p + NB; // [NB] local: this CTA's epilogue warps have written the smem operand
    uint64_t* hs_full_p = hs_full_l + NB;   // [NB] leader: relay
    uint64_t* hs_free = hs_full_p + NB;     // [NB] multicast commit: fc2 finished reading the smem operand
    uint64_t* yfull = hs_free + NB;         // multicast commit
    uint64_t* yfree_l = yfull + 1;          // local
    uint64_t* yfree_p = yfree_l + 1;        // leader: relay
    uint64_t* rfull = yfree_p + 2;          // [EPI_WARPS] residual boxes landed
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(rfull + Cfg::EPI_WARPS);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // provably warp-uniform
    const uint32_t rank = cluster_ctarank();
    const int num_tiles = (M + 255) / 256;
    const int tile0 = (int)blockIdx.x / 2, tile_step = (int)gridDim.x / 2;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&a_map);
        tma_prefetch_desc(&w1_map);
        tma_prefetch_desc(&w2_map);
        tma_prefetch_desc(&x_map);
        for (int s = 0; s < S; ++s) { mbar_init(&wfull[s], 1); mbar_init(&wempty[s], 1); }
        mbar_init(afull, 1);
        mbar_init(aempty, 1);
        for (int s = 0; s < NB; ++s) {
            mbar_init(&hacc_full[s], 1);
            mbar_init(&hacc_free_l[s], Cfg::EPI_WARPS);
            mbar_init(&hacc_free_p[s], 1);
            mbar_init(&hs_full_l[s], Cfg::EPI_WARPS);
            mbar_init(&hs_full_p[s], 1);
            mbar_init(&hs_free[s], 1);
        }
        mbar_init(yfull, 1);
        mbar_init(yfree_l, Cfg::EPI_WARPS);
        mbar_init(yfree_p, 1);
        for (int s = 0; s < Cfg::EPI_WARPS; ++s) mbar_init(&rfull[s], 1);
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc<2>(tmem_ptr, Cfg::TMEM_COLS);
    // the epilogue's vectors (weights: they do not depend on the previous kernel) into shared memory, once per CTA
    for (int i = threadIdx.x; i < 4 * C; i += Cfg::NUM_THREADS) {
        sB1[i] = __ldg(b1 + i);
        sS1[i] = LNF ? __ldg(s1 + i) : 0.f;
    }
    for (int i = threadIdx.x; i < C; i += Cfg::NUM_THREADS) {
        sB2[i] = __ldg(b2 + i);
        sGm[i] = __ldg(gamma + i);
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const uint32_t tm_y = tmem_base, tm_h = tmem_base + (uint32_t)C;
    pdl_launch_dependents();

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (both CTAs)
        if (lane == 0) {
            pdl_wait();
            int slot = 0;
            uint32_t wphase = 0, tcount = 0;
            auto next_slot = [&]() -> uint8_t* {
                mbar_wait(&wempty[slot], wphase ^ 1);
                if (rank == 0) mbar_expect_tx(&wfull[slot], 2 * Cfg::SLOT);
                return sW + slot * Cfg::SLOT;
            };
            auto advance = [&]() { if (++slot == S) { slot = 0; wphase ^= 1; } };
            auto load_w1 = [&](int j) {  // W1 rows of chunk j: this CTA stages 32 of the 64, every k-block
                uint8_t* dst = next_slot();
                const uint32_t lb = mapa_shared(smem_u32(&wfull[slot]), 0);
#pragma unroll
                for (int kb = 0; kb < Cfg::KB_A; ++kb)
                    tma_load_2d_pair(dst + kb * Cfg::W1_KB_BYTES, &w1_map, lb, kb * 64, j * 64 + (int)rank * 32);
                advance();
            };
            auto load_w2 = [&](int jj) {  // W2 columns of chunk jj: this CTA stages C/2 of the C output rows
                uint8_t* dst = next_slot();
                const uint32_t lb = mapa_shared(smem_u32(&wfull[slot]), 0);
                tma_load_2d_pair(dst, &w2_map, lb, jj * 64, (int)rank * (C / 2));
                advance();
            };
            for (int tile = tile0; tile < num_tiles; tile += tile_step, ++tcount) {
                const int row_a = (tile * 2 + (int)rank) * 128;
                mbar_wait(aempty, (tcount & 1) ^ 1);
                if (rank == 0) mbar_expect_tx(afull, 2 * Cfg::A_BYTES);
                const uint32_t la = mapa_shared(smem_u32(afull), 0);
#pragma unroll
                for (int kb = 0; kb < Cfg::KB_A; ++kb) tma_load_2d_pair(sA + kb * 16384, &a_map, la, kb * 64, row_a);
                // same order as the MMA issuer consumes: fc1 runs NB-1 chunks ahead of fc2
                for (int j = 0; j < NJ + NB - 1; ++j) {
                    if (j < NJ) load_w1(j);
                    if (j >= NB - 1) load_w2(j - (NB - 1));
                }
            }
        }
    } else if (warp == 1) {
        if (rank == 0) {
            // -------------------------------------------------------------- MMA issuer (pair leader): the whole warp runs the loop,
            // one elected lane issues (see gemm_kernel) -- these MMAs are 32 / 64 clk of tensor work each, so the ~130 clk of issue
            // latency per MMA of the `if (lane == 0)` form was three times the arithmetic
            const uint32_t lead = elect_one() ? 1u : 0u;
            constexpr uint32_t idesc1 = (1u << 4) | (UmmaFmt<T>::v << 7) | (UmmaFmt<T>::v << 10) | ((uint32_t)(Cfg::HC >> 3) << 17) |
                                        ((uint32_t)(256 >> 4) << 24);
            constexpr uint32_t idesc2 = (1u << 4) | (UmmaFmt<T>::v << 7) | (UmmaFmt<T>::v << 10) | ((uint32_t)(C >> 3) << 17) |
                                        ((uint32_t)(256 >> 4) << 24);
            int slot = 0;
            uint32_t wphase = 0, tcount = 0, j1 = 0, j2 = 0;  // j1 / j2: running chunk counters of fc1 / fc2
            auto wait_slot = [&]() -> uint32_t {
                mbar_wait(&wfull[slot], wphase);
                tc_fence_after();
                return smem_u32(sW + slot * Cfg::SLOT);
            };
            auto release_slot = [&]() {
                tc_commit_if<2>(lead, &wempty[slot]);
                if (++slot == S) { slot = 0; wphase ^= 1; }
            };
            for (int tile = tile0; tile < num_tiles; tile += tile_step, ++tcount) {
                mbar_wait(afull, tcount & 1);
                tc_fence_after();
                for (int j = 0; j < NJ + NB - 1; ++j) {
                    if (j < NJ) {
                        const uint32_t hb = j1 % NB, par = ((j1 / NB) & 1) ^ 1;
                        mbar_wait(&hacc_free_l[hb], par);
                        mbar_wait(&hacc_free_p[hb], par);
                        tc_fence_after();
                        const uint32_t d = tm_h + hb * Cfg::HC;
                        {
                            const uint32_t wb = wait_slot();
#pragma unroll
                            for (int kb = 0; kb < Cfg::KB_A; ++kb) {
                                const uint64_t adesc = make_sw128_kmajor_desc(smem_u32(sA + kb * 16384));
                                const uint64_t bdesc = make_sw128_kmajor_desc(wb + kb * Cfg::W1_KB_BYTES);
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    tc_mma_f16_if<2>(lead, d, adesc + 2 * k, bdesc + 2 * k, idesc1, (kb | k) != 0 ? 1u : 0u);
                            }
                            release_slot();
                        }
                        if (j == NJ - 1) tc_commit_if<2>(lead, aempty);  // the A tile has been read for the last time
                        tc_commit_if<2>(lead, &hacc_full[hb]);
                        ++j1;
                    }
                    if (j >= NB - 1) {
                        const int jj = j - (NB - 1);
                        const uint32_t hb = j2 % NB, par = (j2 / NB) & 1;
                        mbar_wait(&hs_full_l[hb], par);
                        mbar_wait(&hs_full_p[hb], par);
                        if (jj == 0) {  // the previous tile's Y has been read out
                            mbar_wait(yfree_l, (tcount & 1) ^ 1);
                            mbar_wait(yfree_p, (tcount & 1) ^ 1);
                        }
                        tc_fence_after();
                        const uint32_t hs = smem_u32(sH + hb * Cfg::H_BYTES);
                        {
                            const uint32_t wb = wait_slot();
                            const uint64_t adesc = make_sw128_kmajor_desc(hs);
                            const uint64_t bdesc = make_sw128_kmajor_desc(wb);
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                tc_mma_f16_if<2>(lead, tm_y, adesc + 2 * k, bdesc + 2 * k, idesc2, (jj > 0 || k > 0) ? 1u : 0u);
                            release_slot();
                        }
                        tc_commit_if<2>(lead, &hs_free[hb]);
                        ++j2;
                    }
                }
                tc_commit_if<2>(lead, yfull);
            }
        } else if (lane == 0 && rank == 1) {
            // -------------------------------------------------------------- relay (peer): local barriers -> one arrive at the leader
            uint32_t j1 = 0, tcount = 0;
            for (int tile = tile0; tile < num_tiles; tile += tile_step, ++tcount) {
                for (int j = 0; j < NJ; ++j, ++j1) {
                    const uint32_t hb = j1 % NB, par = (j1 / NB) & 1;
                    // relaxed forwards: the relay publishes nothing of its own, and what the peer's epilogue warps wrote
                    // (the smem operand) was fenced by them (fence.proxy.async = MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC) before
                    // their local arrive; a release.cluster here costs MEMBAR.ALL.GPU + ERRBAR on the MMA's critical path
                    mbar_wait(&hacc_free_l[hb], par);
                    mbar_arrive_cluster_relaxed(mapa_shared(smem_u32(&hacc_free_p[hb]), 0));
                    mbar_wait(&hs_full_l[hb], par);
                    mbar_arrive_cluster_relaxed(mapa_shared(smem_u32(&hs_full_p[hb]), 0));
                }
                mbar_wait(yfree_l, tcount & 1);
                mbar_arrive_cluster_relaxed(mapa_shared(smem_u32(yfree_p), 0));
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue warps (both CTAs)
        const int ew = warp - 2;
        const int q = warp & 3;          // TMEM lane quarter: tokens q*32 .. +31 of this CTA's 128
        const int slice = ew >> 2;       // 16 of the chunk's 64 hidden columns / C/4 of the output columns
        const int r = q * 32 + lane;     // token row inside the CTA tile
        const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
        uint32_t j1 = 0, tcount = 0, rph = 0;
        uint8_t* stage_p = (Cfg::STAGE_IN_H ? sH : sStage) + ew * CH * 2048;
        const uint32_t stage_a = smem_u32(stage_p);
        constexpr int CW = C / 4;
        pdl_wait();
        for (int tile = tile0; tile < num_tiles; tile += tile_step, ++tcount) {
            const int row0 = (tile * 2 + (int)rank) * 128 + q * 32;
            uint64_t ra2 = 0, rb2 = 0;
            if (LNF) {
                float2 rs = make_float2(0.f, 0.f);
                if (row0 + lane < M) {
                    if (stat_parts == 0) {
                        rs = __ldg(rowstat + row0 + lane);
                    } else {
                        const float2* rp = rowstat + (size_t)(row0 + lane) * (size_t)stat_parts;
                        float sm = 0.f, sq = 0.f;
                        for (int p = 0; p < stat_parts; ++p) { const float2 v = __ldg(rp + p); sm += v.x; sq += v.y; }  // C / 64 = 2 or 4 parts
                        const float mu = sm * (1.0f / (float)C);
                        const float var = fmaxf(fmaf(-mu, mu, sq * (1.0f / (float)C)), 0.0f);
                        const float rstd = 1.0f / sqrtf(var + LN_EPS_BACKBONE);
                        rs = make_float2(rstd, -mu * rstd);
                    }
                }
                ra2 = pk2(rs.x, rs.x);
                rb2 = pk2(rs.y, rs.y);
            }
            if (!Cfg::STAGE_IN_H && row0 < M && lane == 0) {
                // dedicated staging: the residual boxes of this tile arrive while its chunks are computed
                mbar_expect_tx(&rfull[ew], CH * 2048);
#pragma unroll
                for (int c = 0; c < CH; ++c) tma_load_2d(stage_p + c * 2048, &x_map, &rfull[ew], slice * CW + c * 32, row0);
            }
            // C = 256: the TMEM read of chunk j + 1 is issued BEFORE the GELU of chunk j (fc1 runs NB - 1 chunks ahead, so its
            // accumulator is normally complete) and its latency hides under arithmetic: 327 -> 310 us.  At C = 128 the same change
            // cost registers (spills) and time (463 -> 514 us): there each chunk is read when it is needed.
            constexpr bool PF = C == 256;
            float vbuf[2][16];
            if (PF) {
                const uint32_t hb = j1 % NB, u = (j1 / NB) & 1;
                mbar_wait(&hacc_full[hb], u);
                tc_fence_after();
                TmemLd<16>::ld(tm_h + lane_sel + hb * Cfg::HC + (uint32_t)(slice * 16), vbuf[0]);
            }
#pragma unroll PF ? NJ : 1
            for (int j = 0; j < NJ; ++j, ++j1) {
                const uint32_t hb = j1 % NB, u = (j1 / NB) & 1;
                const int hcol = j * Cfg::HC + slice * 16;
                float (&v)[16] = vbuf[PF ? (j & 1) : 0];
                if (!PF) {
                    mbar_wait(&hacc_full[hb], u);
                    tc_fence_after();
                    TmemLd<16>::ld(tm_h + lane_sel + hb * Cfg::HC + (uint32_t)(slice * 16), v);
                }
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_relaxed(&hacc_free_l[hb]);  // accumulator chunk is in registers
                if (PF && j + 1 < NJ) {
                    const uint32_t hn = (j1 + 1) % NB, un = ((j1 + 1) / NB) & 1;
                    mbar_wait(&hacc_full[hn], un);
                    tc_fence_after();
                    TmemLd<16>::ld(tm_h + lane_sel + hn * Cfg::HC + (uint32_t)(slice * 16), vbuf[(j + 1) & 1]);
                }
                float4 bias[4], sn[4];  // broadcast loads from shared memory
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    bias[i] = reinterpret_cast<const float4*>(sB1 + hcol)[i];
                    if (LNF) sn[i] = reinterpret_cast<const float4*>(sS1 + hcol)[i];
                }
                mbar_wait(&hs_free[hb], u ^ 1);  // fc2 of the chunk that used this operand buffer NB chunks ago is done
                const uint32_t dst = smem_u32(sH + hb * Cfg::H_BYTES) + (uint32_t)(r * 128);
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const float4 c0 = bias[2 * i], c1 = bias[2 * i + 1];
                    uint64_t v01, v23, v45, v67;
                    if (LNF) {
                        const float4 s0 = sn[2 * i], s1v = sn[2 * i + 1];
                        v01 = fma2(ra2, pk2(v[8 * i + 0], v[8 * i + 1]), fma2(rb2, pk2(s0.x, s0.y), pk2(c0.x, c0.y)));
                        v23 = fma2(ra2, pk2(v[8 * i + 2], v[8 * i + 3]), fma2(rb2, pk2(s0.z, s0.w), pk2(c0.z, c0.w)));
                        v45 = fma2(ra2, pk2(v[8 * i + 4], v[8 * i + 5]), fma2(rb2, pk2(s1v.x, s1v.y), pk2(c1.x, c1.y)));
                        v67 = fma2(ra2, pk2(v[8 * i + 6], v[8 * i + 7]), fma2(rb2, pk2(s1v.z, s1v.w), pk2(c1.z, c1.w)));
                    } else {
                        v01 = add2(pk2(v[8 * i + 0], v[8 * i + 1]), pk2(c0.x, c0.y));
                        v23 = add2(pk2(v[8 * i + 2], v[8 * i + 3]), pk2(c0.z, c0.w));
                        v45 = add2(pk2(v[8 * i + 4], v[8 * i + 5]), pk2(c1.x, c1.y));
                        v67 = add2(pk2(v[8 * i + 6], v[8 * i + 7]), pk2(c1.z, c1.w));
                    }
                    const uint32_t piece = (uint32_t)(slice * 2 + i);
                    sts128(dst + ((piece ^ ((uint32_t)r & 7u)) << 4),
                           make_uint4(gelu_pack2<T>(v01), gelu_pack2<T>(v23), gelu_pack2<T>(v45), gelu_pack2<T>(v67)));
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive_relaxed(&hs_full_l[hb]);  // every lane fenced its stores above
            }
            // ---- tile epilogue: x <- x + gamma * (Y + b2), residual in and result out through per-warp 32x32 boxes
            const uint32_t swz = ((uint32_t)lane >> 1) & 3u;
            mbar_wait(yfull, tcount & 1);  // all MMAs of the tile are done: Y is complete and the hidden buffers are idle
            tc_fence_after();
            if (Cfg::STAGE_IN_H && row0 < M && lane == 0) {
                mbar_expect_tx(&rfull[ew], CH * 2048);
#pragma unroll
                for (int c = 0; c < CH; ++c) tma_load_2d(stage_p + c * 2048, &x_map, &rfull[ew], slice * CW + c * 32, row0);
            }
            if (row0 < M) {
                mbar_wait(&rfull[ew], rph);
                rph ^= 1u;
            }
#pragma unroll
            for (int c = 0; c < CH; ++c) {
                const int col = slice * CW + c * 32;
                uint32_t v[32];
                tmem_ld_32x32(tm_y + lane_sel + (uint32_t)col, v);
                tmem_ld_wait();
                if (c == CH - 1) {  // Y has been read out: the next tile's fc2 may overwrite it
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_relaxed(yfree_l);
                }
                if (row0 < M) {
                    const uint32_t row_off = stage_a + (uint32_t)(c * 2048) + (uint32_t)lane * 64u;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint32_t addr = row_off + ((((uint32_t)i) ^ swz) << 4);
                        const float4 c0 = reinterpret_cast<const float4*>(sB2 + col)[2 * i];
                        const float4 c1 = reinterpret_cast<const float4*>(sB2 + col)[2 * i + 1];
                        const float4 g0 = reinterpret_cast<const float4*>(sGm + col)[2 * i];
                        const float4 g1 = reinterpret_cast<const float4*>(sGm + col)[2 * i + 1];
                        const uint4 rv = lds128(addr);
                        const float2 x01 = Cvt<T>::unpack2(rv.x), x23 = Cvt<T>::unpack2(rv.y);
                        const float2 x45 = Cvt<T>::unpack2(rv.z), x67 = Cvt<T>::unpack2(rv.w);
                        const uint64_t v01 = fma2(pk2(g0.x, g0.y), add2(pk2(__uint_as_float(v[8 * i + 0]), __uint_as_float(v[8 * i + 1])), pk2(c0.x, c0.y)), pk2(x01.x, x01.y));
                        const uint64_t v23 = fma2(pk2(g0.z, g0.w), add2(pk2(__uint_as_float(v[8 * i + 2]), __uint_as_float(v[8 * i + 3])), pk2(c0.z, c0.w)), pk2(x23.x, x23.y));
                        const uint64_t v45 = fma2(pk2(g1.x, g1.y), add2(pk2(__uint_as_float(v[8 * i + 4]), __uint_as_float(v[8 * i + 5])), pk2(c1.x, c1.y)), pk2(x45.x, x45.y));
                        const uint64_t v67 = fma2(pk2(g1.z, g1.w), add2(pk2(__uint_as_float(v[8 * i + 6]), __uint_as_float(v[8 * i + 7])), pk2(c1.z, c1.w)), pk2(x67.x, x67.y));
                        float f0, f1, f2, f3, f4, f5, f6, f7;
                        upk2(v01, f0, f1); upk2(v23, f2, f3); upk2(v45, f4, f5); upk2(v67, f6, f7);
                        sts128(addr, make_uint4(Cvt<T>::pack2(f0, f1), Cvt<T>::pack2(f2, f3), Cvt<T>::pack2(f4, f5), Cvt<T>::pack2(f6, f7)));
                    }
                }
            }
            if (row0 < M) {
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
#pragma unroll
                    for (int c = 0; c < CH; ++c) tma_store_2d(&x_map, stage_p + c * 2048, slice * CW + c * 32, row0);
                    bulk_commit();
                }
            }
            // the staging boxes are re-used (next tile's residual, or -- C=256 -- the hidden buffers themselves): every
            // warp's stores must have left shared memory first
            if (lane == 0) bulk_wait_read<0>();
            if (Cfg::STAGE_IN_H) asm volatile("bar.sync 1, %0;" ::"n"(Cfg::EPI_WARPS * 32) : "memory");
            else __syncwarp();
        }
        if (lane == 0) bulk_wait_all();
    }
    tc_fence_before();
    cluster_sync_all();
    if (warp == 1) tmem_dealloc<2>(tmem_base, Cfg::TMEM_COLS);
}

// ============================================================================ depthwise 7x7 (raw + statistics) on the tensor cores
// dwconv_raw_kernel's contract (raw 16-bit convolution = the fc1 A operand, (rstd, -mu rstd) per token) with the 49 taps on the
// tensor pipe.  One MMA per TAP (16 x 16 diagonal B matrices) is bound by the operand feed: each 128 x 16 activation slice is
// re-read from shared memory 49 times (measured and rejected, DESIGN.md).  Here a slice is read SEVEN times:
//   * the seven ROWS of the stencil (dy) are seven accumulating MMAs over row-shifted views of one swizzled tile (a row of 32
//     lanes is 4 KB, so every view starts on a 1024-byte swizzle atom; scripts/ubench/shiftmma.cu checks shifted views);
//   * the seven COLUMNS (dx) sit side by side in the N dimension: B_dy[k = c, n = (dx, c')] = w[dy][dx][c] (c == c'), 0 otherwise,
//     an M = 128, N = 7 x 16 = 112, K = 16 MMA per 16 channels, so TMEM lane p (a SOURCE pixel) ends up holding
//         D[p][dx][c] = sum_dy in[y(p) + dy - 3, x(p), c] * w[dy][dx][c]
//   * the epilogue adds the seven column blocks across lanes: out[y, x, c] = sum_dx D[(y, x + dx - 3)][dx][c], six warp shuffles
//     per value (a warp = 32 consecutive pixels of one image row, or 32 / W whole rows when W <= 32; `shfl` segments of W lanes
//     give the zero padding at the row ends for free) -- three packed half2 shuffles per value pair for fp16 (shfl_add_h2).
// Arithmetic: activations and taps are exact 16-bit operands, products are exact in fp32, accumulation is fp32 (tensor core over
// dy, FHFMA / FFMA over dx).  Differences from dwconv_raw_kernel: the taps are rounded to 16 bits, and (fp16) the six off-centre
// column partial sums cross lanes as fp16 (scripts/emulate_precision.py schemes tc_dw / tc_dw_h: 0.119 -> 0.143 / 0.137 px
// predicted for fp16 trained-like weights, 0.12 px measured; 0.5 px gate).
// Tiling.  A CTA owns ONE 64-channel chunk for the whole launch (its 7 B matrices, 98 KB, are loaded once) and walks "units" of
// 256 source lanes = two M tiles:
//   mode A (W in {8, 16, 32}):  a unit = 256 / W whole image rows; no x halo is needed (neighbours beyond the row are padding)
//   mode B (any other W):       a unit = 8 rows of one 32-lane window [xs, xs + 32), xs = -3 + 26 i; lanes 3..28 produce outputs
// plus 6 halo rows above / below (TMA zero fill outside the image).  TMEM: one 112-column accumulator per 16-channel group (4 x
// 128 columns); the MMA warp runs up to a whole M tile ahead of the four epilogue warpgroups.
//   warp 0        TMA producer          warp 1      MMA issuer (warp-uniform loop, one elected lane issues), TMEM allocator
//   warps 2..17   epilogue: warpgroup g = (warp - 2) / 4 drains group g (channels 16 g .. 16 g + 15 of the chunk)
// Statistics: the four warpgroups' (sum, sum of squares) of a pixel meet in shared memory; warpgroup 3 writes the chunk's partial
// to stat_part[token][k]; ln_stat_finalize_kernel (stages 2-3) or mlp_fused_kernel itself (stages 0-1) adds a token's parts --
// deterministic, no atomics.
struct DwTc2Cfg {
    static constexpr int CC = 64, NB = 112;
    static constexpr int B_BYTES = NB * 128;             // one dy: 112 rows (dx, c') x 64 k
    static constexpr int B_TOTAL = 7 * B_BYTES;          // 98 KB
    static constexpr int A_STAGE = (256 + 6 * 32) * 128; // 56 KB: two M tiles + 6 halo lane-rows (mode A with W < 32 uses less)
    static constexpr int A_STAGES = 2;
    static constexpr int STAT_BYTES = 2 * 3 * 128 * 8;   // [tile parity][warpgroup 0..2][pixel] (sum, sum of squares)
    static constexpr int EPI_WARPS = 16;
    static constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;
    static constexpr int SMEM_BYTES = B_TOTAL + A_STAGES * A_STAGE + STAT_BYTES + 256 + 1024;
    static constexpr int TMEM_COLS = 512;
    static_assert(B_BYTES % 1024 == 0 && A_STAGE % 1024 == 0, "swizzle atoms");
    static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

// acc += mask * (value of lane + DELTA of this lane's `width`-lane segment).  mask = 1 when that lane exists in the segment, else 0
// (the shuffle then returns this lane's own finite value); a mask multiply instead of the shuffle's predicate keeps the shuffles
// free of each other, so the 16 channels' shuffles are in flight together.
template <int DELTA>
__device__ __forceinline__ void shfl_add(float& acc, float v, float mask, int width) {
    if (DELTA == 0) acc += v;
    else if (DELTA > 0) acc = fmaf(__shfl_down_sync(0xffffffffu, v, DELTA, width), mask, acc);
    else acc = fmaf(__shfl_up_sync(0xffffffffu, v, -DELTA, width), mask, acc);
}

// Packed variant for fp16 models: the two channels of a pair cross lanes as ONE 32-bit half2 (half the shuffles -- the LSU / MIO
// path the shuffles share with the stores is what bounds the epilogue), and the mixed-precision FMA (FHFMA: fp16 x fp16 + fp32)
// applies the mask and widens in one instruction per value.  The partial sums that travel are rounded to fp16 (the centre column
// and the accumulation stay fp32): scripts/emulate_precision.py scheme tc_dw_h, 0.137 px against 0.143 px un-rounded.
template <int DELTA>
__device__ __forceinline__ void shfl_add_h2(float& a0, float& a1, float v0, float v1, uint32_t mask_h2, int width) {
    uint32_t h;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(v1), "f"(v0));
    const uint32_t t = DELTA > 0 ? __shfl_down_sync(0xffffffffu, h, DELTA, width) : __shfl_up_sync(0xffffffffu, h, -DELTA, width);
    asm("{\n\t.reg .f16 tl, th, ml, mh;\n\tmov.b32 {tl, th}, %2;\n\tmov.b32 {ml, mh}, %3;\n\t"
        "fma.rn.f32.f16 %0, tl, ml, %0;\n\tfma.rn.f32.f16 %1, th, mh, %1;\n\t}\n"
        : "+f"(a0), "+f"(a1)
        : "r"(t), "r"(mask_h2));
}
__device__ __forceinline__ void stg256(void* p, const uint32_t (&o)[8]) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]),
                 "r"(o[5]), "r"(o[6]), "r"(o[7])
                 : "memory");
}

// CG == 2 (cta_group::2, clusters of two CTAs): the pair works on the SAME channel chunk and on two units at a time (one per CTA);
// each CTA stages HALF of every B matrix (56 of its 112 rows) and the leader issues M = 256 MMAs for both, so the B operand feed per
// CTA and MMA halves (7.5 -> 5.75 KB).  Loads of both CTAs are counted on the leader's barriers, commits are multicast, the peer's
// epilogue warps hand their accumulators back with cluster-scope arrives -- the protocol of gemm_kernel<.., CG = 2>.
template <typename T, int CG>
__global__ void __launch_bounds__(DwTc2Cfg::NUM_THREADS, 1)
dwconv_rawtc_kernel(const __grid_constant__ CUtensorMap x_map, const __grid_constant__ CUtensorMap b_map,
                    const float* __restrict__ bdw, T* __restrict__ out, float2* __restrict__ stat_part, int C, int H, int W,
                    int rowpx /* lanes per image row inside a unit: W (mode A) or 32 (mode B) */,
                    int nwin /* windows per image row: 1 in mode A */, int units_y, int num_units, int b0) {
    using Cfg = DwTc2Cfg;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* sB = smem;
    uint8_t* sA = smem + Cfg::B_TOTAL;
    float2* sStat = reinterpret_cast<float2*>(sA + Cfg::A_STAGES * Cfg::A_STAGE);
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sStat) + Cfg::STAT_BYTES);
    uint64_t* bfull = bars;           // the chunk's B matrices landed
    uint64_t* afull = bars + 1;       // [2]
    uint64_t* aempty = afull + 2;     // [2]
    uint64_t* tfull = aempty + 2;     // [4] accumulator of a 16-channel group complete
    uint64_t* tempty = tfull + 4;     // [4] ... read out by the 4 warps of its warpgroup
    uint64_t* sfull = tempty + 4;     // [2] warpgroups 0..2 have written their statistics of an M tile
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(sfull + 2);

    // the warp index through a shuffle: provably warp-uniform, so the role branches below are uniform branches and the MMA warp's
    // address arithmetic can live in uniform registers
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int NCH = C / Cfg::CC;
    const uint32_t rank = CG == 2 ? cluster_ctarank() : 0u;
    const int unit_id = (int)blockIdx.x / CG;              // CTA (CG == 1) or CTA pair
    const int k = unit_id % NCH;                           // this CTA's (pair's) channel chunk
    const int u0 = unit_id / NCH, ustep = ((int)gridDim.x / CG) / NCH;  // it walks units (u0 + i * ustep) * CG + rank
    constexpr int B_CTA = Cfg::B_BYTES / CG;               // bytes of one B matrix staged by this CTA
    const bool mode_b = nwin > 1 || rowpx != W;
    const int rows_unit = mode_b ? 8 : 256 / W;            // output rows per unit
    const int units_img = nwin * units_y;
    const uint32_t a_bytes = (uint32_t)(256 + 6 * rowpx) * 128u;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&x_map);
        tma_prefetch_desc(&b_map);
        mbar_init(bfull, 1);
        for (int s = 0; s < 2; ++s) { mbar_init(&afull[s], 1); mbar_init(&aempty[s], 1); mbar_init(&sfull[s], 12); }
        for (int s = 0; s < 4; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 4 * CG); }
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc<CG>(tmem_ptr, Cfg::TMEM_COLS);
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr, 0);
    pdl_launch_dependents();

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            // the taps do not depend on the previous kernel: they are fetched while it is still running
            if (CG == 1) {
                mbar_expect_tx(bfull, Cfg::B_TOTAL);
                for (int dy = 0; dy < 7; ++dy) tma_load_2d(sB + dy * B_CTA, &b_map, bfull, 0, (k * 7 + dy) * Cfg::NB);
            } else {  // both CTAs' halves are counted on the leader's barrier
                if (rank == 0) mbar_expect_tx(bfull, Cfg::B_TOTAL);
                const uint32_t lb = mapa_shared(smem_u32(bfull), 0);
                for (int dy = 0; dy < 7; ++dy) tma_load_2d_pair(sB + dy * B_CTA, &b_map, lb, 0, (k * 7 + dy) * Cfg::NB + (int)rank * (Cfg::NB / 2));
            }
            pdl_wait();
            int it = 0;
            for (int up = u0; up * CG < num_units; up += ustep, ++it) {
                const int u = up * CG + (int)rank;  // CG == 2: may be one past the end (odd unit count): a box of zeros
                const int stage = it & 1;
                if (it >= 2) mbar_wait(&aempty[stage], ((it >> 1) - 1) & 1);
                const int b = u / units_img, r = u - b * units_img;
                const int wi = r % nwin, uy = r / nwin;
                const int xs = mode_b ? 26 * wi - 3 : 0;
                if (CG == 1) {
                    mbar_expect_tx(&afull[stage], a_bytes);
                    tma_load_4d(sA + stage * Cfg::A_STAGE, &x_map, &afull[stage], k * Cfg::CC, xs, uy * rows_unit - 3, b0 + b);
                } else {
                    if (rank == 0) mbar_expect_tx(&afull[stage], 2 * a_bytes);
                    tma_load_4d_pair(sA + stage * Cfg::A_STAGE, &x_map, mapa_shared(smem_u32(&afull[stage]), 0), k * Cfg::CC, xs, uy * rows_unit - 3,
                                     u < num_units ? b0 + b : 0x3fffffff);
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (the whole warp, one elected lane issues)
        if (rank == 0) {
            constexpr uint32_t idesc = (1u << 4) | (UmmaFmt<T>::v << 7) | (UmmaFmt<T>::v << 10) | ((uint32_t)(Cfg::NB >> 3) << 17) |
                                       ((uint32_t)((128 * CG) >> 4) << 24);
            const uint32_t lead = elect_one() ? 1u : 0u;
            mbar_wait(bfull, 0);
            // descriptors differ only in the 14-bit start-address field (bytes >> 4): + 2 per 16-channel group (32 B inside the
            // swizzle atom), + rowpx * 8 per stencil row, + 1024 per M tile, + B_BYTES / 16 per B matrix
            const uint64_t b0 = make_sw128_kmajor_desc(smem_u32(sB));
            const uint64_t a00 = make_sw128_kmajor_desc(smem_u32(sA));
            const uint64_t a_dy = (uint64_t)(rowpx * 8);
            int it = 0;
            uint32_t tcount = 0;  // M tiles issued so far: each uses every TMEM accumulator once
            for (int up = u0; up * CG < num_units; up += ustep, ++it) {
                const int stage = it & 1;
                mbar_wait(&afull[stage], (it >> 1) & 1);
                tc_fence_after();
                const uint64_t a0 = a00 + (uint64_t)(stage * (Cfg::A_STAGE >> 4));
#pragma unroll
                for (int mt = 0; mt < 2; ++mt, ++tcount) {
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        // one accumulator after the other: filling two or four in turn (so that an MMA need not wait for its
                        // predecessor on the same accumulator) was measured slower -- 305 / 316 / 373 us at C = 128 -- because
                        // the epilogue of group g then starts later
                        mbar_wait(&tempty[g], (tcount & 1) ^ 1);
                        tc_fence_after();
#pragma unroll
                        for (int dy = 0; dy < 7; ++dy) {
                            const uint64_t adesc = a0 + (uint64_t)(mt * 1024 + 2 * g) + (uint64_t)dy * a_dy;
                            const uint64_t bdesc = b0 + (uint64_t)(dy * (B_CTA >> 4) + 2 * g);
                            tc_mma_f16_if<CG>(lead, tmem_base + (uint32_t)(g * 128), adesc, bdesc, idesc, dy != 0 ? 1u : 0u);
                        }
                        tc_commit_if<CG>(lead, &tfull[g]);
                    }
                }
                tc_commit_if<CG>(lead, &aempty[stage]);
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue
        const int g = (warp - 2) >> 2;   // 16-channel group = TMEM accumulator
        const int q = warp & 3;          // TMEM lane quarter
        const int px = q * 32 + lane;    // pixel (TMEM lane) of the M tile
        const int width = mode_b ? 32 : W;
        constexpr bool PACKED = sizeof(T) == 2 && UmmaFmt<T>::v == 0;  // fp16: packed shuffles (see shfl_add_h2); bf16: fp32 shuffles
        float mk[7];  // mk[dx]: does source lane + dx - 3 lie in this lane's image row (mode A) / window (mode B: its outputs are unused if not)
        uint32_t mkh[7];
#pragma unroll
        for (int dx = 0; dx < 7; ++dx) {
            const int sl = (lane & (width - 1)) + dx - 3;
            mk[dx] = (sl >= 0 && sl < width) ? 1.0f : 0.0f;
            mkh[dx] = (sl >= 0 && sl < width) ? 0x3C003C00u : 0u;
        }
        const int ch0 = k * Cfg::CC + g * 16;
        float bias[16];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4 bb = __ldg(reinterpret_cast<const float4*>(bdw + ch0) + i);
            bias[4 * i] = bb.x; bias[4 * i + 1] = bb.y; bias[4 * i + 2] = bb.z; bias[4 * i + 3] = bb.w;
        }
        const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * 128);
        uint32_t tcount = 0;
        pdl_wait();
        // index arithmetic without integer divisions (they were ~13 % of this loop's instructions): exact multiply-high
        // reciprocals for the unit decode (u * divisor < 2^32), shifts for the power-of-two row width of mode A
        const uint32_t inv_units_img = (uint32_t)((0x100000000ull + (uint32_t)units_img - 1) / (uint32_t)units_img);
        const uint32_t inv_nwin = (uint32_t)((0x100000000ull + (uint32_t)nwin - 1) / (uint32_t)nwin);
        const int lw = 31 - __clz(W);  // mode A: W = 8, 16 or 32
        for (int up = u0; up * CG < num_units; up += ustep) {
            const int u = up * CG + (int)rank;
            const bool unit_ok = CG == 1 || u < num_units;
            const int b = units_img == 1 ? u : (int)__umulhi((uint32_t)u, inv_units_img), r = u - b * units_img;  // (the reciprocal of 1 does not fit 32 bits)
            const int uy = nwin == 1 ? r : (int)__umulhi((uint32_t)r, inv_nwin), wi = r - uy * nwin;
            const int y0 = uy * rows_unit;
            for (int mt = 0; mt < 2; ++mt, ++tcount) {
                int x, y;
                bool valid;
                if (mode_b) {
                    y = y0 + mt * 4 + q;
                    x = 26 * wi - 3 + lane;
                    valid = unit_ok && lane >= 3 && lane <= 28 && x < W && y < H;
                } else {
                    const int p = mt * 128 + px;
                    y = y0 + (p >> lw);
                    x = p & (W - 1);
                    valid = unit_ok && y < H;
                }
                const size_t tok = ((size_t)(b0 + b) * H + y) * W + x;
                mbar_wait(&tfull[g], tcount & 1);
                tc_fence_after();
                float acc[16];
#pragma unroll
                for (int c = 0; c < 16; ++c) acc[c] = bias[c];
                float v[2][16];
                TmemLd<16>::ld(tbase, v[0]);
#pragma unroll
                for (int dx = 0; dx < 7; ++dx) {
                    tmem_ld_wait();
                    if (dx < 6) {
                        TmemLd<16>::ld(tbase + (uint32_t)((dx + 1) * 16), v[(dx + 1) & 1]);
                    } else {
                        // the last column block is in registers: hand the accumulator back to the MMA warp before working on it
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            // the accumulator is in registers (tcgen05.wait::ld above): nothing to publish, relaxed arrives
                            if (CG == 1 || rank == 0) mbar_arrive_relaxed(&tempty[g]);
                            else mbar_arrive_cluster_relaxed(mapa_shared(smem_u32(&tempty[g]), 0));
                        }
                    }
                    if (PACKED && dx != 3) {
#pragma unroll
                        for (int c = 0; c < 16; c += 2) {
                            switch (dx) {
                                case 0: shfl_add_h2<-3>(acc[c], acc[c + 1], v[0][c], v[0][c + 1], mkh[0], width); break;
                                case 1: shfl_add_h2<-2>(acc[c], acc[c + 1], v[1][c], v[1][c + 1], mkh[1], width); break;
                                case 2: shfl_add_h2<-1>(acc[c], acc[c + 1], v[0][c], v[0][c + 1], mkh[2], width); break;
                                case 4: shfl_add_h2<1>(acc[c], acc[c + 1], v[0][c], v[0][c + 1], mkh[4], width); break;
                                case 5: shfl_add_h2<2>(acc[c], acc[c + 1], v[1][c], v[1][c + 1], mkh[5], width); break;
                                default: shfl_add_h2<3>(acc[c], acc[c + 1], v[0][c], v[0][c + 1], mkh[6], width); break;
                            }
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < 16; ++c) {
                            switch (dx) {
                                case 0: shfl_add<-3>(acc[c], v[0][c], mk[0], width); break;
                                case 1: shfl_add<-2>(acc[c], v[1][c], mk[1], width); break;
                                case 2: shfl_add<-1>(acc[c], v[0][c], mk[2], width); break;
                                case 3: shfl_add<0>(acc[c], v[1][c], mk[3], width); break;
                                case 4: shfl_add<1>(acc[c], v[0][c], mk[4], width); break;
                                case 5: shfl_add<2>(acc[c], v[1][c], mk[5], width); break;
                                default: shfl_add<3>(acc[c], v[0][c], mk[6], width); break;
                            }
                        }
                    }
                }
                float s = 0.f, sq = 0.f;
                uint32_t o[8];
#pragma unroll
                for (int c = 0; c < 16; c += 2) {
                    s += acc[c] + acc[c + 1];
                    sq = fmaf(acc[c], acc[c], sq);
                    sq = fmaf(acc[c + 1], acc[c + 1], sq);
                    o[c / 2] = Cvt<T>::pack2(acc[c], acc[c + 1]);
                }
                if (valid) {
                    stg256(out + tok * (size_t)C + ch0, o);  // one 32-byte store: half the LSU wavefronts of two 16-byte ones
                }
                // ---- token statistics
                float2* st = sStat + (tcount & 1) * (3 * 128);
                if (g < 3) {
                    st[g * 128 + px] = make_float2(s, sq);
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&sfull[tcount & 1]);
                } else {
                    mbar_wait(&sfull[tcount & 1], (tcount >> 1) & 1);
                    const float2 p0 = st[px], p1 = st[128 + px], p2 = st[256 + px];
                    if (valid) stat_part[tok * (size_t)NCH + k] = make_float2(((p0.x + p1.x) + p2.x) + s, ((p0.y + p1.y) + p2.y) + sq);
                }
            }
        }
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 1) tmem_dealloc<CG>(tmem_base, Cfg::TMEM_COLS);
}

// Token statistics of dwconv_rawtc_kernel: parts [tokens][NCH] (sum, sum of squares) -> rowstat[token] = (rstd, -mu rstd), parts
// added in index order.  A separate launch (2-3 us under PDL): finishing them inside fc1's epilogue cost that kernel 15 us at K = 512
// (its epilogue warps have no registers or issue slots to spare), finishing them inside the depthwise kernel needs a grid-wide
// hand-over (fence + atomic per tile on an epilogue warpgroup's path: 74 -> 129 us).
__global__ void __launch_bounds__(256) ln_stat_finalize_kernel(const float2* __restrict__ part, float2* __restrict__ rowstat, long long tokens,
                                                               int nch, float inv_c) {
    pdl_launch_dependents();
    pdl_wait();
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= tokens) return;
    const float2* p = part + t * nch;
    float sm = 0.f, sq = 0.f;
    if ((nch & 1) == 0) {
        const float4* p4 = reinterpret_cast<const float4*>(p);
        for (int i0 = 0; i0 < nch / 2; i0 += 4) {
            float4 v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = i0 + i < nch / 2 ? __ldg(p4 + i0 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 4; ++i) { sm += v[i].x; sq += v[i].y; sm += v[i].z; sq += v[i].w; }
        }
    } else {
        for (int i = 0; i < nch; ++i) { const float2 v = __ldg(p + i); sm += v.x; sq += v.y; }
    }
    const float mu = sm * inv_c;
    const float var = fmaxf(fmaf(-mu, mu, sq * inv_c), 0.0f);
    const float rstd = 1.0f / sqrtf(var + LN_EPS_BACKBONE);
    rowstat[t] = make_float2(rstd, -mu * rstd);
}

// ============================================================================ Global Response Normalization (ConvNeXt-V2)
// timm GlobalResponseNorm inside the block's MLP (fc1 -> GELU -> GRN -> fc2), channels-last:
//     g[b, c]  = || h[b, :, :, c] ||_2                       (over the image's tokens)
//     n[b, c]  = g[b, c] / (mean_c g[b, c] + 1e-6)
//     h'       = h + bias[c] + weight[c] * (h * n[b, c])  =  h * (1 + weight[c] * n[b, c]) + bias[c]
// Three launches around the hidden activation the fc1 GEMM wrote: partial sums of squares per (image, token chunk,
// channel) -- no atomics, so the result does not depend on scheduling --, one small CTA per image that finishes the norm
// and turns it into a per-(image, channel) scale, and an in-place scale + bias pass.  Two extra trips of the hidden
// activation through HBM per block: the un-fused first version of this operator.
constexpr int GRN_ROWS = 128;  // tokens per partial sum

// grid (ceil(C4 / 512), ceil(tokens / GRN_ROWS), B); thread = one channel pair
template <typename T>
__global__ void __launch_bounds__(256) grn_sumsq_kernel(const T* __restrict__ h, int tokens, int C4, float* __restrict__ part) {
    const int cp = blockIdx.x * 256 + threadIdx.x;
    if (2 * cp >= C4) return;
    const int chunk = blockIdx.y, b = blockIdx.z, nchunk = gridDim.y;
    const int r0 = chunk * GRN_ROWS, r1 = min(r0 + GRN_ROWS, tokens);
    const uint32_t* p = reinterpret_cast<const uint32_t*>(h + ((size_t)b * tokens + r0) * C4) + cp;
    float s0 = 0.f, s1 = 0.f;
#pragma unroll 8
    for (int r = r0; r < r1; ++r, p += C4 / 2) {
        const float2 v = Cvt<T>::unpack2(__ldg(p));
        s0 = fmaf(v.x, v.x, s0);
        s1 = fmaf(v.y, v.y, s1);
    }
    *reinterpret_cast<float2*>(part + ((size_t)b * nchunk + chunk) * C4 + 2 * cp) = make_float2(s0, s1);
}

// grid (B); scale[b][c] = 1 + weight[c] * g / (mean_c g + eps)
__global__ void __launch_bounds__(256) grn_finalize_kernel(const float* __restrict__ part, int nchunk, int C4,
                                                           const float* __restrict__ weight, float* __restrict__ scale) {
    extern __shared__ float s_g[];  // [C4]
    __shared__ float s_red[8];
    const int b = blockIdx.x, tid = threadIdx.x;
    float local = 0.f;
    for (int c = tid; c < C4; c += 256) {
        float a = 0.f;
        for (int k = 0; k < nchunk; ++k) a += part[((size_t)b * nchunk + k) * C4 + c];  // fixed order
        const float g = sqrtf(a);
        s_g[c] = g;
        local += g;
    }
    local = warp_sum(local);
    if ((tid & 31) == 0) s_red[tid >> 5] = local;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) tot += s_red[i];
    const float inv = 1.0f / (tot / (float)C4 + 1e-6f);
    for (int c = tid; c < C4; c += 256) scale[(size_t)b * C4 + c] = fmaf(weight[c], s_g[c] * inv, 1.0f);
}

// same grid as grn_sumsq_kernel; h <- h * scale[b][c] + bias[c], in place
template <typename T>
__global__ void __launch_bounds__(256) grn_apply_kernel(T* __restrict__ h, int tokens, int C4, const float* __restrict__ scale,
                                                        const float* __restrict__ bias) {
    const int cp = blockIdx.x * 256 + threadIdx.x;
    if (2 * cp >= C4) return;
    const int chunk = blockIdx.y, b = blockIdx.z;
    const int r0 = chunk * GRN_ROWS, r1 = min(r0 + GRN_ROWS, tokens);
    const float2 sc = *reinterpret_cast<const float2*>(scale + (size_t)b * C4 + 2 * cp);
    const float2 bi = *reinterpret_cast<const float2*>(bias + 2 * cp);
    uint32_t* p = reinterpret_cast<uint32_t*>(h + ((size_t)b * tokens + r0) * C4) + cp;
#pragma unroll 8
    for (int r = r0; r < r1; ++r, p += C4 / 2) {
        const float2 v = Cvt<T>::unpack2(*p);
        *p = Cvt<T>::pack2(fmaf(v.x, sc.x, bi.x), fmaf(v.y, sc.y, bi.y));
    }
}

// ============================================================================ LayerNorm2d + 2x2/s2 patchify
// x [B,H,W,C] -> a2 [B,H/2,W/2,4C] with k = (ky*2+kx)*C + c, the A operand of the downsample GEMM
// (timm stage.downsample = LayerNorm2d -> Conv2d(k=2,s=2)).
// 1408 channels (convnextv2_huge stage 2, V4 = 11) at PG = 2 need 160 registers, one CTA per SM: one token per iteration keeps two
template <int C> struct LnPatchifyPG { static constexpr int value = C <= 512 ? 4 : (C <= 1024 ? 2 : 1); };

template <typename T, int C>
__global__ void __launch_bounds__(256) ln_patchify_kernel(const T* __restrict__ x, const float* __restrict__ lnw,
                                                          const float* __restrict__ lnb, T* __restrict__ a2, int B, int H,
                                                          int W) {
    // One warp = PG x-adjacent tokens per iteration: PG independent load / reduction chains in flight, the index arithmetic
    // (three divisions) paid once per PG tokens, and the two LayerNorm reductions of all PG tokens in one recursive-halving
    // pass (warp_sum4).  A lane owns 4 consecutive channels of every 128-channel group.
    constexpr int V4 = (C + 127) / 128;  // a lane's 4-channel groups; the last one is part empty when C % 128 != 0 (192, 352, 704)
    constexpr int PG = LnPatchifyPG<C>::value;  // 4, 2 beyond 512 channels, 1 beyond 1024 (registers)
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int Ho = H >> 1, Wo = W >> 1;
    const int Wq = (W + PG - 1) / PG;
    const long long quads = (long long)B * H * Wq;
    for (long long qd = warp; qd < quads; qd += nwarps) {
        const long long row = qd / Wq;  // b * H + y
        const int x0 = (int)(qd - row * Wq) * PG;
        const long long b = row / H;
        const int y = (int)(row - b * H);
        if ((y >> 1) >= Ho) continue;  // odd H: the last row has no 2x2 patch
        bool ok[PG];
        float4 v[PG][V4];
        float s[4] = {0.f, 0.f, 0.f, 0.f}, q[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int p = 0; p < PG; ++p) {
            const int xx = x0 + p;
            ok[p] = xx < W && (xx >> 1) < Wo;
            const uint2* xp = reinterpret_cast<const uint2*>(x + ((size_t)row * W + (ok[p] ? xx : x0)) * C);
            float a = 0.f;
#pragma unroll
            for (int j = 0; j < V4; ++j) {
                const bool on = (C % 128 == 0) || (lane + 32 * j) * 4 < C;
                const uint2 u = on ? __ldg(xp + lane + 32 * j) : make_uint2(0u, 0u);
                const float2 lo = Cvt<T>::unpack2(u.x), hi = Cvt<T>::unpack2(u.y);
                v[p][j] = make_float4(lo.x, lo.y, hi.x, hi.y);
                a += (lo.x + lo.y) + (hi.x + hi.y);
            }
            s[p] = a;
        }
        warp_sum4(s, lane);
#pragma unroll
        for (int p = 0; p < PG; ++p) {
            const float mean = s[p] * (1.0f / C);
            float a = 0.f;
#pragma unroll
            for (int j = 0; j < V4; ++j) {
                const bool on = (C % 128 == 0) || (lane + 32 * j) * 4 < C;
                v[p][j].x -= mean; v[p][j].y -= mean; v[p][j].z -= mean; v[p][j].w -= mean;
                if (on) a += (v[p][j].x * v[p][j].x + v[p][j].y * v[p][j].y) + (v[p][j].z * v[p][j].z + v[p][j].w * v[p][j].w);
            }
            q[p] = a;
        }
        warp_sum4(q, lane);
#pragma unroll
        for (int p = 0; p < PG; ++p) {
            if (!ok[p]) continue;  // warp-uniform
            const int xx = x0 + p;
            const float rstd = 1.0f / sqrtf(q[p] * (1.0f / C) + LN_EPS_BACKBONE);
            const size_t orow = ((size_t)b * Ho + (y >> 1)) * Wo + (xx >> 1);
            uint2* op = reinterpret_cast<uint2*>(a2 + orow * (4 * C) + (size_t)(((y & 1) << 1) | (xx & 1)) * C);
#pragma unroll
            for (int j = 0; j < V4; ++j) {
                if (!((C % 128 == 0) || (lane + 32 * j) * 4 < C)) continue;
                const float4 g = __ldg(reinterpret_cast<const float4*>(lnw) + lane + 32 * j);  // L1-resident after the first token
                const float4 be = __ldg(reinterpret_cast<const float4*>(lnb) + lane + 32 * j);
                uint2 o;
                o.x = Cvt<T>::pack2(fmaf(v[p][j].x * rstd, g.x, be.x), fmaf(v[p][j].y * rstd, g.y, be.y));
                o.y = Cvt<T>::pack2(fmaf(v[p][j].z * rstd, g.z, be.z), fmaf(v[p][j].w * rstd, g.w, be.w));
                op[lane + 32 * j] = o;
            }
        }
    }
}

// ============================================================================ pool + head
// timm head (num_classes=0): global average pool -> LayerNorm2d(C) -> flatten; then
// generic.py:343-351: LayerNorm(C) -> Linear(C,HID) -> GELU -> Linear(HID,NOUT) -> Sigmoid.  fp32.
__device__ __forceinline__ float block_sum_256(float v, float* s_red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) s_red[wid] = v;
    __syncthreads();
    float r = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) r += s_red[i];
    return r;
}

// One image = one CLUSTER of HEAD_CLUSTER CTAs (a single CTA per image left 111 SMs idle and spent its time waiting on
// its own 512 KB of activations and 1 MB of Linear weights): every CTA pools 1/8 of the tokens, the partial sums meet
// through distributed shared memory (fixed order, so all ranks hold the same bits), every CTA runs the two cheap
// LayerNorms redundantly and computes 1/8 of the hidden layer into rank 0's shared memory; rank 0 finishes.
constexpr int HEAD_CLUSTER = 8;

template <typename T>
__global__ void __launch_bounds__(256) head_kernel(const T* __restrict__ x /*[B,tokens,C]*/, int tokens, int C,
                                                   const float* __restrict__ n0w, const float* __restrict__ n0b,
                                                   const float* __restrict__ n1w, const float* __restrict__ n1b,
                                                   const float* __restrict__ w1 /*[HID][C]*/, const float* __restrict__ b1,
                                                   int HID, const float* __restrict__ w2 /*[NOUT][HID]*/,
                                                   const float* __restrict__ b2, int NOUT, float* __restrict__ coords) {
    extern __shared__ __align__(16) float sm[];
    float* s_feat = sm;              // [C]
    float* s_hid = sm + C;           // [HID]   (rank 0's copy is the live one)
    float* s_red = s_hid + HID;      // [8]
    float* s_sum = s_red + 8;        // [C]     this CTA's share of the pool, read by every rank of the cluster
    float* s_part = s_sum + C;       // [8][C]  per-warp partial pools
    const uint32_t rank = cluster_ctarank();
    const int b = blockIdx.x / HEAD_CLUSTER, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const T* xb = x + (size_t)b * tokens * C;
    // global average pool: warp w of rank r sums tokens 8r + w, + 64, ...; a lane owns 8 consecutive channels per
    // 256-channel group (128-bit loads, every load independent)
    for (int c0 = 0; c0 < C; c0 += 256) {
        const int c = c0 + lane * 8;
        float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (c + 8 <= C) {
#pragma unroll 4
            for (int t = (int)rank * 8 + wid; t < tokens; t += 8 * HEAD_CLUSTER) {
                const uint4 u = __ldg(reinterpret_cast<const uint4*>(xb + (size_t)t * C + c));
                const float2 p0 = Cvt<T>::unpack2(u.x), p1 = Cvt<T>::unpack2(u.y), p2 = Cvt<T>::unpack2(u.z), p3 = Cvt<T>::unpack2(u.w);
                a[0] += p0.x; a[1] += p0.y; a[2] += p1.x; a[3] += p1.y;
                a[4] += p2.x; a[5] += p2.y; a[6] += p3.x; a[7] += p3.y;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) s_part[wid * C + c + j] = a[j];
        }
    }
    __syncthreads();
    for (int c = tid; c < C; c += 256) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) v += s_part[w * C + c];
        s_sum[c] = v;
    }
    cluster_sync_all();
    for (int c = tid; c < C; c += 256) {
        float v = 0.f;
#pragma unroll
        for (int r = 0; r < HEAD_CLUSTER; ++r) v += ld_cluster_f32(mapa_shared(smem_u32(s_sum + c), (uint32_t)r));
        s_feat[c] = v / (float)tokens;
    }
    __syncthreads();
    // two LayerNorms back to back (backbone.head.norm eps 1e-6, head.0 eps 1e-5)
    for (int pass = 0; pass < 2; ++pass) {
        const float* gw = pass == 0 ? n0w : n1w;
        const float* gb = pass == 0 ? n0b : n1b;
        const float eps = pass == 0 ? LN_EPS_BACKBONE : LN_EPS_HEAD;
        float s = 0.f;
        for (int c = tid; c < C; c += 256) s += s_feat[c];
        const float mean = block_sum_256(s, s_red) / (float)C;
        float q = 0.f;
        for (int c = tid; c < C; c += 256) { const float d = s_feat[c] - mean; q = fmaf(d, d, q); }
        const float rstd = 1.0f / sqrtf(block_sum_256(q, s_red) / (float)C + eps);
        for (int c = tid; c < C; c += 256) s_feat[c] = fmaf((s_feat[c] - mean) * rstd, gw[c], gb[c]);
        __syncthreads();
    }
    // Linear(C, HID) + exact GELU: this rank's slice of the outputs, one warp per output, lanes stride the row in float4;
    // the result goes straight into rank 0's hidden vector
    const int per = (HID + HEAD_CLUSTER - 1) / HEAD_CLUSTER;
    const int j_end = min(HID, ((int)rank + 1) * per);
    for (int j = (int)rank * per + wid; j < j_end; j += 8) {
        const float4* wr = reinterpret_cast<const float4*>(w1 + (size_t)j * C);
        const float4* fr = reinterpret_cast<const float4*>(s_feat);
        float s = 0.f;
#pragma unroll 4
        for (int c = lane; c < C / 4; c += 32) {
            const float4 w = __ldg(wr + c);
            const float4 f = fr[c];
            s = fmaf(w.x, f.x, s); s = fmaf(w.y, f.y, s); s = fmaf(w.z, f.z, s); s = fmaf(w.w, f.w, s);
        }
        s = warp_sum(s);
        if (lane == 0) st_cluster_f32(mapa_shared(smem_u32(s_hid + j), 0), gelu_exact(s + b1[j]));
    }
    cluster_sync_all();  // release / acquire: the remote stores are visible to rank 0; the other ranks are done
    if (rank != 0) return;
    for (int j = wid; j < NOUT; j += 8) {
        const float* wr = w2 + (size_t)j * HID;
        float s = 0.f;
        for (int c = lane; c < HID; c += 32) s = fmaf(__ldg(wr + c), s_hid[c], s);
        s = warp_sum(s);
        if (lane == 0) coords[(size_t)b * NOUT + j] = 1.0f / (1.0f + expf(-(s + b2[j])));
    }
}

}  // namespace svb
