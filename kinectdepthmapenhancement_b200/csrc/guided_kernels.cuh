// guided_kernels.cuh -- label-guided cross-bilateral fill (depthmap_enhancement) and
// the MRF filter, for sm_100a.
//
// guided_fill_kernel follows EdgeRefinedSuperpixel/EdgeRefinedSuperpixel.cu:104-205
// (reached from TOFDepthInterpolation.cpp:65 via EdgeRefining, :208-223) with
// race-free semantics: it reads `depth` and writes `out` (the reference overwrites
// its input while neighbouring threads still read it).  Three sweeps of the window:
//   1. same-label weighted mean (spatial x colour),
//   2. mean absolute deviation of the same taps,
//   3. all valid taps, colour sigma MUTATED PER VALID TAP (:170-176) and depth term
//      centred on the sweep-1 mean.
// The per-tap sigma recurrence is sequential in tap order, so one thread owns one
// pixel and walks the taps in the reference's order; the tile + halo is staged in
// shared memory once.  Weights are evaluated as one ex2 of summed log2-domain terms
// with the reference's skip-if-zero guards made explicit.
//
// The guide has C = 1 (GRAY), 3 (BGR) or 4 (BGRX) bytes per pixel; a GRAY pixel g is staged as
// the word {g,0,0,0} and a BGRX pixel as {b,g,r,0}, so the colour distance is that of the BGR
// image (g,0,0) or (b,g,r), bit for bit.
//
// Both guided kernels filter a stream of frames: the frame is blockIdx.z, which offsets every plane by its
// per-frame stride, so frame k of a launch equals a launch on frame k alone, bit for bit.  The depth is float32 or,
// in the U16 instantiations, uint16 millimetres (see guided_depth); a template parameter rather than a branch keeps
// the float32 kernels' code as it was.
//
// mrf_kernel follows MarkovRandomField/MarkovRandomField.cu:4-40 (next row f1).
#pragma once
#include "common.cuh"

namespace kdme {

struct GuidedParams {
    int width, height, radius;
    const float* depth;
    const uint16_t* depth16;  // the depth as uint16 millimetres, read instead of `depth` by the U16 kernels
    const int32_t* labels;  // nullable
    const uint8_t* bgr;     // RAW guide, packed C-channel pixels (kernel template parameter C = 1, 3 or 4)
    long long bgr_step;
    float* out;
    float sigma_c, sigma_d;
    // upsampling form (SURVEY.md 8(d) config 3, label-guided variant): when depth_lo or depth_lo16 is non-null the
    // depth plane is the sparse scatter of a wl x hl low-res map (see upsample_site) and `depth` is ignored
    const float* depth_lo;
    const uint16_t* depth_lo16;   // read instead of depth_lo by the U16 kernels
    int wl, hl;
    // per-frame strides (frame = blockIdx.z): depth samples (width*height, or wl*hl for the upsampling), guide bytes
    // (height*bgr_step), labels (width*height; 0 without labels), output floats (width*height)
    long long depth_stride, bgr_stride, labels_stride, out_stride;
    float spatial[31 * 31];  // the reference's fp32 LUT (EdgeRefinedSuperpixel.cpp:46-55)
};

// low-res sample index landing on high-res coordinate x, or -1: x_hi(xl) = floor((2 xl + 1) * W / (2 wl))
__device__ __forceinline__ int guided_upsample_site(int x, int W, int wl) {
    long long num = 2LL * wl * x - W;
    int xl = (num <= 0) ? 0 : (int)((num + 2LL * W - 1) / (2LL * W));
    if (xl >= wl) return -1;
    return ((int)(((2LL * xl + 1) * W) / (2LL * wl)) == x) ? xl : -1;
}

// Depth at image pixel (gx, gy) of `frame`: every depth read of both guided kernels goes through here.  The
// upsampling reads the low-res sample landing on the pixel (0 where none does).  A uint16 sample s reads as the
// float (float)s, exactly (s <= 50 is a hole, as for the float input).
template <bool U16, class P>
__device__ __forceinline__ float guided_depth(const P& p, long long frame, int gx, int gy) {
    if (p.depth_lo || p.depth_lo16) {
        const int xl = guided_upsample_site(gx, p.width, p.wl), yl = guided_upsample_site(gy, p.height, p.hl);
        if ((xl < 0) | (yl < 0)) return 0.f;
        const long long i = (long long)frame * p.depth_stride + (long long)yl * p.wl + xl;
        if constexpr (U16) return (float)__ldg(p.depth_lo16 + i); else return __ldg(p.depth_lo + i);
    }
    const long long i = (long long)frame * p.depth_stride + (long long)gy * p.width + gx;
    if constexpr (U16) return (float)__ldg(p.depth16 + i); else return __ldg(p.depth + i);
}

template <int TW, int TH, int C, bool U16>
__global__ void __launch_bounds__(TW * TH) guided_fill_kernel(const __grid_constant__ GuidedParams p) {
    constexpr int NT = TW * TH;
    const int R = p.radius, WS = 2 * R + 1, SP = TW + 2 * R, SH = TH + 2 * R;
    extern __shared__ __align__(16) uint8_t smem_gf[];
    float* sD = reinterpret_cast<float*>(smem_gf);
    uint32_t* sG = reinterpret_cast<uint32_t*>(sD + SP * SH);
    int32_t* sLab = reinterpret_cast<int32_t*>(sG + SP * SH);
    __shared__ float sL[31 * 31];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const long long frame = blockIdx.z;
    const uint8_t* bgr = p.bgr + frame * p.bgr_stride;
    const int32_t* labels = p.labels ? p.labels + frame * p.labels_stride : nullptr;
    for (int idx = tid; idx < SP * SH; idx += NT) {
        int sy = idx / SP, sx = idx - sy * SP;
        int gx = x0 - R + sx, gy = y0 - R + sy;
        bool in = (gx >= 0) & (gx < p.width) & (gy >= 0) & (gy < p.height);
        float d = 0.f;
        uint32_t g = 0u;
        int32_t l = 0;
        if (in) {
            d = guided_depth<U16>(p, frame, gx, gy);
            const uint8_t* q = bgr + (long long)gy * p.bgr_step + C * gx;
            if constexpr (C == 1) g = (uint32_t)__ldg(q);
            else g = (uint32_t)__ldg(q) | ((uint32_t)__ldg(q + 1) << 8) | ((uint32_t)__ldg(q + 2) << 16);
            if (labels) l = __ldg(labels + (long long)gy * p.width + gx);
        }
        sD[idx] = (d > kValidDepth) ? d : 0.f;  // 0 marks "not a sample" (also out of bounds)
        sG[idx] = g;
        sLab[idx] = l;
    }
    for (int idx = tid; idx < WS * WS; idx += NT) {
        const float s = p.spatial[idx];
        sL[idx] = (s != 0.0f) ? log2f(s) : 0.0f;  // skip-if-zero guard (:129-130, :185-186)
    }
    __syncthreads();

    const int lx = tid % TW, ly = tid / TW;
    const int gx = x0 + lx, gy = y0 + ly;
    if (gx >= p.width || gy >= p.height) return;
    const int pc = (ly + R) * SP + lx + R;
    const uint32_t gpix = sG[pc];
    const int32_t lp = sLab[pc];
    const float kZero = -(float)kExpZeroArg;
    const float l2e = (float)kLog2e;
    const float sc0 = p.sigma_c;
    const float den0 = 2 * (sc0 * sc0);
    const float inv_den0 = (sc0 != 0.0f) ? 1.0f / den0 : 0.f;   // sweep 1: one reciprocal per pixel, not a division per tap

    // accumulation origin: first sample in the window (keeps fp32 sums small)
    float d0 = 0.f;
    for (int t = 0; t < WS * WS && d0 == 0.f; ++t) {
        const int i = t / WS, j = t - i * WS;
        d0 = sD[(ly + i) * SP + lx + j];
    }

    // ---- sweep 1: same-label weighted mean (:116-139)
    float acc = 0.f, wsum = 0.f;
    for (int i = 0; i < WS; ++i)
        for (int j = 0; j < WS; ++j) {
            const int q = (ly + i) * SP + lx + j;
            const float d = sD[q];
            if (d == 0.f || sLab[q] != lp) continue;
            const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
            const float cd = (float)__dp4a(ad, ad, 0u);
            float lg = sL[i * WS + j] + kWeightBias;
            if (sc0 != 0.0f) {
                const float a = -cd * inv_den0;
                if (a >= kZero) lg = fmaf(a, l2e, lg);
            }
            const float f = ex2_approx(lg);
            acc = fmaf(f, d - d0, acc);
            wsum += f;
        }
    float o = 0.f;
    if (wsum > 0.f) {
        const float delta = acc / wsum;   // mean = d0 + delta
        const float mean = d0 + delta;    // the reference's fp32 w_average
        // ---- sweep 2: mean absolute deviation of the same taps (:143-156)
        float dev = 0.f;
        int count = 0;
        for (int i = 0; i < WS; ++i)
            for (int j = 0; j < WS; ++j) {
                const int q = (ly + i) * SP + lx + j;
                const float d = sD[q];
                if (d == 0.f || sLab[q] != lp) continue;
                dev += fabsf((d - d0) - delta);
                count++;
            }
        if (count != 0) dev /= (float)count;
        // 5.0*deviation/pow(w_average,2.0f): double expression, fp32 square (:171)
        const float adaptive = (float)(5.0 * (double)dev / (double)(mean * mean));
        // ---- sweep 3: all samples, mutating colour sigma (:158-195)
        const float sq = (p.sigma_d != 0.0f) ? sqrtf(l2e / (2.0f * p.sigma_d * p.sigma_d)) : 0.f;
        const float e_thr = (float)1.2247448713915890e1;  // sqrt(150)
        float sigma = sc0;
        float num = 0.f, den = 0.f;
        bool poisoned = false;
        for (int i = 0; i < WS; ++i)
            for (int j = 0; j < WS; ++j) {
                const int q = (ly + i) * SP + lx + j;
                const float d = sD[q];
                if (d == 0.f) continue;
                const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
                const float cd = (float)__dp4a(ad, ad, 0u);
                float lg = sL[i * WS + j] + kWeightBias;
                if (sigma != 0.0f) {
                    if (adaptive > sigma * 0.3f) sigma = adaptive; else sigma *= 0.3f;
                    const float dn = 2 * (sigma * sigma);
                    // fast reciprocal where it is safe; the exact quotient near underflow, where -0/0 = NaN
                    // (sigma^2 underflowed to 0 and cd == 0) and cd/denormal must behave as in IEEE arithmetic
                    const float a = (dn > 1.0e-30f) ? -cd * __frcp_rn(dn) : -cd / dn;
                    if (a != a) poisoned = true;       // expf(NaN) = NaN != 0 -> filter *= NaN
                    else if (a >= kZero) lg = fmaf(a, l2e, lg);
                }
                const float e = (d - d0) - delta;
                const float es = e * sq;
                if (p.sigma_d != 0.0f && !(fabsf(es) > e_thr)) lg = fmaf(-es, es, lg);
                const float f = ex2_approx(lg);
                num = fmaf(f, e, num);
                den += f;
            }
        if (poisoned) o = __int_as_float(0x7fc00000);
        else o = (den == 0.0f) ? 0.0f : mean + num / den;
    }
    p.out[frame * p.out_stride + (long long)gy * p.width + gx] = o;
}

// -----------------------------------------------------------------------------
// Fast form of the same three sweeps for the common case: compile-time radius (fully unrolled window, no
// index arithmetic), branch-free taps (validity / label tests become selects), the log2-domain spatial LUT
// read straight from the constant bank as an FFMA operand, the colour distance through the 2^23 magic
// accumulator (no int->float conversion), one MUFU.RCP instead of an IEEE division per sweep-3 tap, and
// the same-label predicate of sweep 1 kept as a bit mask for sweep 2.  Preconditions (host-checked): the
// colour skip-if-zero guard cannot fire in sweep 1 (sigma_c >= 30.63) and sigma_c, sigma_d != 0.  The
// per-valid-tap colour-sigma recurrence, its underflow to 0 and the -0/0 NaN poisoning are kept exactly.
template <int R>
struct GuidedFastParams {
    int width, height;
    const float* depth;
    const uint16_t* depth16;
    const int32_t* labels;  // nullable
    const uint8_t* bgr;
    long long bgr_step;
    float* out;
    float sigma_c, nk0 /* -log2e/(2 sigma_c^2) */, sq /* sqrt(log2e/(2 sigma_d^2)) */;
    const float* depth_lo;
    const uint16_t* depth_lo16;
    int wl, hl;
    long long depth_stride, bgr_stride, labels_stride, out_stride;   // as in GuidedParams
    float ltab[(2 * R + 1) * (2 * R + 1)];   // log2(S_ij) + kWeightBias, or kWeightBias where S_ij == 0
};

template <int R, int TW, int TH, int C, bool U16>
__global__ void __launch_bounds__(TW * TH) guided_fill_fast_kernel(const __grid_constant__ GuidedFastParams<R> p) {
    constexpr int NT = TW * TH, WS = 2 * R + 1, SP = TW + 2 * R, SH = TH + 2 * R;
    static_assert(WS * WS <= 64, "the same-label mask is one 64-bit word");
    __shared__ float sD[SP * SH];
    __shared__ uint32_t sG[SP * SH];
    __shared__ int32_t sLab[SP * SH];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const long long frame = blockIdx.z;
    const uint8_t* bgr = p.bgr + frame * p.bgr_stride;
    const int32_t* labels = p.labels ? p.labels + frame * p.labels_stride : nullptr;
    for (int idx = tid; idx < SP * SH; idx += NT) {
        int sy = idx / SP, sx = idx - sy * SP;
        int gx = x0 - R + sx, gy = y0 - R + sy;
        bool in = (gx >= 0) & (gx < p.width) & (gy >= 0) & (gy < p.height);
        float d = 0.f;
        uint32_t g = 0u;
        int32_t l = 0;
        if (in) {
            d = guided_depth<U16>(p, frame, gx, gy);
            const uint8_t* q = bgr + (long long)gy * p.bgr_step + C * gx;
            if constexpr (C == 1) g = (uint32_t)__ldg(q);
            else g = (uint32_t)__ldg(q) | ((uint32_t)__ldg(q + 1) << 8) | ((uint32_t)__ldg(q + 2) << 16);
            if (labels) l = __ldg(labels + (long long)gy * p.width + gx);
        }
        sD[idx] = (d > kValidDepth) ? d : 0.f;
        sG[idx] = g;
        sLab[idx] = l;
    }
    __syncthreads();
    const int lx = tid % TW, ly = tid / TW;
    const int gx = x0 + lx, gy = y0 + ly;
    if (gx >= p.width || gy >= p.height) return;
    const int base = ly * SP + lx;
    const uint32_t gpix = sG[base + R * SP + R];
    const int32_t lp = sLab[base + R * SP + R];
    // accumulation origin: the centre sample, else the first sample of the window (rare, divergent)
    float d0 = sD[base + R * SP + R];
    if (d0 == 0.f) {
        for (int t = 0; t < WS * WS && d0 == 0.f; ++t) d0 = sD[base + (t / WS) * SP + (t % WS)];
    }
    const float nk0 = p.nk0;

    // ---- sweep 1: same-label weighted mean (:116-139)
    float acc = 0.f, wsum = 0.f;
    unsigned long long same = 0ull;
#pragma unroll
    for (int i = 0; i < WS; ++i)
#pragma unroll
        for (int j = 0; j < WS; ++j) {
            const int q = base + i * SP + j;
            const float d = sD[q];
            const bool pr = (d != 0.f) & (sLab[q] == lp);
            const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
            const float cdf = __uint_as_float(__dp4a(ad, ad, kMagicValid)) - 8388608.0f;
            const float f = ex2_approx(fmaf(cdf, nk0, p.ltab[i * WS + j]));
            if (pr) {   // predicated accumulation (no selects)
                acc = fmaf(f, d - d0, acc);
                wsum += f;
                same |= 1ull << (i * WS + j);
            }
        }
    float o = 0.f;
    if (wsum > 0.f) {
        const float delta = acc / wsum;   // mean = d0 + delta
        const float mean = d0 + delta;    // the reference's fp32 w_average
        // ---- sweep 2: mean absolute deviation of the same taps (:143-156)
        float dev = 0.f;
#pragma unroll
        for (int i = 0; i < WS; ++i)
#pragma unroll
            for (int j = 0; j < WS; ++j) {
                const float x = fabsf((sD[base + i * SP + j] - d0) - delta);
                if ((same >> (i * WS + j)) & 1ull) dev += x;
            }
        const int count = __popcll(same);
        if (count != 0) dev /= (float)count;
        // 5.0*deviation/pow(w_average,2.0f): double expression, fp32 square (:171)
        const float adaptive = (float)(5.0 * (double)dev / (double)(mean * mean));
        // ---- sweep 3: all samples, mutating colour sigma (:158-195)
        const float kZero = -(float)kExpZeroArg;
        const float l2e = (float)kLog2e;
        const float sq = p.sq;
        const float e_thr = (float)1.2247448713915890e1;  // sqrt(150)
        float sigma = p.sigma_c;
        float num = 0.f, den = 0.f;
#pragma unroll
        for (int i = 0; i < WS; ++i)
#pragma unroll
            for (int j = 0; j < WS; ++j) {
                const int q = base + i * SP + j;
                const float d = sD[q];
                const bool v = d != 0.f;
                const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
                const float cd = __uint_as_float(__dp4a(ad, ad, kMagicValid)) - 8388608.0f;
                float lg = p.ltab[i * WS + j];
                // the recurrence advances once per VALID tap while sigma != 0 (:170-176); branch-free
                const bool adv = v & (sigma != 0.0f);
                const float t = sigma * 0.3f;
                const float sn = (adaptive > t) ? adaptive : t;
                sigma = adv ? sn : sigma;
                // a = -cd / (2 sigma^2) evaluated as (-cd * rcp(sigma^2)) with the factor 1/2 folded into the constants
                // (a power of two: same bits)
                const float s2 = sigma * sigma;
                float rc;
                asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(s2));
                const float a2 = -cd * rc;                      // 2a
                // 2 sigma^2 <= 1e-30: cd >= 1 is beyond the fp32 expf() cut-off (factor skipped) and cd == 0 gives -0
                // (factor 1) -- either way nothing is added; the one exception, -0/0 = NaN, is handled after the sweep
                if (adv & (s2 > 0.5e-30f) & (a2 >= 2.0f * kZero)) lg = fmaf(a2, 0.5f * l2e, lg);
                const float e = (d - d0) - delta;
                const float es = e * sq;
                if (!(fabsf(es) > e_thr)) lg = fmaf(-es, es, lg);
                const float f = ex2_approx(lg);
                if (v) {
                    num = fmaf(f, e, num);
                    den += f;
                }
            }
        // NaN poisoning (:170-176 with sigma^2 underflowed to exactly 0 and cd == 0: expf(-0/0) = NaN).  sigma never
        // increases once the sweep has started, so it can only have happened if the FINAL sigma squares to 0: rare,
        // re-walked here with the recurrence alone
        bool poisoned = false;
        if (sigma != 0.0f ? (2 * (sigma * sigma) == 0.0f) : true) {
            float sg = p.sigma_c;
            for (int t2 = 0; t2 < WS * WS; ++t2) {
                const int q = base + (t2 / WS) * SP + (t2 % WS);
                if (sD[q] == 0.f || sg == 0.0f) continue;
                const float tt = sg * 0.3f;
                sg = (adaptive > tt) ? adaptive : tt;
                if (2 * (sg * sg) == 0.0f) {
                    const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
                    if (__dp4a(ad, ad, 0u) == 0u) poisoned = true;
                }
            }
        }
        if (poisoned) o = __int_as_float(0x7fc00000);
        else o = (den == 0.0f) ? 0.0f : mean + num / den;
    }
    p.out[frame * p.out_stride + (long long)gy * p.width + gx] = o;
}

// MarkovRandomField.cu:4-40: out = (d_p + sum f d_q) / (1 + sum f), f = smooth * expf(-sigma_c * cd)
// over valid taps; evaluated as d_p + sum f (d_q - d_p) / (1 + sum f).
template <int TW, int TH>
__global__ void __launch_bounds__(TW * TH)
mrf_kernel(const float* __restrict__ depth, const uint32_t* __restrict__ guide4, int guide_pitch,
           float* __restrict__ out, int width, int height, int R, float color_sigma, float smooth_sigma) {
    constexpr int NT = TW * TH;
    const int WS = 2 * R + 1, SP = TW + 2 * R, SH = TH + 2 * R;
    extern __shared__ __align__(16) uint8_t smem_mrf[];
    float* sD = reinterpret_cast<float*>(smem_mrf);
    uint32_t* sG = reinterpret_cast<uint32_t*>(sD + SP * SH);
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    for (int idx = tid; idx < SP * SH; idx += NT) {
        int sy = idx / SP, sx = idx - sy * SP;
        int gx = x0 - R + sx, gy = y0 - R + sy;
        bool in = (gx >= 0) & (gx < width) & (gy >= 0) & (gy < height);
        sD[idx] = in ? __ldg(depth + (long long)gy * width + gx) : 0.f;
        sG[idx] = in ? __ldg(guide4 + (long long)gy * guide_pitch + gx) : 0u;
    }
    __syncthreads();
    const int lx = tid % TW, ly = tid / TW;
    const int gx = x0 + lx, gy = y0 + ly;
    if (gx >= width || gy >= height) return;
    const int pc = (ly + R) * SP + lx + R;
    const uint32_t gpix = sG[pc];
    const float dp = sD[pc];
    const float nk = -color_sigma * (float)kLog2e;
    float num = 0.f, den = 1.0f;
    for (int i = 0; i < WS; ++i)
        for (int j = 0; j < WS; ++j) {
            const int q = (ly + i) * SP + lx + j;
            const float d = sD[q];
            if (!(d > kValidDepth)) continue;
            const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
            const float cd = (float)__dp4a(ad, ad, 0u);
            const float f = (color_sigma != 0.0f) ? smooth_sigma * ex2_approx(cd * nk) : 0.f;
            num = fmaf(f, d - dp, num);
            den += f;
        }
    out[(long long)gy * width + gx] = (den == 0.0f) ? 0.0f : dp + num / den;
}

// Projection_GPU::bilateralfilter -- Projection_GPU.cu:213-246 (next row f2): depth-only bilateral on the
// z of a packed float3 cloud, centred on the pixel's own z, weights expf(-dz^2/(2 sd^2)) * S; then
// x,y = normalized.x,y * z.  Race-free (reads `in`, writes `out`).
template <int TW, int TH>
__global__ void __launch_bounds__(TW * TH)
depth_bilateral_xyz_kernel(const float* __restrict__ normalized, const float* __restrict__ in,
                           float* __restrict__ out, const float* __restrict__ ltab /*log2 S, [ws*ws]*/,
                           int width, int height, int R, float nkd /* -log2e/(2 sd^2) */) {
    constexpr int NT = TW * TH;
    const int WS = 2 * R + 1, SP = TW + 2 * R, SH = TH + 2 * R;
    extern __shared__ __align__(16) uint8_t smem_dbx[];
    float* sZ = reinterpret_cast<float*>(smem_dbx);
    float* sL = sZ + SP * SH;
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    for (int idx = tid; idx < SP * SH; idx += NT) {
        int sy = idx / SP, sx = idx - sy * SP;
        int gx = x0 - R + sx, gy = y0 - R + sy;
        bool inb = (gx >= 0) & (gx < width) & (gy >= 0) & (gy < height);
        sZ[idx] = inb ? __ldg(in + 3 * ((long long)gy * width + gx) + 2) : 0.f;
    }
    for (int idx = tid; idx < WS * WS; idx += NT) sL[idx] = __ldg(ltab + idx);
    __syncthreads();
    const int lx = tid % TW, ly = tid / TW;
    const int gx = x0 + lx, gy = y0 + ly;
    if (gx >= width || gy >= height) return;
    const float zc = sZ[(ly + R) * SP + lx + R];
    float num = 0.f, den = 0.f;
    for (int i = 0; i < WS; ++i) {
        float rn = 0.f, rd = 0.f;
        for (int j = 0; j < WS; ++j) {
            const float zq = sZ[(ly + i) * SP + lx + j];
            if (!(zq > kValidDepth)) continue;
            const float e = zq - zc;
            const float f = ex2_approx(fmaf(e * nkd, e, sL[i * WS + j] + kWeightBias));
            rn = fmaf(f, e, rn);
            rd += f;
        }
        num += rn;
        den += rd;
    }
    const float z = (den == 0.0f) ? 0.0f : zc + num / den;
    const long long k = (long long)gy * width + gx;
    out[3 * k + 0] = __ldg(normalized + 3 * k + 0) * z;
    out[3 * k + 1] = __ldg(normalized + 3 * k + 1) * z;
    out[3 * k + 2] = z;
}

// main.cpp:217-308 (next row f4): sum of Euclidean distances between two packed float3 clouds over pixels
// whose z are both in (50, 15000), and their count.  acc[0] += sum (double), acc[1] += count (as double).
__global__ void __launch_bounds__(256) mean_3d_error_kernel(const float* __restrict__ pts,
                                                            const float* __restrict__ truth, long long n,
                                                            double* __restrict__ acc) {
    double s = 0.0, c = 0.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        const float z = pts[3 * k + 2], zt = truth[3 * k + 2];
        if (z > 50.0f && z < 15000.0f && zt > 50.0f && zt < 15000.0f) {
            const float dz = z - zt, dy = pts[3 * k + 1] - truth[3 * k + 1], dx = pts[3 * k] - truth[3 * k];
            s += (double)sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dz, dz), __fmul_rn(dy, dy)), __fmul_rn(dx, dx)));
            c += 1.0;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    __shared__ double ss[8], sc[8];
    if ((threadIdx.x & 31) == 0) { ss[threadIdx.x >> 5] = s; sc[threadIdx.x >> 5] = c; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) { s += ss[w]; c += sc[w]; }
        atomicAdd(acc, s);
        atomicAdd(acc + 1, c);
    }
}

}  // namespace kdme
