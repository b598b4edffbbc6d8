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
// shared memory once.  Weights and sums are in double (guided_sweeps), with the
// reference's skip-if-zero guards made explicit.
//
// The guide has C = 1 (GRAY), 3 (BGR) or 4 (BGRX) bytes per pixel; a GRAY pixel g is staged as
// the word {g,0,0,0} and a BGRX pixel as {b,g,r,0}, so the colour distance is that of the BGR
// image (g,0,0) or (b,g,r), bit for bit.
//
// The guided kernel filters a stream of frames: the frame is blockIdx.z, which offsets every plane by its
// per-frame stride, so frame k of a launch equals a launch on frame k alone, bit for bit.  The depth is float32 or,
// in the U16 instantiations, uint16 millimetres (see guided_depth); a template parameter rather than a branch keeps
// the float32 kernels' code as it was.
//
// mrf_kernel follows MarkovRandomField/MarkovRandomField.cu:4-40 (next row f1).
#pragma once
#include <type_traits>
#include "common.cuh"

namespace kdme {

// The parameters of guided_fill_kernel<WS_CT, ...>, whose window is WS_CT wide, or 2 radius + 1 for WS_CT = 0.
template <int WS_CT>
struct GuidedParams {
    int width, height;
    const float* depth;
    const uint16_t* depth16;  // the depth as uint16 millimetres, read instead of `depth` by the U16 kernels
    const int32_t* labels;  // nullable
    const uint8_t* bgr;     // RAW guide, packed C-channel pixels (kernel template parameter C = 1, 3 or 4)
    long long bgr_step;
    float* out;
    float sigma_c;
    int radius;
    double kc, kd;   // 1/(2 sigma_c^2), 1/(2 sigma_d^2) in double; 0 where that sigma is 0 (factor skipped)
    // upsampling form (SURVEY.md 8(d) config 3, label-guided variant): when depth_lo or depth_lo16 is non-null the
    // depth plane is the sparse scatter of a wl x hl low-res map (see upsample_site) and `depth` is ignored
    const float* depth_lo;
    const uint16_t* depth_lo16;   // read instead of depth_lo by the U16 kernels
    int wl, hl;
    // per-frame strides (frame = blockIdx.z): depth samples (width*height, or wl*hl for the upsampling), guide bytes
    // (height*bgr_step), labels (width*height; 0 without labels), output floats (width*height)
    long long depth_stride, bgr_stride, labels_stride, out_stride;
    // The spatial factors: the reference's fp32 LUT S (EdgeRefinedSuperpixel.cpp:46-55), or 1 where S is 0 (the
    // skip-if-zero guard, :129-130, :185-186).  A compile-time window reads them as doubles from the constant bank;
    // the run-time window holds up to 31 x 31 of them as fp32 and stages them into shared doubles.
    std::conditional_t<(WS_CT > 0), double, float> sfac[WS_CT > 0 ? WS_CT * WS_CT : 31 * 31];
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

// The three sweeps of the pixel whose window starts at staged index `base`, in double (DESIGN.md section 2): the
// mean, the deviation and both weighted sums are those of the fp64 oracle (orc_guided_fill_f64), in its tap order.
// At a depth edge the output moves by about 2 kd Var(d) times the sweep-1 mean (over 100x for surfaces 1.5 m apart at
// sigma_d = 70), so fp32 weights or sums cannot keep such pixels within 1e-3 mm.  What stays fp32 is what the
// reference's formula holds in fp32 and the oracle keeps: the colour-sigma recurrence, 2 sigma^2 (its underflow to 0
// decides the -0/0 NaN) and `adaptive` from the fp32 mean.  A skipped factor (argument past the expf() zero cut, or
// its sigma 0) adds 0 to the exponent; sfac[t] is the spatial factor S, or 1 where the fp32 S is 0.
// WS_CT > 0 is a compile-time window (fully unrolled); 0 takes the window `ws` at run time.
template <int WS_CT>
__device__ __forceinline__ float guided_sweeps(const float* sD, const uint32_t* sG, const int32_t* sLab, int SP,
                                               int ws, int base, const double* sfac, float sigma_c, double kc,
                                               double kd) {
    const int WS = (WS_CT > 0) ? WS_CT : ws;
    const int pc = base + (WS / 2) * SP + WS / 2;
    const uint32_t gpix = sG[pc];
    const int32_t lp = sLab[pc];
    const double cut = kExpZeroArg;

    // ---- sweep 1: same-label weighted mean (:116-139), summed about the first such sample d0
    double acc = 0.0, wsum = 0.0, d0 = 0.0;
#pragma unroll (WS_CT > 0 ? WS_CT : 1)
    for (int i = 0; i < WS; ++i)
#pragma unroll (WS_CT > 0 ? WS_CT : 1)
        for (int j = 0; j < WS; ++j) {
            const int q = base + i * SP + j;
            const float d = sD[q];
            if (d == 0.f || sLab[q] != lp) continue;
            const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
            const double qc = (double)__dp4a(ad, ad, 0u) * kc;
            const double f = sfac[i * WS + j] * exp(-((qc <= cut) ? qc : 0.0));
            if (wsum == 0.0) d0 = d;
            acc = fma(f, (double)d - d0, acc);
            wsum += f;
        }
    if (!(wsum > 0.0)) return 0.f;
    const double m = d0 + acc / wsum;

    // ---- sweep 2: mean absolute deviation of the same taps (:143-156)
    double dev = 0.0;
    int count = 0;
#pragma unroll (WS_CT > 0 ? WS_CT : 1)
    for (int i = 0; i < WS; ++i)
#pragma unroll (WS_CT > 0 ? WS_CT : 1)
        for (int j = 0; j < WS; ++j) {
            const int q = base + i * SP + j;
            const float d = sD[q];
            if (d == 0.f || sLab[q] != lp) continue;
            dev += fabs((double)d - m);
            count++;
        }
    dev /= (double)count;
    // 5.0*deviation/pow(w_average,2.0f): double expression, fp32 square (:171)
    const float mf = (float)m;
    const float adaptive = (float)(5.0 * dev / (double)__fmul_rn(mf, mf));

    // ---- sweep 3: all samples, colour sigma MUTATED PER VALID TAP (:158-195)
    float sigma = sigma_c;
    double inv = 1.0 / (double)(2 * (sigma * sigma));   // 1 / (2 sigma^2), refreshed when sigma changes
    double num = 0.0, den = 0.0;
    bool poisoned = false;
#pragma unroll (WS_CT > 0 ? WS_CT : 1)
    for (int i = 0; i < WS; ++i)
#pragma unroll (WS_CT > 0 ? WS_CT : 1)
        for (int j = 0; j < WS; ++j) {
            const int q = base + i * SP + j;
            const float d = sD[q];
            if (d == 0.f) continue;
            double arg = 0.0;
            if (sigma != 0.0f) {
                const float t = sigma * 0.3f;
                const float sn = (adaptive > t) ? adaptive : t;
                if (sn != sigma) {
                    sigma = sn;
                    inv = 1.0 / (double)(2 * (sigma * sigma));   // 2 sigma^2 underflowed to 0: inv = +inf
                }
                const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
                const double qc = (double)__dp4a(ad, ad, 0u) * inv;
                if (qc != qc) poisoned = true;                  // 0 * inf: expf(-0/0) = NaN != 0 -> filter *= NaN
                else if (qc <= cut) arg = qc;
            }
            const double e = (double)d - m;
            const double z = e * e * kd;
            if (z <= cut) arg += z;
            const double f = sfac[i * WS + j] * exp(-arg);
            num = fma(f, (double)d, num);
            den += f;
        }
    if (poisoned) return __int_as_float(0x7fc00000);
    return (den == 0.0) ? 0.0f : (float)(num / den);
}

// One pixel per thread over a TW x TH tile whose tile + halo (depth, packed guide, labels) is staged in shared memory
// once.  A compile-time window (WS_CT > 0: windows 3..7) keeps the tile in static shared arrays and the fully
// unrolled sweeps read the spatial factors straight from the constant bank; the run-time window (WS_CT = 0) sizes
// the tile at launch (dynamic shared memory) and stages the factors into shared doubles.
template <int WS_CT, int TW, int TH, int C, bool U16>
__global__ void __launch_bounds__(TW * TH) guided_fill_kernel(const __grid_constant__ GuidedParams<WS_CT> p) {
    constexpr int NT = TW * TH;
    const int R = (WS_CT > 0) ? WS_CT / 2 : p.radius, WS = 2 * R + 1, SP = TW + 2 * R, SH = TH + 2 * R;
    const int tid = threadIdx.x;
    float* sD;
    uint32_t* sG;
    int32_t* sLab;
    const double* sfac;
    if constexpr (WS_CT > 0) {
        constexpr int N = (TW + WS_CT - 1) * (TH + WS_CT - 1);
        __shared__ float sDs[N];
        __shared__ uint32_t sGs[N];
        __shared__ int32_t sLabs[N];
        sD = sDs; sG = sGs; sLab = sLabs;
        sfac = p.sfac;
    } else {
        extern __shared__ __align__(16) uint8_t smem_gf[];
        __shared__ double sS[31 * 31];
        sD = reinterpret_cast<float*>(smem_gf);
        sG = reinterpret_cast<uint32_t*>(sD + SP * SH);
        sLab = reinterpret_cast<int32_t*>(sG + SP * SH);
        for (int idx = tid; idx < WS * WS; idx += NT) sS[idx] = p.sfac[idx];
        sfac = sS;
    }
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
    __syncthreads();

    const int lx = tid % TW, ly = tid / TW;
    const int gx = x0 + lx, gy = y0 + ly;
    if (gx >= p.width || gy >= p.height) return;
    p.out[frame * p.out_stride + (long long)gy * p.width + gx] =
        guided_sweeps<WS_CT>(sD, sG, sLab, SP, WS, ly * SP + lx, sfac, p.sigma_c, p.kc, p.kd);
}

// m * 2^a for a tap weight whose log2 is a, as a double.  Heavy taps (a >= -100) take ex2 of a itself, so their
// argument is rounded near 0 rather than near kWeightBias; lighter ones are lifted by 2^32 into ex2.approx.ftz's
// normal range and scaled back exactly in double, which keeps the weights the reference holds as fp32 subnormals.
__device__ __forceinline__ double ex2_weight(float a, float m = 1.0f) {
    const bool light = a < -100.f;
    return (double)(ex2_approx(light ? a + kWeightBias : a) * m) * (light ? 0x1p-32 /* 2^-kWeightBias */ : 1.0);
}

// MarkovRandomField.cu:4-40: out = (d_p + sum f d_q) / (1 + sum f), f = smooth * expf(-sigma_c * cd)
// over valid taps; f == 0 where fp32 expf() returns 0 (kExpZeroArg).  Sums in double: up to 961 taps of equal
// weight would otherwise round to more than 1e-3 mm.
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
    // sigma_c == 0 weights every tap 0 (the reference skips expf there): no argument passes a +inf cut
    const float cut = (color_sigma != 0.0f) ? -(float)(kExpZeroArg * kLog2e) : __int_as_float(0x7f800000);
    const double sm = smooth_sigma;
    double num = dp, den = 1.0;
    for (int i = 0; i < WS; ++i)
        for (int j = 0; j < WS; ++j) {
            const int q = (ly + i) * SP + lx + j;
            const float d = sD[q];
            const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
            const float a = (float)__dp4a(ad, ad, 0u) * nk;
            if (!(d > kValidDepth) || !(a >= cut)) continue;
            const double f = sm * ex2_weight(a);
            num = fma(f, (double)d, num);
            den += f;
        }
    out[(long long)gy * width + gx] = (den == 0.0) ? 0.0f : (float)(num / den);
}

// Projection_GPU::bilateralfilter -- Projection_GPU.cu:213-246 (next row f2): depth-only bilateral on the
// z of a packed float3 cloud, centred on the pixel's own z, weights expf(-dz^2/(2 sd^2)) * S; then
// x,y = normalized.x,y * z.  Race-free (reads `in`, writes `out`).  A tap is skipped where fp32 expf() returns 0,
// |dz| > e_cut = sqrt(2 kExpZeroArg) sd: without the cut a hole whose valid taps all lie just past it gets filled.
// A hole whose taps all lie near the cut is a weighted mean of weights ~2^-150 S: there the log2 depth term
// (~ -150) carries the rounding errors of both fp32 products and of the constant, recovered with FMAs, and
// the product with S is formed in double, down to 2^-299.  Sums in double, as in mrf_kernel; the window's z and S
// are staged in shared memory as doubles too, so a tap converts one value, not four.
template <int TW, int TH>
__global__ void __launch_bounds__(TW * TH)
depth_bilateral_xyz_kernel(const float* __restrict__ normalized, const float* __restrict__ in,
                           float* __restrict__ out, const float* __restrict__ stab /*S, [ws*ws]*/,
                           int width, int height, int R, float nkd /* -log2e/(2 sd^2) */,
                           float nkd_lo /* its rounding error */, float e_cut) {
    constexpr int NT = TW * TH;
    const int WS = 2 * R + 1, SP = TW + 2 * R, SH = TH + 2 * R;
    extern __shared__ __align__(16) uint8_t smem_dbx[];
    double* sZd = reinterpret_cast<double*>(smem_dbx);
    double* sS = sZd + SP * SH;
    float* sZ = reinterpret_cast<float*>(sS + WS * WS);
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    for (int idx = tid; idx < SP * SH; idx += NT) {
        int sy = idx / SP, sx = idx - sy * SP;
        int gx = x0 - R + sx, gy = y0 - R + sy;
        bool inb = (gx >= 0) & (gx < width) & (gy >= 0) & (gy < height);
        sZ[idx] = inb ? __ldg(in + 3 * ((long long)gy * width + gx) + 2) : 0.f;
        sZd[idx] = sZ[idx];
    }
    for (int idx = tid; idx < WS * WS; idx += NT) sS[idx] = __ldg(stab + idx);
    __syncthreads();
    const int lx = tid % TW, ly = tid / TW;
    const int gx = x0 + lx, gy = y0 + ly;
    if (gx >= width || gy >= height) return;
    const float zc = sZ[(ly + R) * SP + lx + R];
    double num = 0.0, den = 0.0;
    for (int i = 0; i < WS; ++i)
        for (int j = 0; j < WS; ++j) {
            const int q = (ly + i) * SP + lx + j;
            const float zq = sZ[q];
            const float e = zq - zc;
            if (!(zq > kValidDepth) || !(fabsf(e) <= e_cut)) continue;
            const float p = __fmul_rn(e, nkd), pe = fmaf(e, nkd, -p) + e * nkd_lo;
            const float dt = __fmul_rn(p, e), dte = fmaf(p, e, -dt) + pe * e;   // log2 depth factor = dt + dte
            const double f = ex2_weight(dt, fmaf(dte, (float)kLn2, 1.0f)) * sS[i * WS + j];
            num = fma(f, sZd[q], num);
            den += f;
        }
    const float z = (den == 0.0) ? 0.0f : (float)(num / den);
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
