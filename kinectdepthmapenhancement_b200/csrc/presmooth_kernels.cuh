// presmooth_kernels.cuh -- colour bilateral pre-smooth of the guide image.
//
// Stands in for the third-party call cv::gpu::bilateralFilter(color, smooth, 5,
// 30.0f, 30.0f) at JointBilateralFilter/JointBilateralFilter.cu:285 (OpenCV 2.4.3
// gpu module, not vendored in the reference): circular window dx^2+dy^2 <= r^2,
// weight = exp(-space2/(2 ss^2)) * exp(-L1(dBGR)^2/(2 sc^2)), reflect-101 border,
// round-to-nearest-even saturation to u8.
//
// Both exponentials come from LUTs built on the host (space: ksize^2 entries,
// colour: 766 entries indexed by the integer L1 distance), multiplied in fp32 and
// accumulated with one FFMA per channel in tap order (dy outer, dx inner), so the
// result is bit-identical to the CPU restatement of the same definition given the
// same LUTs.
//
// Input: packed u8 rows of C channels per pixel (template parameter C): C = 3 packed BGR
// (cv::gpu::GpuMat CV_8UC3), C = 4 BGRX/BGRA (the 4th byte is never read into a weight),
// C = 1 GRAY/IR.  Output: the internal u8x4 {B,G,R,0} guide (16-byte alignable rows, one
// 32-bit word per pixel) that the JBF kernel stages with TMA; a GRAY pixel g becomes the word
// {g,0,0,0}, so every output equals the BGR path's on the image (g,0,0) bit for bit, and the
// L1 colour distance reduces to |dg| (OpenCV's 1-channel definition).
#pragma once
#include "common.cuh"

namespace kdme {

constexpr int kPsMaxK = 9;  // largest supported pre-smooth kernel size

struct PresmoothParams {
    int width, height, n_frames;
    const uint8_t* bgr;          // [n][H][bgr_step]
    long long bgr_step;          // bytes per row
    long long bgr_frame_stride;  // bytes
    uint32_t* guide4;            // [n][H][guide_pitch]
    int guide_pitch;             // words
    long long guide_frame_stride;  // words
    int ksize;
    const float* space_lut;  // [ksize*ksize], < 0 outside the circle
    const float* color_lut;  // [766]
    // peer-memory halos (see JbfParams): rows outside [band0, band1) come from the neighbour GPU's band
    const uint8_t* bgr_up;   // row r < band0  -> bgr_up + r * bgr_step
    const uint8_t* bgr_dn;   // row r >= band1 -> bgr_dn + (r - band1) * bgr_step
    int band0, band1;
};

__device__ __forceinline__ const uint8_t* presmooth_row(const PresmoothParams& p, const uint8_t* src, int gy) {
    if (p.bgr_up != nullptr && gy < p.band0) return p.bgr_up + (long long)gy * p.bgr_step;
    if (p.bgr_dn != nullptr && gy >= p.band1) return p.bgr_dn + (long long)(gy - p.band1) * p.bgr_step;
    return src + (long long)gy * p.bgr_step;
}

__device__ __forceinline__ int reflect101(int p, int len) {
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = (p < 0) ? -p : 2 * (len - 1) - p;
    return p;
}

template <int TW, int TH, int C>
__global__ void __launch_bounds__(TW * TH) presmooth_kernel(const PresmoothParams p) {
    grid_launch_dependents();   // PDL: the filter's prologue (LUTs, descriptors, barrier) may start now
    constexpr int NT = TW * TH;
    constexpr int RMAX = kPsMaxK / 2;
    constexpr int SPM = TW + 2 * RMAX, SHM = TH + 2 * RMAX;
    __shared__ uint32_t sPix[SPM * SHM];
    __shared__ float sCol[768];
    __shared__ float sSp[kPsMaxK * kPsMaxK];
    const int r = p.ksize / 2;
    const int SP = TW + 2 * r, SH = TH + 2 * r;
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH, frame = blockIdx.z;
    const uint8_t* src = p.bgr + (long long)frame * p.bgr_frame_stride;

    for (int idx = tid; idx < SP * SH; idx += NT) {
        int sy = idx / SP, sx = idx - sy * SP;
        int gx = reflect101(x0 - r + sx, p.width), gy = reflect101(y0 - r + sy, p.height);
        const uint8_t* q = presmooth_row(p, src, gy) + C * gx;
        if constexpr (C == 1) sPix[idx] = (uint32_t)__ldg(q);
        else sPix[idx] = (uint32_t)__ldg(q) | ((uint32_t)__ldg(q + 1) << 8) | ((uint32_t)__ldg(q + 2) << 16);
    }
    for (int idx = tid; idx < 766; idx += NT) sCol[idx] = __ldg(p.color_lut + idx);
    for (int idx = tid; idx < p.ksize * p.ksize; idx += NT) sSp[idx] = __ldg(p.space_lut + idx);
    __syncthreads();

    const int lx = tid % TW, ly = tid / TW;
    const int gx = x0 + lx, gy = y0 + ly;
    if (gx >= p.width || gy >= p.height) return;
    const uint32_t c = sPix[(ly + r) * SP + lx + r];
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, ws = 0.f;
    for (int dy = 0; dy < p.ksize; ++dy) {
        for (int dx = 0; dx < p.ksize; ++dx) {
            const float sw = sSp[dy * p.ksize + dx];
            if (sw < 0.f) continue;
            const uint32_t q = sPix[(ly + dy) * SP + lx + dx];
            const uint32_t ad = __vabsdiffu4(q, c);
            const uint32_t l1 = __dp4a(ad, 0x01010101u, 0u);
            const float w = __fmul_rn(sw, sCol[l1]);
            s0 = __fmaf_rn(w, (float)(q & 0xffu), s0);
            if constexpr (C != 1) {   // GRAY: channels 1 and 2 are 0 and stay 0
                s1 = __fmaf_rn(w, (float)((q >> 8) & 0xffu), s1);
                s2 = __fmaf_rn(w, (float)((q >> 16) & 0xffu), s2);
            }
            ws = __fadd_rn(ws, w);
        }
    }
    const float v0 = fminf(fmaxf(rintf(__fdiv_rn(s0, ws)), 0.f), 255.f);
    const float v1 = fminf(fmaxf(rintf(__fdiv_rn(s1, ws)), 0.f), 255.f);
    const float v2 = fminf(fmaxf(rintf(__fdiv_rn(s2, ws)), 0.f), 255.f);
    const uint32_t o = (uint32_t)v0 | ((uint32_t)v1 << 8) | ((uint32_t)v2 << 16);
    p.guide4[(long long)frame * p.guide_frame_stride + (long long)gy * p.guide_pitch + gx] = o;
}

// One output pixel: {rint(s0 / ws), rint(s1 / ws), rint(s2 / ws)} clamped to bytes and packed, bit-identical to
// fminf(fmaxf(rintf(__fdiv_rn(s, ws)), 0), 255) per channel for 0 <= s <= 255 ws, ws >= 1 (the centre tap has weight
// 1), without the three IEEE divisions: q = s * rcp(ws) lies within 6e-5 of the correctly rounded quotient (two
// roundings of 2^-23 relative at magnitude <= 255), so the two can only round to different integers when q is that
// close to a half-integer -- then, and only then, the exact divisions are evaluated (cold, out of line).  The
// rounding itself is the 1.5 * 2^23 trick (round-to-nearest-even; the byte appears in the low mantissa bits).
__device__ __noinline__ uint32_t presmooth_pack_exact(float s0, float s1, float s2, float ws) {
    const float v0 = fminf(fmaxf(rintf(__fdiv_rn(s0, ws)), 0.f), 255.f);
    const float v1 = fminf(fmaxf(rintf(__fdiv_rn(s1, ws)), 0.f), 255.f);
    const float v2 = fminf(fmaxf(rintf(__fdiv_rn(s2, ws)), 0.f), 255.f);
    return (uint32_t)v0 | ((uint32_t)v1 << 8) | ((uint32_t)v2 << 16);
}
__device__ __forceinline__ uint32_t presmooth_pack(float s0, float s1, float s2, float ws) {
    const float kMagic = 12582912.0f, kTie = 2.5e-4f;
    const float inv = rcp_approx(ws);
    const float q0 = __fmul_rn(s0, inv), q1 = __fmul_rn(s1, inv), q2 = __fmul_rn(s2, inv);
    const float m0 = __fadd_rn(q0, kMagic), m1 = __fadd_rn(q1, kMagic), m2 = __fadd_rn(q2, kMagic);
    const float d0 = fabsf(__fsub_rn(q0, __fsub_rn(m0, kMagic))), d1 = fabsf(__fsub_rn(q1, __fsub_rn(m1, kMagic))),
                d2 = fabsf(__fsub_rn(q2, __fsub_rn(m2, kMagic)));
    // d in [0, 0.5]: the largest of the three decides
    if (fmaxf(fmaxf(d0, d1), d2) > 0.5f - kTie) return presmooth_pack_exact(s0, s1, s2, ws);
    const uint32_t b0 = min(__float_as_uint(m0) & 0x1ffu, 255u), b1 = min(__float_as_uint(m1) & 0x1ffu, 255u),
                   b2 = min(__float_as_uint(m2) & 0x1ffu, 255u);
    return b0 | (b1 << 8) | (b2 << 16);
}
// GRAY: presmooth_pack(s0, 0, 0, ws) (the zero channels give d = 0 and byte 0), one channel of work.
__device__ __noinline__ uint32_t presmooth_pack1_exact(float s0, float ws) {
    return (uint32_t)fminf(fmaxf(rintf(__fdiv_rn(s0, ws)), 0.f), 255.f);
}
__device__ __forceinline__ uint32_t presmooth_pack1(float s0, float ws) {
    const float kMagic = 12582912.0f, kTie = 2.5e-4f;
    const float q0 = __fmul_rn(s0, rcp_approx(ws));
    const float m0 = __fadd_rn(q0, kMagic);
    if (fabsf(__fsub_rn(q0, __fsub_rn(m0, kMagic))) > 0.5f - kTie) return presmooth_pack1_exact(s0, ws);
    return min(__float_as_uint(m0) & 0x1ffu, 255u);
}

// ksize == 5 (the reference's call): 13 taps fully unrolled, 4 pixels per thread along x.  Each
// staged pixel is converted ONCE to float b, g, r and a packed u8x4 word, kept as four shared-memory
// planes so a thread fetches its 8-column row segment with conflict-free 16-byte LDS; a tap is then
// VABSDIFF4 + IDP.4A (L1 norm) + LDS (colour LUT) + FMUL + 3 FFMA + FADD.
// C = 4 stages 4 pixels with one 16-byte load (byte 3 masked off); C = 1 stages 4 pixels with one 32-bit load and
// keeps only the b plane and the word plane: one FFMA per tap instead of three.
template <int TW, int TH, int PY, int C>
__global__ void __launch_bounds__((TW / 4) * (TH / PY)) presmooth5_kernel(const PresmoothParams p) {
    grid_launch_dependents();   // PDL: the filter's prologue (LUTs, descriptors, barrier) may start now
    static_assert(TH % PY == 0 && (PY == 1 || PY == 2), "a thread owns PY rows");
    static_assert(C == 1 || C == 3 || C == 4, "GRAY, BGR or BGRX");
    constexpr int NT = (TW / 4) * (TH / PY), R = 2, SP = TW + 8, SH = TH + 2 * R;   // 4 halo columns each side (16-byte rows)
    constexpr int XO = 4 - R;                                               // first used column of a staged row
    constexpr int SPH_GR = (C == 1) ? 4 : SP * SH;                          // the g and r planes (unused for GRAY)
    __shared__ __align__(16) float sB[SP * SH];
    __shared__ __align__(16) float sG[SPH_GR];
    __shared__ __align__(16) float sR[SPH_GR];
    __shared__ __align__(16) uint32_t sP[SP * SH];
    __shared__ float sCol[768];
    __shared__ float sSp[25];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH, frame = blockIdx.z;
    const uint8_t* src = p.bgr + (long long)frame * p.bgr_frame_stride;
    constexpr int SW = TW + 2 * R;   // staged (used) columns per row
    // reflect-101 only matters for tiles that touch the image border (CTA-uniform)
    const bool interior = (x0 >= R) && (y0 >= R) && (x0 + TW + R <= p.width) && (y0 + TH + R <= p.height);
    // Tiles whose 72 staged columns [x0 - 4, x0 + TW + 4) lie inside the row, on 4-byte aligned rows (CTA-uniform):
    // a thread stages 4 pixels = 12 bytes = three 32-bit loads, splits them with shifts and stores each plane with one
    // 16-byte STS -- 3 loads and 4 stores per 4 pixels instead of 12 and 16.  Rows reflect (101) as in the general path.
    // BGRX: one 16-byte load per 4 pixels, so 16-byte aligned rows; GRAY: one 32-bit load per 4 pixels.
    constexpr uintptr_t kWideAlign = (C == 4) ? 15 : 3;
    const bool wide = (x0 >= 4) && (x0 + TW + 4 <= p.width) &&
                      (((reinterpret_cast<uintptr_t>(p.bgr) | reinterpret_cast<uintptr_t>(p.bgr_up) |
                         reinterpret_cast<uintptr_t>(p.bgr_dn) | (uintptr_t)p.bgr_step | (uintptr_t)p.bgr_frame_stride) & kWideAlign) == 0);
    if (wide && C == 1) {
        constexpr int NG = SP / 4, GIT = (NG * SH + NT - 1) / NT;
        uint32_t w0[GIT];
#pragma unroll
        for (int it = 0; it < GIT; ++it) {
            const int g = tid + it * NT;
            w0[it] = 0u;
            if (g < NG * SH) {
                const int sy = g / NG, gc = g - sy * NG;
                int gy = y0 - R + sy;
                if (!interior) gy = reflect101(gy, p.height);
                w0[it] = __ldg(reinterpret_cast<const uint32_t*>(presmooth_row(p, src, gy) + (x0 - 4 + 4 * gc)));
            }
        }
#pragma unroll
        for (int it = 0; it < GIT; ++it) {
            const int g = tid + it * NT;
            if (g < NG * SH) {
                const int sy = g / NG, gc = g - sy * NG;
                const int o = sy * SP + 4 * gc;
                const uint32_t a = w0[it];
                *reinterpret_cast<float4*>(sB + o) = make_float4((float)(a & 0xffu), (float)((a >> 8) & 0xffu), (float)((a >> 16) & 0xffu), (float)(a >> 24));
                *reinterpret_cast<uint4*>(sP + o) = make_uint4(a & 0xffu, (a >> 8) & 0xffu, (a >> 16) & 0xffu, a >> 24);
            }
        }
    } else if (wide && C == 4) {
        constexpr int NG = SP / 4, GIT = (NG * SH + NT - 1) / NT;
        uint4 w[GIT];
#pragma unroll
        for (int it = 0; it < GIT; ++it) {
            const int g = tid + it * NT;
            w[it] = make_uint4(0u, 0u, 0u, 0u);
            if (g < NG * SH) {
                const int sy = g / NG, gc = g - sy * NG;
                int gy = y0 - R + sy;
                if (!interior) gy = reflect101(gy, p.height);
                w[it] = __ldg(reinterpret_cast<const uint4*>(presmooth_row(p, src, gy) + 4 * (x0 - 4 + 4 * gc)));
            }
        }
#pragma unroll
        for (int it = 0; it < GIT; ++it) {
            const int g = tid + it * NT;
            if (g < NG * SH) {
                const int sy = g / NG, gc = g - sy * NG;
                const int o = sy * SP + 4 * gc;
                const uint4 v = w[it];   // one pixel per word: b g r x
                *reinterpret_cast<float4*>(sB + o) = make_float4((float)(v.x & 0xffu), (float)(v.y & 0xffu), (float)(v.z & 0xffu), (float)(v.w & 0xffu));
                *reinterpret_cast<float4*>(sG + o) = make_float4((float)((v.x >> 8) & 0xffu), (float)((v.y >> 8) & 0xffu), (float)((v.z >> 8) & 0xffu), (float)((v.w >> 8) & 0xffu));
                *reinterpret_cast<float4*>(sR + o) = make_float4((float)((v.x >> 16) & 0xffu), (float)((v.y >> 16) & 0xffu), (float)((v.z >> 16) & 0xffu), (float)((v.w >> 16) & 0xffu));
                *reinterpret_cast<uint4*>(sP + o) = make_uint4(v.x & 0xffffffu, v.y & 0xffffffu, v.z & 0xffffffu, v.w & 0xffffffu);
            }
        }
    } else if (wide) {
        constexpr int NG = SP / 4, GIT = (NG * SH + NT - 1) / NT;
        uint32_t w0[GIT], w1[GIT], w2[GIT];
#pragma unroll
        for (int it = 0; it < GIT; ++it) {
            const int g = tid + it * NT;
            w0[it] = w1[it] = w2[it] = 0u;
            if (g < NG * SH) {
                const int sy = g / NG, gc = g - sy * NG;
                int gy = y0 - R + sy;
                if (!interior) gy = reflect101(gy, p.height);
                const uint32_t* q = reinterpret_cast<const uint32_t*>(presmooth_row(p, src, gy) + 3 * (x0 - 4 + 4 * gc));
                w0[it] = __ldg(q); w1[it] = __ldg(q + 1); w2[it] = __ldg(q + 2);
            }
        }
#pragma unroll
        for (int it = 0; it < GIT; ++it) {
            const int g = tid + it * NT;
            if (g < NG * SH) {
                const int sy = g / NG, gc = g - sy * NG;
                const int o = sy * SP + 4 * gc;
                // little endian: w0 = b0 g0 r0 b1 | w1 = g1 r1 b2 g2 | w2 = r2 b3 g3 r3
                const uint32_t a = w0[it], b = w1[it], c = w2[it];
                *reinterpret_cast<float4*>(sB + o) = make_float4((float)(a & 0xffu), (float)(a >> 24), (float)((b >> 16) & 0xffu), (float)((c >> 8) & 0xffu));
                *reinterpret_cast<float4*>(sG + o) = make_float4((float)((a >> 8) & 0xffu), (float)(b & 0xffu), (float)(b >> 24), (float)((c >> 16) & 0xffu));
                *reinterpret_cast<float4*>(sR + o) = make_float4((float)((a >> 16) & 0xffu), (float)((b >> 8) & 0xffu), (float)(c & 0xffu), (float)(c >> 24));
                *reinterpret_cast<uint4*>(sP + o) = make_uint4(a & 0xffffffu, (a >> 24) | ((b & 0xffffu) << 8), (b >> 16) | ((c & 0xffu) << 16), c >> 8);
            }
        }
    } else
    {   // warp w stages rows w, w + NWARP, ...; lane l columns l, l + 32, l + 64: no index division, the row pointer is
        // warp-uniform, and all byte loads of the thread are issued before the first use (memory-level parallelism)
        constexpr int NWARP = NT / 32, RIT = (SH + NWARP - 1) / NWARP, CIT = (SW + 31) / 32;
        const int warp = tid >> 5, lane = tid & 31;
        uint32_t vb[RIT][CIT], vg[RIT][CIT], vr[RIT][CIT];
#pragma unroll
        for (int rr = 0; rr < RIT; ++rr) {
            const int sy = warp + rr * NWARP;
            int gy = y0 - R + sy;
            if (!interior) gy = reflect101(gy, p.height);
            const uint8_t* rowp = presmooth_row(p, src, (sy < SH) ? gy : 0);
#pragma unroll
            for (int k = 0; k < CIT; ++k) {
                const int sx = lane + 32 * k;
                vb[rr][k] = vg[rr][k] = vr[rr][k] = 0u;
                if (sy < SH && sx < SW) {
                    int gx = x0 - R + sx;
                    if (!interior) gx = reflect101(gx, p.width);
                    const uint8_t* q = rowp + C * gx;
                    vb[rr][k] = __ldg(q);
                    if constexpr (C != 1) { vg[rr][k] = __ldg(q + 1); vr[rr][k] = __ldg(q + 2); }
                }
            }
        }
#pragma unroll
        for (int rr = 0; rr < RIT; ++rr) {
            const int sy = warp + rr * NWARP;
#pragma unroll
            for (int k = 0; k < CIT; ++k) {
                const int sx = lane + 32 * k;
                if (sy < SH && sx < SW) {
                    const int o = sy * SP + XO + sx;
                    if constexpr (C == 1) {
                        sB[o] = (float)vb[rr][k]; sP[o] = vb[rr][k];
                    } else {
                        sB[o] = (float)vb[rr][k]; sG[o] = (float)vg[rr][k]; sR[o] = (float)vr[rr][k];
                        sP[o] = vb[rr][k] | (vg[rr][k] << 8) | (vr[rr][k] << 16);
                    }
                }
            }
        }
    }
    for (int idx = tid; idx < 766; idx += NT) sCol[idx] = __ldg(p.color_lut + idx);
    if (tid < 25) sSp[tid] = __ldg(p.space_lut + tid);
    __syncthreads();

    // each thread owns a 4 x PY block of pixels.  PY = 2 (large launches): a staged row segment is fetched once
    // and serves the taps of both output rows (6 row fetches per 8 pixels instead of 10 -- shared-memory
    // wavefronts bound the kernel); PY = 1 (one frame): twice the warps, half the serial work per thread.
    // Per pixel the taps are visited dy-major, dx-minor either way: same sums, same bits.
    const int lx = tid % (TW / 4), ly = tid / (TW / 4);   // ly indexes groups of PY rows
    const uint32_t sCol_addr = smem_u32(sCol);
    uint32_t c[PY][4];
    float s0[PY][4], s1[PY][4], s2[PY][4], ws[PY][4];
#pragma unroll
    for (int o = 0; o < PY; ++o) {
        const uint4 c4 = *reinterpret_cast<const uint4*>(sP + (PY * ly + o + R) * SP + 4 * lx + 4);
        c[o][0] = c4.x; c[o][1] = c4.y; c[o][2] = c4.z; c[o][3] = c4.w;
#pragma unroll
        for (int k = 0; k < 4; ++k) { s0[o][k] = 0.f; s1[o][k] = 0.f; s2[o][k] = 0.f; ws[o][k] = 0.f; }
    }
#pragma unroll
    for (int sr = 0; sr < 4 + PY; ++sr) {
        // columns [4*lx, 4*lx + 12) of the staged row: pixel k, tap dx sits at local column XO + k + dx
        float rb[12], rg[12], rr[12];
        uint32_t rp[12];
        const int base = (PY * ly + sr) * SP + 4 * lx;
#pragma unroll
        for (int v = 0; v < 3; ++v) {
            if constexpr (C == 1) {
                const float4 b4 = *reinterpret_cast<const float4*>(sB + base + 4 * v);
                const uint4 p4 = *reinterpret_cast<const uint4*>(sP + base + 4 * v);
                rb[4 * v] = b4.x; rb[4 * v + 1] = b4.y; rb[4 * v + 2] = b4.z; rb[4 * v + 3] = b4.w;
                rp[4 * v] = p4.x; rp[4 * v + 1] = p4.y; rp[4 * v + 2] = p4.z; rp[4 * v + 3] = p4.w;
            } else {
                const float4 b4 = *reinterpret_cast<const float4*>(sB + base + 4 * v);
                const float4 g4 = *reinterpret_cast<const float4*>(sG + base + 4 * v);
                const float4 r4 = *reinterpret_cast<const float4*>(sR + base + 4 * v);
                const uint4 p4 = *reinterpret_cast<const uint4*>(sP + base + 4 * v);
                rb[4 * v] = b4.x; rb[4 * v + 1] = b4.y; rb[4 * v + 2] = b4.z; rb[4 * v + 3] = b4.w;
                rg[4 * v] = g4.x; rg[4 * v + 1] = g4.y; rg[4 * v + 2] = g4.z; rg[4 * v + 3] = g4.w;
                rr[4 * v] = r4.x; rr[4 * v + 1] = r4.y; rr[4 * v + 2] = r4.z; rr[4 * v + 3] = r4.w;
                rp[4 * v] = p4.x; rp[4 * v + 1] = p4.y; rp[4 * v + 2] = p4.z; rp[4 * v + 3] = p4.w;
            }
        }
#pragma unroll
        for (int o = 0; o < PY; ++o) {
            const int dy = sr - o;
            if (dy < 0 || dy > 4) continue;   // compile time
#pragma unroll
            for (int dx = 0; dx < 5; ++dx) {
                if ((dx - 2) * (dx - 2) + (dy - 2) * (dy - 2) > 4) continue;  // outside the circle (compile time)
                const float sw = sSp[dy * 5 + dx];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int col = XO + k + dx;
                    // IDP.4A with weights 4 and the table's shared-memory address as accumulator: the byte address of
                    // sCol[L1 distance] in one instruction (no separate index scaling)
                    const uint32_t ad = __vabsdiffu4(rp[col], c[o][k]);
                    const float w = __fmul_rn(sw, lds_f32(__dp4a(ad, 0x04040404u, sCol_addr)));
                    s0[o][k] = __fmaf_rn(w, rb[col], s0[o][k]);
                    if constexpr (C != 1) {
                        s1[o][k] = __fmaf_rn(w, rg[col], s1[o][k]);
                        s2[o][k] = __fmaf_rn(w, rr[col], s2[o][k]);
                    }
                    ws[o][k] = __fadd_rn(ws[o][k], w);
                }
            }
        }
    }
    const int gx = x0 + 4 * lx;
    if (gx >= p.width) return;
#pragma unroll
    for (int o = 0; o < PY; ++o) {
        const int gy = y0 + PY * ly + o;
        if (gy >= p.height) continue;
        uint32_t ov[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if constexpr (C == 1) ov[k] = presmooth_pack1(s0[o][k], ws[o][k]);
            else ov[k] = presmooth_pack(s0[o][k], s1[o][k], s2[o][k], ws[o][k]);
        }
        uint32_t* dst = p.guide4 + (long long)frame * p.guide_frame_stride + (long long)gy * p.guide_pitch + gx;
        if (gx + 3 < p.width && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
            *reinterpret_cast<uint4*>(dst) = make_uint4(ov[0], ov[1], ov[2], ov[3]);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (gx + k < p.width) dst[k] = ov[k];
        }
    }
}

// packed C-channel guide -> internal u8x4 without smoothing (pre-smooth disabled, MRF)
template <int C>
__global__ void bgr_to_guide4_kernel(const uint8_t* bgr, long long bgr_step, long long bgr_frame_stride,
                                     uint32_t* guide4, int guide_pitch, long long guide_frame_stride, int width,
                                     int height) {
    const int gx = blockIdx.x * blockDim.x + threadIdx.x, gy = blockIdx.y;
    const int frame = blockIdx.z;
    if (gx >= width || gy >= height) return;
    const uint8_t* q = bgr + (long long)frame * bgr_frame_stride + (long long)gy * bgr_step + C * gx;
    if constexpr (C == 1)
        guide4[(long long)frame * guide_frame_stride + (long long)gy * guide_pitch + gx] = (uint32_t)__ldg(q);
    else
        guide4[(long long)frame * guide_frame_stride + (long long)gy * guide_pitch + gx] =
            (uint32_t)__ldg(q) | ((uint32_t)__ldg(q + 1) << 8) | ((uint32_t)__ldg(q + 2) << 16);
}

// internal u8x4 -> continuous image of the caller's format (getSmoothImage_Device, JointBilateralFilter.cpp:47-49):
// GRAY gives byte 0, BGR bytes 0..2, BGRX bytes 0..2 and 255 as the 4th byte
template <int C>
__global__ void guide4_to_image_kernel(const uint32_t* guide4, int guide_pitch, uint8_t* img, int width, int height) {
    const int gx = blockIdx.x * blockDim.x + threadIdx.x, gy = blockIdx.y;
    if (gx >= width || gy >= height) return;
    const uint32_t v = guide4[(long long)gy * guide_pitch + gx];
    if constexpr (C == 4) {
        reinterpret_cast<uint32_t*>(img)[(long long)gy * width + gx] = v | 0xff000000u;
    } else {
        uint8_t* q = img + ((long long)gy * width + gx) * C;
        q[0] = (uint8_t)(v & 0xff);
        if constexpr (C == 3) {
            q[1] = (uint8_t)((v >> 8) & 0xff);
            q[2] = (uint8_t)((v >> 16) & 0xff);
        }
    }
}

}  // namespace kdme
