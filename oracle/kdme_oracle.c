/*
 * kdme_oracle.c -- CPU oracle for the joint-bilateral depth-enhancement hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product path (the package
 * kinectdepthmapenhancement_b200/ or its C-ABI library) may include, link or
 * call this file.  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs use it, and only as the checker or the
 * reported CPU baseline.
 *
 * It is an independently written restatement, in plain C, of the arithmetic the
 * reference performs on its GPU for this path.  Each function cites the
 * reference file:line it follows (paths relative to the reference checkout):
 *
 *   JointBilateralFilter/JointBilateralFilter.cpp:3-6,31-40   constants, spatial LUT
 *   JointBilateralFilter/JointBilateralFilter.cu:4-83         two-pass JBF kernel
 *   JointBilateralFilter/JointBilateralFilter.cu:285          guide pre-smooth call
 *   EdgeRefinedSuperpixel/EdgeRefinedSuperpixel.cu:104-205    guided cross-bilateral fill
 *   EdgeRefinedSuperpixel/EdgeRefinedSuperpixel.cpp:4-7,46-55 its constants and LUT
 *   ArrayBuffer/ArrayBuffer.cu:9-22, ArrayBuffer/Buffer2D.cu:13-140  device buffers
 *   MarkovRandomField/MarkovRandomField.cu:4-40               (next row f1)
 *   Projection_GPU/Projection_GPU.cu:213-246                  (next row f2)
 *   DimensionConvertor/DimensionConvertor.h:34-75             (next row f3)
 *   main.cpp:217-308                                          (next row f4, error metric)
 *
 * Parity pinning: the reference holds NO golden vectors, tests or fixtures for
 * this path (SURVEY.md section 4).  The restatement is pinned instead against
 * the reference's own kernel text compiled for the host (oracle/_ref, built by
 * oracle/build_ref.py from the sources where they lie in a reference checkout):
 * tests/test_oracle.py asserts bit-for-bit equality in fp32 against the
 * committed golden vectors always, and live whenever oracle/_ref is populated.  The third-party guide pre-smooth
 * (cv::gpu::bilateralFilter, OpenCV 2.4.3, not in the reference) is
 * "parity unpinned": restated from its published algorithm and cross-checked
 * against cv2.bilateralFilter (OpenCV 4.13 CPU) in tests/.
 *
 * Build: gcc -O2 -fopenmp -ffp-contract=off -fno-fast-math (see oracle/Makefile).
 * -ffp-contract=off keeps the fp32 evaluation un-fused on every host.
 *
 * Deviation from the reference shared by every function here: the reference
 * launches grid (W/32, H/24) with no in-kernel guard, so rows/cols beyond the
 * last full 32x24 block are never written (JointBilateralFilter.cu:289).  The
 * oracle computes every pixel.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_API __attribute__((visibility("default")))

/* fp32 expf underflows to exactly 0 below -150*ln2 (no FTZ; denormals kept).
 * The reference's skip-if-zero guards (JointBilateralFilter.cu:30-33,63-68)
 * therefore fire when the exponent argument is beyond this bound. */
#define ORC_EXP_ZERO_ARG 103.97207708399179

/* ------------------------------------------------------------------------- */
/* Spatial LUT -- JointBilateralFilter.cpp:31-40 (same text in
 * EdgeRefinedSuperpixel.cpp:46-55).  powf(x, 2.0f) of a small integer is exact
 * and equals x*x; evaluated in fp32 on the host exactly as the reference does. */
ORC_API void orc_spatial_lut(float *lut, int window_size, float spatial_sigma)
{
    for (int i = 0; i < window_size; i++) {
        for (int j = 0; j < window_size; j++) {
            float fx = (float)(j - window_size / 2);
            float fy = (float)(i - window_size / 2);
            float dis_x = fx * fx;
            float dis_y = fy * fy;
            float den = 2.0f * (spatial_sigma * spatial_sigma);
            lut[i * window_size + j] = expf(-(dis_x + dis_y) / den);
        }
    }
}

/* ------------------------------------------------------------------------- */
/* Guide pre-smooth -- stands in for cv::gpu::bilateralFilter(color, smooth, 5,
 * 30.0f, 30.0f) at JointBilateralFilter.cu:285.  OpenCV 2.4.3 gpu module
 * (pinned by release_x64.props:13) is not vendored in the reference; this is
 * its published algorithm: circular window dx^2+dy^2 <= (ksize/2)^2, weight
 * exp(-space2/(2 ss^2)) * exp(-L1(dBGR)^2/(2 sc^2)), reflect-101 border,
 * round-to-nearest-even saturate to u8.  Weights are taken from two fp32 LUTs
 * multiplied in fp32 and accumulated with one fused multiply-add per channel in
 * tap order (cy outer, cx inner), so a device implementation fed the same LUTs
 * is bit-exact.
 * PARITY UNPINNED for this stage (third-party, no reference fixture). */
static int orc_reflect101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) {
        if (p < 0) p = -p;
        else p = 2 * (len - 1) - p;
    }
    return p;
}

ORC_API void orc_presmooth_luts(float *space_lut /*[ksize*ksize], <0 = outside circle*/,
                                float *color_lut /*[766]*/, int ksize,
                                float sigma_color, float sigma_spatial)
{
    int r = ksize / 2;
    float ss = -0.5f / (sigma_spatial * sigma_spatial);
    float sc = -0.5f / (sigma_color * sigma_color);
    for (int dy = -r; dy <= r; dy++)
        for (int dx = -r; dx <= r; dx++) {
            int s2 = dx * dx + dy * dy;
            space_lut[(dy + r) * ksize + (dx + r)] = (s2 > r * r) ? -1.0f : expf((float)s2 * ss);
        }
    for (int n = 0; n <= 765; n++) color_lut[n] = expf((float)(n * n) * sc);
}

ORC_API void orc_presmooth_bgr(const uint8_t *src, size_t src_step, uint8_t *dst, size_t dst_step,
                               int dst_channels /*3 or 4 (4th = 0)*/, int width, int height,
                               int ksize, float sigma_color, float sigma_spatial)
{
    int r = ksize / 2;
    float *space_lut = (float *)malloc(sizeof(float) * ksize * ksize);
    float color_lut[766];
    orc_presmooth_luts(space_lut, color_lut, ksize, sigma_color, sigma_spatial);
#pragma omp parallel for schedule(dynamic, 4)
    for (int y = 0; y < height; y++) {
        for (int x = 0; x < width; x++) {
            const uint8_t *c = src + (size_t)y * src_step + (size_t)x * 3;
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, ws = 0.f;
            for (int dy = -r; dy <= r; dy++) {
                int yy = orc_reflect101(y + dy, height);
                for (int dx = -r; dx <= r; dx++) {
                    float sw = space_lut[(dy + r) * ksize + (dx + r)];
                    if (sw < 0.f) continue;
                    int xx = orc_reflect101(x + dx, width);
                    const uint8_t *q = src + (size_t)yy * src_step + (size_t)xx * 3;
                    int l1 = abs((int)q[0] - (int)c[0]) + abs((int)q[1] - (int)c[1]) +
                             abs((int)q[2] - (int)c[2]);
                    float wgt = sw * color_lut[l1];
                    s0 = fmaf(wgt, (float)q[0], s0);   /* one rounding per tap: a device FFMA is bit-identical */
                    s1 = fmaf(wgt, (float)q[1], s1);
                    s2 = fmaf(wgt, (float)q[2], s2);
                    ws = ws + wgt;
                }
            }
            uint8_t *o = dst + (size_t)y * dst_step + (size_t)x * dst_channels;
            float v0 = nearbyintf(s0 / ws), v1 = nearbyintf(s1 / ws), v2 = nearbyintf(s2 / ws);
            o[0] = (uint8_t)(v0 < 0.f ? 0.f : (v0 > 255.f ? 255.f : v0));
            o[1] = (uint8_t)(v1 < 0.f ? 0.f : (v1 > 255.f ? 255.f : v1));
            o[2] = (uint8_t)(v2 < 0.f ? 0.f : (v2 > 255.f ? 255.f : v2));
            if (dst_channels == 4) o[3] = 0;
        }
    }
    free(space_lut);
}

/* ------------------------------------------------------------------------- */
/* Two-pass joint bilateral filter, fp32, reference tap order --
 * JointBilateralFilter.cu:4-83.  `guide` is the (pre-smoothed) packed BGR image
 * indexed (y*width+x)*3+c exactly as the kernel does (it ignores the GpuMat
 * step, :22-24).  depth_sigma == 0 leaves depth_filter uninitialised in the
 * reference (:58-60); defined here as "factor skipped". */
static inline float orc_cdiff_f32(const uint8_t *g, int p, int q)
{
    float a0 = (float)g[p * 3 + 0] - (float)g[q * 3 + 0];
    float a1 = (float)g[p * 3 + 1] - (float)g[q * 3 + 1];
    float a2 = (float)g[p * 3 + 2] - (float)g[q * 3 + 2];
    return a0 * a0 + a1 * a1 + a2 * a2; /* left-to-right, as :22-24 */
}

ORC_API void orc_jbf_f32(int width, int height, const float *depth, const uint8_t *guide,
                         const float *spatial, float *out, int window_size, float color_sigma,
                         float depth_sigma, int n_threads)
{
    int half = window_size / 2;
    (void)n_threads;
#pragma omp parallel for schedule(dynamic, 2) num_threads(n_threads > 0 ? n_threads : 1)
    for (int y = 0; y < height; y++) {
        for (int x = 0; x < width; x++) {
            float w_average = 0.0f, weight = 0.0f;
            for (int i = -half; i <= half; i++) {
                for (int j = -half; j <= half; j++) {
                    int xj = x + j, yi = y + i;
                    if (xj >= 0 && xj < width && yi >= 0 && yi < height &&
                        depth[yi * width + xj] > 50.0f) {
                        float cd = orc_cdiff_f32(guide, y * width + x, yi * width + xj);
                        float cf = 0.0f;
                        if (color_sigma != 0.0f) cf = expf(-cd / (2 * (color_sigma * color_sigma)));
                        float f = 1.0f;
                        float s = spatial[(i + half) * window_size + (j + half)];
                        if (s != 0.0f) f *= s;
                        if (cf != 0.0f) f *= cf;
                        w_average += depth[yi * width + xj] * f;
                        weight += f;
                    }
                }
            }
            if (weight > 0.0f) {
                w_average /= weight;
                float num = 0.0f, den = 0.0f;
                for (int i = -half; i <= half; i++) {
                    for (int j = -half; j <= half; j++) {
                        int xj = x + j, yi = y + i;
                        if (xj >= 0 && xj < width && yi >= 0 && yi < height &&
                            depth[yi * width + xj] > 50.0f) {
                            float cd = orc_cdiff_f32(guide, y * width + x, yi * width + xj);
                            float cf = 0.0f;
                            if (color_sigma != 0.0f)
                                cf = expf(-cd / (2 * (color_sigma * color_sigma)));
                            float dd = depth[yi * width + xj] - w_average;
                            dd = dd * dd;
                            float df = 0.0f; /* sigma_d == 0: skipped */
                            if (depth_sigma != 0.0f)
                                df = expf(-dd / (2.0f * (depth_sigma * depth_sigma)));
                            float f = 1.0f;
                            float s = spatial[(i + half) * window_size + (j + half)];
                            if (s != 0.0f) f *= s;
                            if (cf != 0.0f) f *= cf;
                            if (df != 0.0f) f *= df;
                            num += depth[yi * width + xj] * f;
                            den += f;
                        }
                    }
                }
                out[y * width + x] = (den == 0.0f) ? 0.0f : num / den;
            } else {
                out[y * width + x] = 0.0f;
            }
        }
    }
}

/* Same formula evaluated in fp64 ("exact-math" oracle).  The only fp32 artefact
 * kept is the skip-if-zero rule, made explicit: a factor whose exponent
 * argument is below -150 ln2 is zero in fp32 and therefore skipped.  The
 * spatial LUT stays the reference's fp32 table (it is data, built on the host,
 * JointBilateralFilter.cpp:31-40).  No product underflow exists in fp64, so
 * out > 0 exactly where a valid tap exists (mask == window dilation). */
ORC_API void orc_jbf_f64(int width, int height, const float *depth, const uint8_t *guide,
                         const float *spatial, float *out, double *mean_out /*nullable*/,
                         int window_size, float color_sigma, float depth_sigma, int n_threads,
                         double mean_shift_ulps)
{
    /* mean_shift_ulps: the pass-1 mean is displaced by that many fp32 ulps before pass 2.  The
     * reference keeps w_average in a float (JointBilateralFilter.cu:16,40), so every output in
     * the envelope spanned by shifts of about +-1 ulp is a faithful evaluation of its formula;
     * tests use +-2 ulps to bound the conditioning of each pixel (DESIGN.md, "Tolerance"). */
    int half = window_size / 2;
    double kc = (color_sigma != 0.0f) ? 1.0 / (2.0 * (double)color_sigma * (double)color_sigma) : 0.0;
    double kd = (depth_sigma != 0.0f) ? 1.0 / (2.0 * (double)depth_sigma * (double)depth_sigma) : 0.0;
    (void)n_threads;
#pragma omp parallel for schedule(dynamic, 2) num_threads(n_threads > 0 ? n_threads : 1)
    for (int y = 0; y < height; y++) {
        for (int x = 0; x < width; x++) {
            double a = 0.0, wt = 0.0;
            const uint8_t *gp = guide + (size_t)(y * width + x) * 3;
            for (int pass = 0; pass < 2; pass++) {
                double m = 0.0, num = 0.0, den = 0.0;
                if (pass == 1) {
                    if (!(wt > 0.0)) break;
                    m = a / wt;
                    if (mean_out) mean_out[y * width + x] = m;
                    if (mean_shift_ulps != 0.0) {
                        float mf = (float)m;
                        m += mean_shift_ulps * (double)(nextafterf(mf, INFINITY) - mf);
                    }
                }
                for (int i = -half; i <= half; i++) {
                    for (int j = -half; j <= half; j++) {
                        int xj = x + j, yi = y + i;
                        if (!(xj >= 0 && xj < width && yi >= 0 && yi < height)) continue;
                        double d = (double)depth[yi * width + xj];
                        if (!(depth[yi * width + xj] > 50.0f)) continue;
                        const uint8_t *gq = guide + (size_t)(yi * width + xj) * 3;
                        double c0 = (double)gp[0] - gq[0], c1 = (double)gp[1] - gq[1],
                               c2 = (double)gp[2] - gq[2];
                        double cd = c0 * c0 + c1 * c1 + c2 * c2;
                        double f = 1.0;
                        float s = spatial[(i + half) * window_size + (j + half)];
                        if (s != 0.0f) f *= (double)s;
                        if (color_sigma != 0.0f && cd * kc <= ORC_EXP_ZERO_ARG) f *= exp(-cd * kc);
                        if (pass == 0) {
                            a += d * f;
                            wt += f;
                        } else {
                            double e = d - m;
                            if (depth_sigma != 0.0f && e * e * kd <= ORC_EXP_ZERO_ARG)
                                f *= exp(-e * e * kd);
                            num += d * f;
                            den += f;
                        }
                    }
                }
                if (pass == 1) out[y * width + x] = (den == 0.0) ? 0.0f : (float)(num / den);
            }
            if (!(wt > 0.0)) {
                out[y * width + x] = 0.0f;
                if (mean_out) mean_out[y * width + x] = 0.0;
            }
        }
    }
}

/* ------------------------------------------------------------------------- */
/* Guided cross-bilateral fill -- EdgeRefinedSuperpixel.cu:104-205, with the
 * race-free semantics (read `depth`, write `out`): the reference writes in
 * place while neighbouring threads still read (:197-203 vs :122,135,164,191),
 * which has no defined result.  `labels` may be NULL (all pixels one label).
 * color_sigma is a by-value kernel parameter mutated per valid tap in pass 2
 * (:170-176); restated literally, including the double-precision expression
 * 5.0*deviation/pow(w_average,2.0f) (pow(float,float) is the float overload in
 * CUDA C++, so the square is rounded to fp32 before the division). */
ORC_API void orc_guided_fill_f32(int width, int height, const float *depth, const uint8_t *guide,
                                 const int32_t *labels, const float *spatial, float *out,
                                 int window_size, float color_sigma_in, float depth_sigma,
                                 int n_threads)
{
    int half = window_size / 2;
    (void)n_threads;
#pragma omp parallel for schedule(dynamic, 2) num_threads(n_threads > 0 ? n_threads : 1)
    for (int y = 0; y < height; y++) {
        for (int x = 0; x < width; x++) {
            float color_sigma = color_sigma_in;
            float w_average = 0.0f, weight = 0.0f;
            int lp = labels ? labels[y * width + x] : 0;
            for (int i = -half; i <= half; i++)
                for (int j = -half; j <= half; j++) {
                    int xj = x + j, yi = y + i;
                    if (xj >= 0 && xj < width && yi >= 0 && yi < height &&
                        depth[yi * width + xj] > 50.0f &&
                        lp == (labels ? labels[yi * width + xj] : 0)) {
                        float cd = orc_cdiff_f32(guide, y * width + x, yi * width + xj);
                        float cf = 0.0f;
                        if (color_sigma != 0.0f) cf = expf(-cd / (2 * (color_sigma * color_sigma)));
                        float f = 1.0f;
                        float s = spatial[(i + half) * window_size + (j + half)];
                        if (s != 0.0f) f *= s;
                        if (cf != 0.0f) f *= cf;
                        w_average += depth[yi * width + xj] * f;
                        weight += f;
                    }
                }
            if (weight > 0.0f) {
                w_average /= weight;
                int count = 0;
                float deviation = 0.0f;
                for (int i = -half; i <= half; i++)
                    for (int j = -half; j <= half; j++) {
                        int xj = x + j, yi = y + i;
                        if (xj >= 0 && xj < width && yi >= 0 && yi < height &&
                            depth[yi * width + xj] > 50.0f &&
                            lp == (labels ? labels[yi * width + xj] : 0)) {
                            deviation += fabsf(depth[yi * width + xj] - w_average);
                            count++;
                        }
                    }
                if (count != 0) deviation /= (float)count;
                float num = 0.0f, den = 0.0f;
                for (int i = -half; i <= half; i++)
                    for (int j = -half; j <= half; j++) {
                        int xj = x + j, yi = y + i;
                        if (xj >= 0 && xj < width && yi >= 0 && yi < height &&
                            depth[yi * width + xj] > 50.0f) {
                            float cd = orc_cdiff_f32(guide, y * width + x, yi * width + xj);
                            float cf = 0.0f;
                            if (color_sigma != 0.0f) {
                                float wa2 = w_average * w_average;
                                float adaptive = (float)(5.0 * (double)deviation / (double)wa2);
                                if (adaptive > color_sigma * 0.3f) color_sigma = adaptive;
                                else color_sigma *= 0.3f;
                                cf = expf(-cd / (2 * (color_sigma * color_sigma)));
                            }
                            float dd = depth[yi * width + xj] - w_average;
                            dd = dd * dd;
                            float df = 0.0f;
                            if (depth_sigma != 0.0f)
                                df = expf(-dd / (2.0f * (depth_sigma * depth_sigma)));
                            float f = 1.0f;
                            float s = spatial[(i + half) * window_size + (j + half)];
                            if (s != 0.0f) f *= s;
                            if (cf != 0.0f) f *= cf;
                            if (df != 0.0f) f *= df;
                            num += depth[yi * width + xj] * f;
                            den += f;
                        }
                    }
                out[y * width + x] = (den == 0.0f) ? 0.0f : num / den;
            } else {
                out[y * width + x] = 0.0f;
            }
        }
    }
}

/* fp64 evaluation of the same three sweeps ("exact-math" oracle for the guided fill).  Sums,
 * mean and deviation are in double; the colour-sigma recurrence stays the reference's fp32
 * sequence (it is a discrete state machine: sigma *= 0.3f or sigma = adaptive, :172-175) driven
 * by the fp32 rounding of 5.0*deviation/mean^2; the skip-if-zero guards are the explicit
 * arg < -150 ln2 tests; -0/0 (sigma^2 underflowed to 0 with cd == 0) poisons the pixel with NaN
 * exactly as expf(NaN) does in the reference.  The sweep-1 mean is summed about the first
 * same-label sample d0, m = d0 + sum f (d - d0) / sum f (d - d0 is exact in double), so a window of
 * one depth has that depth as its mean and a deviation of exactly 0 whatever the weights' rounding.
 *
 * guard_out (nullable) flags the pixels at which the fp32 formula jumps: some quantity that decides
 * a branch lies within ORC_GUARD_ULPS fp32 ulps of its threshold, so an evaluation whose inputs
 * differ from these by rounding alone may take the other side (DESIGN.md section 2):
 *   1  a colour argument cd/dn (sweep 1 or sweep 3) or a sweep-3 depth argument e^2 kd at the
 *      expf() zero cut, past which the factor is skipped and the tap gets full weight;
 *   2  the recurrence test adaptive > sigma*0.3f, whose fp32 `adaptive` rounds 5*dev/mean^2;
 *   4  2 sigma^2 at the fp32 underflow boundary with sigma = adaptive: it decides -0/0 = NaN.
 * adaptive == 0 (a window of one depth, deviation exactly 0) is exact, so it flags nothing. */
#define ORC_GUARD_ULPS 8.0

static int orc_near_cut(double arg)
{
    const double cut = ORC_EXP_ZERO_ARG;
    const double ulp = (double)(nextafterf((float)cut, INFINITY) - (float)cut);
    return fabs(arg - cut) <= ORC_GUARD_ULPS * ulp;
}

ORC_API void orc_guided_fill_f64(int width, int height, const float *depth, const uint8_t *guide,
                                 const int32_t *labels, const float *spatial, float *out,
                                 double *mean_out /*nullable*/, uint8_t *guard_out /*nullable*/,
                                 int window_size, float color_sigma_in, float depth_sigma, int n_threads)
{
    int half = window_size / 2;
    double kd = (depth_sigma != 0.0f) ? 1.0 / (2.0 * (double)depth_sigma * (double)depth_sigma) : 0.0;
    (void)n_threads;
#pragma omp parallel for schedule(dynamic, 2) num_threads(n_threads > 0 ? n_threads : 1)
    for (int y = 0; y < height; y++) {
        for (int x = 0; x < width; x++) {
            int lp = labels ? labels[y * width + x] : 0;
            const uint8_t *gp = guide + (size_t)(y * width + x) * 3;
            double a = 0.0, wt = 0.0, d0 = 0.0;
            int guard = 0;
            double den0 = 2.0 * (double)color_sigma_in * (double)color_sigma_in;
            for (int i = -half; i <= half; i++)
                for (int j = -half; j <= half; j++) {
                    int xj = x + j, yi = y + i;
                    if (!(xj >= 0 && xj < width && yi >= 0 && yi < height)) continue;
                    if (!(depth[yi * width + xj] > 50.0f)) continue;
                    if (lp != (labels ? labels[yi * width + xj] : 0)) continue;
                    const uint8_t *gq = guide + (size_t)(yi * width + xj) * 3;
                    double c0 = (double)gp[0] - gq[0], c1 = (double)gp[1] - gq[1], c2 = (double)gp[2] - gq[2];
                    double cd = c0 * c0 + c1 * c1 + c2 * c2;
                    double f = 1.0;
                    float s = spatial[(i + half) * window_size + (j + half)];
                    if (s != 0.0f) f *= (double)s;
                    if (color_sigma_in != 0.0f) {
                        if (orc_near_cut(cd / den0)) guard |= 1;
                        if (cd / den0 <= ORC_EXP_ZERO_ARG) f *= exp(-cd / den0);
                    }
                    if (wt == 0.0) d0 = (double)depth[yi * width + xj];
                    a += ((double)depth[yi * width + xj] - d0) * f;
                    wt += f;
                }
            if (mean_out) mean_out[y * width + x] = 0.0;
            if (guard_out) guard_out[y * width + x] = 0;
            if (!(wt > 0.0)) { out[y * width + x] = 0.0f; continue; }
            double m = d0 + a / wt;
            if (mean_out) mean_out[y * width + x] = m;
            double dev = 0.0; int count = 0;
            for (int i = -half; i <= half; i++)
                for (int j = -half; j <= half; j++) {
                    int xj = x + j, yi = y + i;
                    if (!(xj >= 0 && xj < width && yi >= 0 && yi < height)) continue;
                    if (!(depth[yi * width + xj] > 50.0f)) continue;
                    if (lp != (labels ? labels[yi * width + xj] : 0)) continue;
                    dev += fabs((double)depth[yi * width + xj] - m);
                    count++;
                }
            if (count != 0) dev /= (double)count;
            float mf = (float)m;
            float adaptive = (float)(5.0 * dev / (double)(mf * mf));
            float sigma = color_sigma_in;
            double num = 0.0, den = 0.0;
            int poisoned = 0;
            for (int i = -half; i <= half; i++)
                for (int j = -half; j <= half; j++) {
                    int xj = x + j, yi = y + i;
                    if (!(xj >= 0 && xj < width && yi >= 0 && yi < height)) continue;
                    if (!(depth[yi * width + xj] > 50.0f)) continue;
                    const uint8_t *gq = guide + (size_t)(yi * width + xj) * 3;
                    double c0 = (double)gp[0] - gq[0], c1 = (double)gp[1] - gq[1], c2 = (double)gp[2] - gq[2];
                    double cd = c0 * c0 + c1 * c1 + c2 * c2;
                    double f = 1.0;
                    float s = spatial[(i + half) * window_size + (j + half)];
                    if (s != 0.0f) f *= (double)s;
                    if (sigma != 0.0f) {
                        float t = sigma * 0.3f;
                        float hi = fmaxf(fabsf(adaptive), fabsf(t));
                        if (adaptive != 0.0f && fabsf(adaptive - t) <= (float)ORC_GUARD_ULPS * (nextafterf(hi, INFINITY) - hi)) guard |= 2;
                        if (adaptive > t) sigma = adaptive; else sigma = t;
                        float dn = 2 * (sigma * sigma);   /* fp32: may underflow to 0 */
                        if (adaptive != 0.0f && sigma == adaptive && dn <= (float)ORC_GUARD_ULPS * 0x1p-149f) guard |= 4;
                        if (dn == 0.0f) { if (cd == 0.0) poisoned = 1; /* cd > 0: expf(-inf) = 0, skipped */ }
                        else {
                            if (orc_near_cut(cd / (double)dn)) guard |= 1;
                            if (cd / (double)dn <= ORC_EXP_ZERO_ARG) f *= exp(-cd / (double)dn);
                        }
                    }
                    double e = (double)depth[yi * width + xj] - m;
                    if (depth_sigma != 0.0f) {
                        if (orc_near_cut(e * e * kd)) guard |= 1;
                        if (e * e * kd <= ORC_EXP_ZERO_ARG) f *= exp(-e * e * kd);
                    }
                    num += (double)depth[yi * width + xj] * f;
                    den += f;
                }
            if (guard_out) guard_out[y * width + x] = (uint8_t)guard;
            if (poisoned) out[y * width + x] = NAN;
            else out[y * width + x] = (den == 0.0) ? 0.0f : (float)(num / den);
        }
    }
}

/* ------------------------------------------------------------------------- */
/* Upsampling (config 3).  The reference only declares it in a comment
 * (JointBilateralFilter.h:14); SURVEY.md 8(d) defines it: each low-res sample
 * (xl,yl) lands at high-res pixel (floor((xl+.5)*wh/wl), floor((yl+.5)*hh/hl)),
 * every other high-res pixel is a hole, then the two-pass fill of
 * JointBilateralFilter.cu:4-83 runs on the sparse image.  This scatters the
 * sparse image; the callers run orc_jbf_* on it. */
ORC_API void orc_scatter_lowres(const float *depth_lo, int wl, int hl, float *sparse_hi, int wh,
                                int hh)
{
    memset(sparse_hi, 0, sizeof(float) * (size_t)wh * hh);
    for (int yl = 0; yl < hl; yl++)
        for (int xl = 0; xl < wl; xl++) {
            int xh = (int)(((int64_t)(2 * xl + 1) * wh) / (2 * wl));
            int yh = (int)(((int64_t)(2 * yl + 1) * hh) / (2 * hl));
            sparse_hi[(size_t)yh * wh + xh] = depth_lo[yl * wl + xl];
        }
}

/* ------------------------------------------------------------------------- */
/* Device buffers -- ArrayBuffer.h:12-15 (weighted_d {d,w}, 8 bytes AoS).
 * All element-wise; `buf` is interleaved d,w,d,w,...  n = width*height. */
ORC_API void orc_buf_init(float *buf, int width, int height)
{ /* ArrayBuffer.cu:9-22 */
    for (size_t k = 0; k < (size_t)width * height; k++) { buf[2 * k] = 0.0f; buf[2 * k + 1] = 0.0f; }
}
ORC_API void orc_buf_insert_f32(float *buf, const float *data, int width, int height)
{ /* Buffer2D.cu:33-50: d = data, w = 1 */
    for (size_t k = 0; k < (size_t)width * height; k++) { buf[2 * k] = data[k]; buf[2 * k + 1] = 1.0f; }
}
ORC_API void orc_buf_insert_f32x2(float *buf, const float *data_xy, int width, int height)
{ /* Buffer2D.cu:123-140: d = data.x, w = y (the ROW INDEX -- reference quirk, :137) */
    for (int y = 0; y < height; y++)
        for (int x = 0; x < width; x++) {
            size_t k = (size_t)y * width + x;
            buf[2 * k] = data_xy[2 * k];
            buf[2 * k + 1] = (float)y;
        }
}
ORC_API void orc_buf_get_depth(const float *buf, float *out, int width, int height)
{ /* Buffer2D.cu:59-70 */
    for (size_t k = 0; k < (size_t)width * height; k++) out[k] = buf[2 * k];
}
ORC_API void orc_buf_get_weight(const float *buf, float *out, int width, int height)
{ /* Buffer2D.cu:79-89 */
    for (size_t k = 0; k < (size_t)width * height; k++) out[k] = buf[2 * k + 1];
}
ORC_API void orc_buf_update(float *buf, const float *data, int width, int height)
{ /* Buffer2D.cu:97-113 -> updateWaitedDepth :13-30.  Un-fused fp32; the
     int casts truncate toward zero as C does (:20). */
    for (size_t k = 0; k < (size_t)width * height; k++) {
        float d = data[k];
        float rd = buf[2 * k], rw = buf[2 * k + 1];
        if ((double)d > 50.0) {
            if (rd != 0.0f) {
                if ((float)abs((int)rd - (int)d) < d * 0.01f) {
                    float t1 = rd * (rw + 1);
                    float t2 = d * rw;
                    rd = (t1 + t2) / (rw * 2 + 1);
                    rw = rw + 1.0f;
                }
            } else {
                rd = d;
                rw = 1.0f;
            }
        }
        buf[2 * k] = rd;
        buf[2 * k + 1] = rw;
    }
}

/* ------------------------------------------------------------------------- */
/* "Next" rows (SURVEY.md 8(f)). */

/* f1: MarkovRandomField.cu:4-40 -- one-pass colour-weighted mean seeded with
 * the centre depth (valid or not) and denominator 1. */
ORC_API void orc_mrf_f32(int width, int height, const float *depth, const uint8_t *guide, float *out,
                         int window_size, float color_sigma, float smooth_sigma, int n_threads)
{
    int half = window_size / 2;
    (void)n_threads;
#pragma omp parallel for schedule(dynamic, 2) num_threads(n_threads > 0 ? n_threads : 1)
    for (int y = 0; y < height; y++)
        for (int x = 0; x < width; x++) {
            float num = depth[y * width + x], den = 1.0f;
            for (int i = -half; i <= half; i++)
                for (int j = -half; j <= half; j++) {
                    int xj = x + j, yi = y + i;
                    if (xj >= 0 && xj < width && yi >= 0 && yi < height &&
                        depth[yi * width + xj] > 50.0f) {
                        float cd = orc_cdiff_f32(guide, y * width + x, yi * width + xj);
                        float cf = 0.0f;
                        if (color_sigma != 0.0f) cf = expf(-color_sigma * cd);
                        float f = smooth_sigma;
                        f *= cf;
                        num += depth[yi * width + xj] * f;
                        den += f;
                    }
                }
            out[y * width + x] = (den == 0.0f) ? 0.0f : num / den;
        }
}

/* fp64 evaluation of f1: same formula and tap order as orc_mrf_f32, accumulated in double; the only
 * fp32 artefact kept is that expf() == 0 below -150 ln2. */
ORC_API void orc_mrf_f64(int width, int height, const float *depth, const uint8_t *guide, float *out,
                         int window_size, float color_sigma, float smooth_sigma, int n_threads)
{
    int half = window_size / 2;
    (void)n_threads;
#pragma omp parallel for schedule(dynamic, 2) num_threads(n_threads > 0 ? n_threads : 1)
    for (int y = 0; y < height; y++)
        for (int x = 0; x < width; x++) {
            const uint8_t *gp = guide + 3 * ((size_t)y * width + x);
            double num = depth[y * width + x], den = 1.0;
            for (int i = -half; i <= half; i++)
                for (int j = -half; j <= half; j++) {
                    int xj = x + j, yi = y + i;
                    if (xj >= 0 && xj < width && yi >= 0 && yi < height &&
                        depth[yi * width + xj] > 50.0f) {
                        const uint8_t *gq = guide + 3 * ((size_t)yi * width + xj);
                        double cd = 0.0;
                        for (int c = 0; c < 3; c++) cd += ((double)gp[c] - gq[c]) * ((double)gp[c] - gq[c]);
                        double a = (double)color_sigma * cd;
                        double f = (color_sigma != 0.0f && a <= ORC_EXP_ZERO_ARG) ? exp(-a) : 0.0;
                        f *= (double)smooth_sigma;
                        num += (double)depth[yi * width + xj] * f;
                        den += f;
                    }
                }
            out[y * width + x] = (den == 0.0) ? 0.0f : (float)(num / den);
        }
}

/* f3: DimensionConvertor.h:34-75 via DimensionConvertor.cu:3-23 -- pixel
 * (u,v,z) -> camera XYZ; cx, cy are ints (DimensionConvertor.cpp:8-9).
 * Order of operations kept: subtract, divide by focal, multiply by z. */
ORC_API void orc_projective_to_real(const float *depth, float *xyz, int width, int height, float fx,
                                    float fy, int cx, int cy)
{
    for (int v = 0; v < height; v++)
        for (int u = 0; u < width; u++) {
            size_t k = (size_t)v * width + u;
            float z = depth[k];
            float px = (float)u, py = (float)v;
            py = (float)cy - py;
            px = px - (float)cx;
            px /= fx;
            py /= fy;
            px *= z;
            py *= z;
            xyz[3 * k + 0] = px;
            xyz[3 * k + 1] = py;
            xyz[3 * k + 2] = z;
        }
}

/* f2: Projection_GPU.cu:213-246 -- depth-only bilateral on the z of a point cloud, centred on the
 * pixel's own z (valid or not), weights expf(-dz^2/(2 sd^2)) * S (plain products, no skip guards),
 * then x,y = normalized.x,y * z.  Race-free restatement: reads `in`, writes `out` (the reference
 * overwrites optimized3d in place while neighbours read it).  xyz are packed float3. */
ORC_API void orc_depth_bilateral_xyz(const float *normalized, const float *in, float *out, const float *spatial,
                                     int window_size, float depth_sigma, int width, int height, int n_threads)
{
    int half = window_size / 2;
    (void)n_threads;
#pragma omp parallel for schedule(dynamic, 2) num_threads(n_threads > 0 ? n_threads : 1)
    for (int y = 0; y < height; y++)
        for (int x = 0; x < width; x++) {
            float num = 0.0f, den = 0.0f;
            float zc = in[3 * (y * width + x) + 2];
            for (int i = -half; i <= half; i++)
                for (int j = -half; j <= half; j++) {
                    int xj = x + j, yi = y + i;
                    if (xj >= 0 && xj < width && yi >= 0 && yi < height && in[3 * (yi * width + xj) + 2] > 50.0f) {
                        float zq = in[3 * (yi * width + xj) + 2];
                        float dd = zq - zc;
                        dd = dd * dd;
                        float f = expf(-dd / (2.0f * (depth_sigma * depth_sigma)));
                        f *= spatial[(i + half) * window_size + (j + half)];
                        num += zq * f;
                        den += f;
                    }
                }
            float z = (den == 0.0f) ? 0.0f : num / den;
            out[3 * (y * width + x) + 2] = z;
            out[3 * (y * width + x) + 0] = normalized[3 * (y * width + x) + 0] * z;
            out[3 * (y * width + x) + 1] = normalized[3 * (y * width + x) + 1] * z;
        }
}

/* f4: main.cpp:217-308 -- mean Euclidean distance (mm) between a method's cloud and the averaged
 * ground-truth cloud over pixels where both z are in (50, 15000); sequential float accumulation as
 * the reference does (pow(float,2.0f) is the float overload; sqrtf). */
ORC_API float orc_mean_3d_error(const float *pts, const float *truth, int n, int *count_out)
{
    float sum = 0.0f;
    int count = 0;
    for (int k = 0; k < n; k++) {
        float z = pts[3 * k + 2], zt = truth[3 * k + 2];
        if (z > 50.0f && z < 15000.0f && zt > 50.0f && zt < 15000.0f) {
            float dz = z - zt, dy = pts[3 * k + 1] - truth[3 * k + 1], dx = pts[3 * k] - truth[3 * k];
            sum += sqrtf(dz * dz + dy * dy + dx * dx);
            count++;
        }
    }
    if (count_out) *count_out = count;
    return sum / (float)count;
}

/* fp64 evaluation of f2 (same formula; the only fp32 artefact kept is that expf() == 0 below -150 ln2). */
ORC_API void orc_depth_bilateral_xyz_f64(const float *normalized, const float *in, float *out, const float *spatial,
                                         int window_size, float depth_sigma, int width, int height, int n_threads)
{
    int half = window_size / 2;
    double kd = 1.0 / (2.0 * (double)depth_sigma * (double)depth_sigma);
    (void)n_threads;
#pragma omp parallel for schedule(dynamic, 2) num_threads(n_threads > 0 ? n_threads : 1)
    for (int y = 0; y < height; y++)
        for (int x = 0; x < width; x++) {
            double num = 0.0, den = 0.0;
            double zc = in[3 * (y * width + x) + 2];
            for (int i = -half; i <= half; i++)
                for (int j = -half; j <= half; j++) {
                    int xj = x + j, yi = y + i;
                    if (xj >= 0 && xj < width && yi >= 0 && yi < height && in[3 * (yi * width + xj) + 2] > 50.0f) {
                        double zq = in[3 * (yi * width + xj) + 2];
                        double a = (zq - zc) * (zq - zc) * kd;
                        double f = (a <= ORC_EXP_ZERO_ARG) ? exp(-a) : 0.0;
                        f *= (double)spatial[(i + half) * window_size + (j + half)];
                        num += zq * f;
                        den += f;
                    }
                }
            float z = (den == 0.0) ? 0.0f : (float)(num / den);
            out[3 * (y * width + x) + 2] = z;
            out[3 * (y * width + x) + 0] = normalized[3 * (y * width + x) + 0] * z;
            out[3 * (y * width + x) + 1] = normalized[3 * (y * width + x) + 1] * z;
        }
}
