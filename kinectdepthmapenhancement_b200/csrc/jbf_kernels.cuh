// jbf_kernels.cuh -- two-pass joint bilateral depth filter for sm_100a.
//
// Computes what joint_bilateral_filtering computes (reference:
// JointBilateralFilter/JointBilateralFilter.cu:4-83) for every pixel of every
// frame, but organised for Blackwell:
//
//   * one CTA = one TW x TH output tile; the depth tile and the smoothed-guide
//     tile, each with its radius-r halo, are staged into shared memory by TMA
//     (cp.async.bulk.tensor, zero fill outside the image == the reference's
//     bounds test, .cu:21) -- or by plain coalesced loads when the frame pitch
//     is not 16-byte aligned, or by an on-the-fly low-res scatter (Upsampling);
//   * one sweep emits a "magic" word per staged sample that carries validity
//     (d > 50; holes and NaN read as depth 0);
//   * each thread owns 4 horizontally adjacent pixels and sweeps the window row
//     by row; a staged row segment is fetched once with 16-byte LDS and reused
//     by all 4 pixels (4*(2r+1) taps per 2r+4 fetched columns);
//   * a tap costs: VABSDIFF4 + IDP.4A (exact integer colour distance, validity
//     folded in through the accumulator) + FADD + FFMA (spatial-LUT row entry
//     + colour term) [+ FADD, FSETP, predicated FFMA for the depth-range term
//     in pass 2] + ONE MUFU.EX2 + FFMA + FADD.  No expf, no division, no
//     branch per tap;
//   * precision: depths enter as X = d*sq - fl(d0*sq) around a per-thread origin d0
//     (one rounding, relative to the small difference), pass-1 weights carry no
//     bias, row sums are combined with 2Sum, the mean is the correctly rounded
//     quotient of the compensated sums: every well-conditioned pixel lands within
//     1-2 ulps of the fp64 evaluation of the reference formula, independently of
//     the tile it falls in;
//   * pixels whose window holds no sample near the pass-1 mean (den/wsum tiny)
//     amplify the rounding of that mean beyond what fp32 can absorb: they are
//     queued and re-evaluated in fp64 by jbf_refine_kernel (one warp per pixel,
//     taps split across lanes, warp-shuffle reductions);
//   * the epilogue can also write the back-projected float3 cloud
//     (DimensionConvertor::projectiveToReal fused, main.cpp:179 + :182).
//
// The reference's quirks are kept: > 50 validity, hole filling (centre need not
// be valid), skip-if-zero guards (spatial: folded into the LUT; colour: cannot
// fire on this path, the host routes such sigmas to the generic kernel; depth:
// explicit |e| > sqrt(150) compare), two passes with the range term centred on
// the pass-1 mean.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace kdme {

enum StageMode : int { kStagePlain = 0, kStageTma = 1, kStageUpsample = 2 };

struct JbfParams {
    int width, height, n_frames;
    const void* depth;           // [n][H][W] float32, or uint16 millimetres when depth_u16 (plain / TMA)
    const uint32_t* guide4;      // [n][H][guide_pitch] u8x4 BGR0  (smoothed guide)
    float* out;                  // [n][H][W]
    long long depth_frame_stride;   // elements
    long long guide_frame_stride;   // words
    int guide_pitch;                // words per row
    const float* ltab;           // generic kernel: [(2r+1)][(2r+1)] log2(S_ij)+bias, or bias where S_ij == 0
    const float* ltab_pairs;     // pass 2: [(2r+1)][LPP][2] = {L[i][j], L[i][j-1]}, j = 1..2r, bias kWeightBias
    const float* ltab_pairs1;    // pass 1: same layout, bias `bias1` (0 whenever no pass-1 weight can flush)
    const float* slut;           // the reference's raw fp32 spatial LUT [(2r+1)^2] (fp64 refinement path)
    float nkc;                   // -log2e / (2 sigma_c^2)
    float sq, inv_sq;            // depth scale sqrt(log2e/(2 sigma_d^2)) and inverse
    float e_thr;                 // sqrt(150): scaled |d - m| beyond which fp32 expf() == 0
    float flag_scale;            // a pixel is refined in fp64 when den < wsum * flag_scale (ill-conditioned)
    double kc, kd;               // 1/(2 sigma_c^2), 1/(2 sigma_d^2) (fp64 refinement path)
    int mode;                    // StageMode
    // upsample: the low-res depth [n][hl][wl], float32 (depth_lo) or uint16 millimetres (depth_lo16, when non-null),
    // read through upsample_sample.  A pointer pair rather than `depth` and depth_u16: with the block's layout and this
    // null test as they are, jbf_upsample_gather_kernel keeps its code (any other form re-scheduled it, 0.5 % slower)
    const float* depth_lo;
    const uint16_t* depth_lo16;
    long long lo_frame_stride;   // samples per low-res frame (wl * hl)
    int wl, hl;
    const int* ups_inv_x;        // upsample, optional: low-res column landing on high-res column x, or -1 ([width]); null = compute
    const int* ups_inv_y;        // same for rows ([height])
    // row-band mode: the arrays hold `height` rows (band + halos); output rows are
    // [y_off, y_off + out_rows) of them and `out` holds only those.  Results do not depend on where
    // tiles start vertically, so a band equals the same rows of the whole image bit for bit.
    // Whole-image mode: y_off = 0, out_rows = height.
    int y_off, out_rows;
    // load balance of small launches: tile rows [0, nbig_rows) have the template's height TH, the rows below
    // are cut into tiles of `ts` rows (a multiple of 2: whole warps), so that the work beyond a whole number
    // of big tiles per SM is spread over many SMs instead of landing on a few.  All big: nbig_rows = INT_MAX.
    int nbig_rows, ts;
    // half_units != 0: every small tile appears twice in the grid (consecutive blockIdx.y), once per pixel pair --
    // see jbf_fast_body's PSEL
    int half_units;
    // peer-memory halos (row bands over NVLink): rows [band0, band1) of the arrays are this rank's own;
    // when depth_up / depth_dn are non-null, rows above / below are read straight from the neighbour
    // GPU's band through these peer-mapped pointers (depth_up + row*W for row < band0,
    // depth_dn + (row - band1)*W for row >= band1) instead of from local halo copies.
    const float* depth_up;
    const float* depth_dn;
    int band0, band1;
    // fused back-projection epilogue (DimensionConvertor::projectiveToReal, DimensionConvertor.h:34-48):
    // when xyz != nullptr the kernel also writes float3 {x, y, z} per pixel, [n][out_rows][W][3]
    float* xyz;
    float fx, fy;
    int cx, cy;
    int y_img0;                  // image row of array row 0 (bands), for the back-projection's v
    // ill-conditioned pixels are queued here by the filter kernel and re-evaluated in fp64 by
    // jbf_refine_kernel: q_count[0] = number pushed (may exceed q_capacity: the excess is dropped and
    // counted), q_items = linear output indices (frame * out_rows * W + oy * W + x)
    unsigned int* q_count;       // [0] pushed by this launch
    unsigned int* q_count_prev;  // the previous launch's counter (two alternate): re-armed by this launch's filter kernel
    unsigned int* q_items;
    unsigned int q_capacity;
    // 1: the plain / TMA depth is uint16 millimetres, read by the DT = uint16_t instantiations (whole frames only: no
    // row bands, no peer halos).  Kept in q_capacity's padding, so the layout of the block stays as it was.
    int depth_u16;
    unsigned long long* stats;   // [0] += pixels refined in fp64, [1] += pixels dropped (queue full)
};

template <int R, int TW, int TH>
struct JbfTile {
    static constexpr int WS = 2 * R + 1;
    static constexpr int RP = (R + 3) & ~3;        // halo columns rounded up to a 16-byte multiple
    static constexpr int SP = TW + 2 * RP;         // staged row pitch (words)
    static constexpr int SH = TH + 2 * R;          // staged rows
    static constexpr int NT = (TW / 4) * TH;       // threads per CTA
    static constexpr int NW = 2 * RP + 4;          // words fetched per row per thread
    static constexpr int C0 = RP - R;              // first used column of the fetched segment
    static constexpr int PLANE = ((SP * SH * 4 + 127) / 128) * 128;
    static constexpr int LPP = (WS - 1 + 1) & ~1;  // pairs per LUT row, padded to an even count (16-byte rows)
    static constexpr int LBYTES = ((WS * LPP * 2 * 4 + 127) / 128) * 128;   // one paired table
    static constexpr int SMEM = 3 * PLANE + 2 * LBYTES + 128;
    // uint16 TMA staging: halo columns rounded up to 8, so that every box starts on a 16-byte boundary of the row as
    // the float32 boxes do (RP * 4 bytes); SP16 * SH half-words fit in one plane
    static constexpr int RP16 = (R + 7) & ~7;
    static constexpr int SP16 = TW + 2 * RP16;
    static_assert((SP16 * 2) % 16 == 0 && SP16 * SH * 2 <= PLANE, "uint16 TMA box: 16-byte rows inside one plane");
};

// low-res sample (xl, yl) of `frame`: every upsampling kernel reads the low-res depth through here.  Its type is a
// run-time branch, so the upsampling kernels have one instantiation for both types.
__device__ __forceinline__ float upsample_sample(const JbfParams& p, int frame, int xl, int yl) {
    const long long i = (long long)frame * p.lo_frame_stride + (long long)yl * p.wl + xl;
    return p.depth_lo16 ? load_depth<uint16_t>(p.depth_lo16, i) : load_depth<float>(p.depth_lo, i);
}

// pass-1 row sums are first added plainly in groups of this many window rows, the group sums are then
// combined error-free (2Sum); the gather-form upsampling kernel uses the same grouping
constexpr int kRowsPer2Sum = 3;

// Knuth 2Sum on both lanes: a + b == s + t exactly; a <- s, lo += t.
__device__ __forceinline__ void two_sum2(f32x2& a, const f32x2 b, f32x2& lo) {
    const f32x2 s = add2(a, b);
    const f32x2 bb = sub2(s, a);
    const f32x2 t = add2(sub2(a, sub2(s, bb)), sub2(b, bb));
    a = s;
    lo = add2(lo, t);
}

// PSEL: 0 = the thread computes its 4 pixels; 1 / 2 = only pixels (0,1) / (2,3) of its group -- a HALF work unit: the
// other pair's instruction stream does not exist in that instantiation, so the warp costs half the MUFU / FMA time.
// Launches of a few waves hand the tiles beyond a whole number per SM out as such halves (JbfParams::half_units):
// a warp instruction costs the same pipe time however few lanes are active (tools/mufu_lanes.cu), so work can only
// be cut finer than a warp by dropping instructions.  Same arithmetic per pixel (the accumulation origin is still
// that of the 4-pixel group): results are bit-identical whichever way a pixel is computed.
// DT: the plain / TMA depth is float32 or uint16 millimetres (JbfParams::depth_u16); every step from stage B on is the
// same for both.
template <int R, int TW, int TH, int PSEL, class DT>
__device__ __forceinline__ void jbf_fast_body(const CUtensorMap& tm_depth, const CUtensorMap& tm_guide, const JbfParams& p) {
    using T = JbfTile<R, TW, TH>;
    constexpr int WS = T::WS, RP = T::RP, SP = T::SP, SH = T::SH, NT = T::NT, NW = T::NW, C0 = T::C0;
    constexpr int LPP = T::LPP;

    extern __shared__ __align__(128) uint8_t smem_fast[];
    float* sD = reinterpret_cast<float*>(smem_fast);
    uint32_t* sG = reinterpret_cast<uint32_t*>(smem_fast + T::PLANE);
    uint32_t* sM = reinterpret_cast<uint32_t*>(smem_fast + 2 * T::PLANE);
    float* sL1 = reinterpret_cast<float*>(smem_fast + 3 * T::PLANE);
    float* sL2 = reinterpret_cast<float*>(smem_fast + 3 * T::PLANE + T::LBYTES);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_fast + 3 * T::PLANE + 2 * T::LBYTES);
    float* sRed = reinterpret_cast<float*>(smem_fast + 3 * T::PLANE + 2 * T::LBYTES + 16);   // 2 * NT/32 <= 16 floats

    const int tid = threadIdx.x;
    const bool big = (int)blockIdx.y < p.nbig_rows;
    const int th_eff = big ? TH : p.ts;                       // rows of this tile
    const int she = th_eff + 2 * R;                           // staged rows this tile needs
    const int x0 = blockIdx.x * TW, frame = blockIdx.z;
    const int small_idx = ((int)blockIdx.y - p.nbig_rows) >> (p.half_units ? 1 : 0);   // two half units per small tile
    const int y0 = p.y_off + (big ? (int)blockIdx.y * TH : p.nbig_rows * TH + small_idx * p.ts);
    const int sx0 = x0 - RP, sy0 = y0 - R;  // image coords of staged (0,0)
    // a tile whose halo crosses into a neighbour GPU's rows stages with plain loads (peer pointers);
    // every other tile keeps the launch's staging mode (CTA-uniform)
    const bool seam = (p.depth_up != nullptr && sy0 < p.band0) || (p.depth_dn != nullptr && sy0 + SH > p.band1);
    const int mode = seam ? (int)kStagePlain : p.mode;

    // ---------------- stage A: raw depth + guide tile with halo -> shared memory
    if (mode == kStageTma) {
        if (tid == 0) {
            tma_prefetch_desc(&tm_depth);
            tma_prefetch_desc(&tm_guide);
            mbar_init(bar, 1);
            fence_mbar_init();
        }
    }
    // spatial LUT rows (log2 domain, paired for the packed math; host data, not produced by a prior kernel)
    for (int idx = tid; idx < WS * LPP * 2; idx += NT) {
        sL1[idx] = __ldg(p.ltab_pairs1 + idx);
        sL2[idx] = __ldg(p.ltab_pairs + idx);
    }
    // programmatic dependent launch: everything above overlaps the tail of the pre-smooth kernel; the
    // guide it writes is only read below this point (no-op when launched without the attribute)
    grid_dependency_wait();
    // re-arm the queue counter the PREVIOUS launch used (its refine kernel has completed: it precedes this
    // kernel's stream predecessor, or is it); this launch pushes to the other one
    if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) *p.q_count_prev = 0u;
    if (mode == kStageTma) {
        __syncthreads();
        if (tid == 0) {
            if constexpr (std::is_same<DT, uint16_t>::value) {
                // the uint16 tile (SP16 columns from x0 - RP16) lands in sM, free until stage B, and is widened
                // into sD below
                mbar_expect_tx(bar, (uint32_t)(SP * SH * 4 + T::SP16 * SH * 2));
                tma_load_3d(sM, &tm_depth, bar, x0 - T::RP16, sy0, frame);
            } else {
                mbar_expect_tx(bar, 2u * SP * SH * 4u);
                tma_load_3d(sD, &tm_depth, bar, sx0, sy0, frame);
            }
            tma_load_3d(sG, &tm_guide, bar, sx0, sy0, frame);
        }
    } else {
        const uint32_t* gsrc = p.guide4 + (long long)frame * p.guide_frame_stride;
        const DT* dsrc = static_cast<const DT*>(p.depth) + (long long)frame * p.depth_frame_stride;
        // upsample: the low-res sample (if any) of every staged column and row, computed once per tile
        // (sM is free until stage B: its first SP + SH words hold the two maps)
        int* colmap = reinterpret_cast<int*>(sM);
        int* rowmap = colmap + SP;
        if (mode == kStageUpsample) {
            for (int t = tid; t < SP + SH; t += NT) {
                if (t < SP) {
                    const int gx = sx0 + t;
                    colmap[t] = (gx >= 0 && gx < p.width) ? upsample_site(gx, p.width, p.wl) : -1;
                } else {
                    const int gy = sy0 + (t - SP);
                    rowmap[t - SP] = (gy >= 0 && gy < p.height) ? upsample_site(gy, p.height, p.hl) : -1;
                }
            }
            __syncthreads();
        }
        for (int idx = tid; idx < SP * she; idx += NT) {
            int sy = idx / SP, sx = idx - sy * SP;
            int gx = sx0 + sx, gy = sy0 + sy;
            bool in = (gx >= 0) & (gx < p.width) & (gy >= 0) & (gy < p.height);
            float d = 0.f;
            uint32_t g = 0u;
            if (in) {
                g = __ldg(gsrc + (long long)gy * p.guide_pitch + gx);
                if (mode == kStagePlain) {
                    if constexpr (std::is_same<DT, uint16_t>::value) {
                        d = load_depth<DT>(dsrc, (long long)gy * p.width + gx);
                    } else {
                        const float* row = dsrc + (long long)gy * p.width;
                        if (p.depth_up != nullptr && gy < p.band0) row = p.depth_up + (long long)gy * p.width;
                        else if (p.depth_dn != nullptr && gy >= p.band1) row = p.depth_dn + (long long)(gy - p.band1) * p.width;
                        d = load_depth<float>(row, gx);
                    }
                } else {  // scatter the low-res sample onto its high-res site
                    const int xl = colmap[sx], yl = rowmap[sy];
                    if ((xl >= 0) & (yl >= 0)) d = upsample_sample(p, frame, xl, yl);
                }
            }
            sD[idx] = d;
            sG[idx] = g;
        }
    }
    if (mode == kStageTma) mbar_wait(bar, 0);
    __syncthreads();
    if constexpr (std::is_same<DT, uint16_t>::value) {
        // a pass of its own: stage B writes sM[idx] in the loop that would read the uint16 tile from it
        if (mode == kStageTma) {
            const uint16_t* s16 = reinterpret_cast<const uint16_t*>(sM) + (T::RP16 - RP);
            for (int idx = tid; idx < SP * she; idx += NT) {
                const int sy = idx / SP, sx = idx - sy * SP;
                sD[idx] = (float)s16[sy * T::SP16 + sx];
            }
            __syncthreads();
        }
    }

    // ---------------- stage B: validity word per staged sample; holes (and NaN) read as depth 0.  The range of the
    // valid staged depths decides (CTA-uniformly) whether pass 2 needs the skip-if-zero compare at all.
    float lmin = 3.0e38f, lmax = -3.0e38f;
    for (int idx = tid; idx < SP * she; idx += NT) {
        const float d = sD[idx];
        const bool v = d > kValidDepth;
        sD[idx] = v ? d : 0.f;
        sM[idx] = v ? kMagicValid : kMagicInvalid;
        lmin = v ? fminf(lmin, d) : lmin;
        lmax = v ? fmaxf(lmax, d) : lmax;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lmin = fminf(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
        lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    }
    if ((tid & 31) == 0) { sRed[2 * (tid >> 5)] = lmin; sRed[2 * (tid >> 5) + 1] = lmax; }
    __syncthreads();
    float tmin = 3.0e38f, tmax = -3.0e38f;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) { tmin = fminf(tmin, sRed[2 * w]); tmax = fmaxf(tmax, sRed[2 * w + 1]); }
    // every tap's |d - mean| is below the tile's depth range (means lie between the window's samples): if that range,
    // in the scaled units of pass 2 and with a margin for its roundings, stays below the fp32 expf() cut-off, no tap
    // of this tile can have its range factor skipped
    // (worth its code only for the larger windows: measured +2-3 % for r >= 6 on 3840x2160 frames, a loss below)
    const bool guard_free = (R >= 6) && !((tmax - tmin) * p.sq >= p.e_thr * 0.999f);

    // ---------------- compute: 4 pixels per thread
    const int lx = tid % (TW / 4), ly = tid / (TW / 4);
    if (ly >= th_eff) return;   // short tile: whole warps leave (th_eff is even, a tile row is 16 threads)
    const int colbase = 4 * lx;  // staged column of the fetched segment's first word
    uint32_t gp[4];
    float d0 = 0.f;
    {
        const int c = (ly + R) * SP + RP + colbase;
        const uint4 g4 = *reinterpret_cast<const uint4*>(sG + c);
        const float4 d4 = *reinterpret_cast<const float4*>(sD + c);
        const uint4 m4 = *reinterpret_cast<const uint4*>(sM + c);
        gp[0] = g4.x; gp[1] = g4.y; gp[2] = g4.z; gp[3] = g4.w;
        // per-thread accumulation origin (raw millimetres): first valid own pixel, else the first valid
        // sample of the thread's windows (own row first, then top to bottom) -- a function of the image
        // around the thread only, so results do not depend on the tile a pixel falls in
        bool has = true;
        d0 = (m4.x == kMagicValid) ? d4.x
           : (m4.y == kMagicValid) ? d4.y
           : (m4.z == kMagicValid) ? d4.z
           : (m4.w == kMagicValid) ? d4.w : (has = false, 0.f);
        if (!has) {
            // 16-byte reads of the validity plane, as the sweeps below do; the first valid column of the row
            // segment [C0, C0 + WS + 3) wins
#pragma unroll 1
            for (int rr = 0; rr <= WS && !has; ++rr) {
                const int rowoff = ((rr == 0) ? (ly + R) : (ly + rr - 1)) * SP + colbase;
                int first = NW;
#pragma unroll
                for (int v = NW / 4 - 1; v >= 0; --v) {
                    const uint4 q4 = *reinterpret_cast<const uint4*>(sM + rowoff + 4 * v);
                    if (4 * v + 3 >= C0 && 4 * v + 3 < C0 + WS + 3 && q4.w == kMagicValid) first = 4 * v + 3;
                    if (4 * v + 2 >= C0 && 4 * v + 2 < C0 + WS + 3 && q4.z == kMagicValid) first = 4 * v + 2;
                    if (4 * v + 1 >= C0 && 4 * v + 1 < C0 + WS + 3 && q4.y == kMagicValid) first = 4 * v + 1;
                    if (4 * v + 0 >= C0 && 4 * v + 0 < C0 + WS + 3 && q4.x == kMagicValid) first = 4 * v + 0;
                }
                if (first < NW) { d0 = sD[rowoff + first]; has = true; }
            }
        }
    }
    // scaled units: X = d*sq - cO with cO = fl(d0*sq); fma(d, sq, -cO) rounds once, relative to the
    // (small) difference; c_err = d0*sq - cO exactly, restored in the epilogue
    const float sq = p.sq;
    const float cO = __fmul_rn(d0, sq);
    const float c_err = fmaf(d0, sq, -cO);
    const float ncO = -cO;
    const float nkc = p.nkc;
    float delta[4], num[4], den[4], wsum[4];
    bool any[4];

    // Pixels (0,1) and (2,3) of the thread share one tap column, so the FADD/FFMA of two taps issue as one
    // FADD2/FFMA2 (scalar operands broadcast, LUT entries pre-paired as {L[j], L[j-1]}).  Per tap PAIR:
    // 2 VABSDIFF4 + 2 IDP.4A + FADD2 + FFMA2 + 2 MUFU.EX2 + FFMA2 + FADD2 (pass 1), plus FADD2 + 2 FSETP +
    // 2 predicated FFMA (pass 2).
    const f32x2 kNeg23 = pack2(-8388608.0f, -8388608.0f);
    const f32x2 nkc2 = pack2(nkc, nkc);

#define KDME_LOAD_ROW(SL)                                                                              \
    const int rowoff = (ly + i) * SP + colbase;                                                        \
    uint32_t gq[NW], mq[NW];                                                                           \
    float dq[NW];                                                                                      \
    f32x2 LPr[LPP];                                                                                    \
    _Pragma("unroll") for (int v = 0; v < NW / 4; ++v) {                                               \
        const uint4 g4 = *reinterpret_cast<const uint4*>(sG + rowoff + 4 * v);                         \
        const float4 d4 = *reinterpret_cast<const float4*>(sD + rowoff + 4 * v);                       \
        const uint4 m4 = *reinterpret_cast<const uint4*>(sM + rowoff + 4 * v);                         \
        gq[4 * v] = g4.x; gq[4 * v + 1] = g4.y; gq[4 * v + 2] = g4.z; gq[4 * v + 3] = g4.w;            \
        dq[4 * v] = d4.x; dq[4 * v + 1] = d4.y; dq[4 * v + 2] = d4.z; dq[4 * v + 3] = d4.w;            \
        mq[4 * v] = m4.x; mq[4 * v + 1] = m4.y; mq[4 * v + 2] = m4.z; mq[4 * v + 3] = m4.w;            \
    }                                                                                                  \
    _Pragma("unroll") for (int v = 0; v < LPP / 2; ++v) {                                              \
        const float4 l4 = *reinterpret_cast<const float4*>(SL + (i * LPP + 2 * v) * 2);                \
        LPr[2 * v] = pack2(l4.x, l4.y);                                                                \
        LPr[2 * v + 1] = pack2(l4.z, l4.w);                                                            \
    }

    // ---------------- pass 1: spatial x colour weighted mean (JointBilateralFilter.cu:16-40)
    {
        f32x2 accP[2] = {0ull, 0ull}, wsP[2] = {0ull, 0ull};
        f32x2 accL[2] = {0ull, 0ull}, wsL[2] = {0ull, 0ull};   // 2Sum low words of the window sums
        f32x2 gaccP[2] = {0ull, 0ull}, gwsP[2] = {0ull, 0ull}; // sums of the current group of rows
#pragma unroll 1
        for (int i = 0; i < WS; ++i) {
            KDME_LOAD_ROW(sL1)
            // per-row partial sums, combined below without rounding error
            f32x2 raccP[2] = {0ull, 0ull}, rwsP[2] = {0ull, 0ull};
#pragma unroll
            for (int c = C0; c < C0 + WS + 3; ++c) {
                const float dsh = fmaf(dq[c], sq, ncO);
                const f32x2 dsh2 = pack2(dsh, dsh);
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                    if (PSEL != 0 && pr != PSEL - 1) continue;   /* compile time */
                    const int j0 = c - C0 - 2 * pr;   // tap column index of the pair's first pixel; second uses j0-1
                    const bool v0 = (j0 >= 0 && j0 < WS), v1 = (j0 - 1 >= 0 && j0 - 1 < WS);
                    if (v0 && v1) {
                        const uint32_t ad0 = __vabsdiffu4(gp[2 * pr], gq[c]), ad1 = __vabsdiffu4(gp[2 * pr + 1], gq[c]);
                        const f32x2 xx = pack2(__uint_as_float(__dp4a(ad0, ad0, mq[c])),
                                               __uint_as_float(__dp4a(ad1, ad1, mq[c])));
                        const f32x2 ar = fma2(add2(xx, kNeg23), nkc2, LPr[j0 - 1]);
                        float a0, a1;
                        unpack2(ar, a0, a1);
                        const f32x2 ff = pack2(ex2_approx(a0), ex2_approx(a1));
                        raccP[pr] = fma2(ff, dsh2, raccP[pr]);
                        rwsP[pr] = add2(rwsP[pr], ff);
                    } else if (v0 || v1) {   // window edge: only one pixel of the pair sees this column
                        const int k = v0 ? 2 * pr : 2 * pr + 1;
                        const int j = v0 ? j0 : j0 - 1;
                        float l_lo, l_hi;
                        unpack2(LPr[(j == 0) ? 0 : j - 1], l_lo, l_hi);   // L[0] = pair 0 hi, L[j] = pair j-1 lo
                        const float lj = (j == 0) ? l_hi : l_lo;
                        const uint32_t ad = __vabsdiffu4(gp[k], gq[c]);
                        const float cdf = __uint_as_float(__dp4a(ad, ad, mq[c])) - 8388608.0f;
                        const float f = ex2_approx(fmaf(cdf, nkc, lj));
                        const f32x2 ff = v0 ? pack2(f, 0.f) : pack2(0.f, f);
                        raccP[pr] = fma2(ff, dsh2, raccP[pr]);
                        rwsP[pr] = add2(rwsP[pr], ff);
                    }
                }
            }
            // row sums -> sums of a group of kRowsPer2Sum rows (plain adds: a fraction of the window's magnitude)
            // -> window sums (2Sum, error-free)
#pragma unroll
            for (int pr = 0; pr < 2; ++pr) {
                    if (PSEL != 0 && pr != PSEL - 1) continue;   /* compile time */ gaccP[pr] = add2(gaccP[pr], raccP[pr]); gwsP[pr] = add2(gwsP[pr], rwsP[pr]); }
            if ((i % kRowsPer2Sum) == kRowsPer2Sum - 1 || i == WS - 1) {
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                    if (PSEL != 0 && pr != PSEL - 1) continue;   /* compile time */
                    two_sum2(accP[pr], gaccP[pr], accL[pr]);
                    two_sum2(wsP[pr], gwsP[pr], wsL[pr]);
                    gaccP[pr] = 0ull; gwsP[pr] = 0ull;
                }
            }
        }
        float acc[4], accl[4], wsl[4];
        unpack2(accP[0], acc[0], acc[1]); unpack2(accP[1], acc[2], acc[3]);
        unpack2(wsP[0], wsum[0], wsum[1]); unpack2(wsP[1], wsum[2], wsum[3]);
        unpack2(accL[0], accl[0], accl[1]); unpack2(accL[1], accl[2], accl[3]);
        unpack2(wsL[0], wsl[0], wsl[1]); unpack2(wsL[1], wsl[2], wsl[3]);
        // pass-1 weighted mean in scaled units relative to cO: (acc + accl) / (wsum + wsl), correctly
        // rounded quotient of the compensated sums (one Newton-style residual step)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            any[k] = wsum[k] > 0.f;
            const float dh = acc[k] / wsum[k];
            float res = fmaf(-dh, wsum[k], acc[k]);
            res += accl[k];
            res = fmaf(-dh, wsl[k], res);
            delta[k] = any[k] ? (dh + res / wsum[k]) : 0.f;
        }
    }

    // ---------------- pass 2: range term centred on the pass-1 mean (JointBilateralFilter.cu:43-73)
    if (guard_free) {
        // No range factor can underflow in this tile: no compare, no predication.  Evaluated with flipped signs so
        // that every operation packs: en = delta - dsh = -e, A = fma2(en, en, -(arg)) = -(arg - e^2) (rounding is
        // symmetric: the same bits as fmaf(-e, e, arg)), f = 2^(-A), num' = sum f en = -num.
        const f32x2 delP[2] = {pack2(delta[0], delta[1]), pack2(delta[2], delta[3])};
        const f32x2 kPos23 = pack2(8388608.0f, 8388608.0f);
        f32x2 numP[2] = {0ull, 0ull}, denP[2] = {0ull, 0ull};
#pragma unroll 1
        for (int i = 0; i < WS; ++i) {
            KDME_LOAD_ROW(sL2)
            f32x2 rnumP[2] = {0ull, 0ull}, rdenP[2] = {0ull, 0ull};
#pragma unroll
            for (int c = C0; c < C0 + WS + 3; ++c) {
                const float dsh = fmaf(dq[c], sq, ncO);
                const f32x2 ndsh2 = pack2(-dsh, -dsh);
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                    if (PSEL != 0 && pr != PSEL - 1) continue;   /* compile time */
                    const int j0 = c - C0 - 2 * pr;
                    const bool v0 = (j0 >= 0 && j0 < WS), v1 = (j0 - 1 >= 0 && j0 - 1 < WS);
                    if (v0 && v1) {
                        const uint32_t ad0 = __vabsdiffu4(gp[2 * pr], gq[c]), ad1 = __vabsdiffu4(gp[2 * pr + 1], gq[c]);
                        const f32x2 xx = pack2(__uint_as_float(__dp4a(ad0, ad0, mq[c])),
                                               __uint_as_float(__dp4a(ad1, ad1, mq[c])));
                        // -(arg): (2^23 - x) * nkc - L == -((x - 2^23) * nkc + L) exactly (sign symmetry of every rounding)
                        const f32x2 nar = fma2(sub2(kPos23, xx), nkc2, neg2(LPr[j0 - 1]));
                        const f32x2 en = add2(ndsh2, delP[pr]);
                        const f32x2 A = fma2(en, en, nar);
                        float a0, a1;
                        unpack2(A, a0, a1);
                        const f32x2 ff = pack2(ex2_approx(-a0), ex2_approx(-a1));
                        rnumP[pr] = fma2(ff, en, rnumP[pr]);
                        rdenP[pr] = add2(rdenP[pr], ff);
                    } else if (v0 || v1) {
                        const int k = v0 ? 2 * pr : 2 * pr + 1;
                        const int j = v0 ? j0 : j0 - 1;
                        float l_lo, l_hi;
                        unpack2(LPr[(j == 0) ? 0 : j - 1], l_lo, l_hi);
                        const float lj = (j == 0) ? l_hi : l_lo;
                        const uint32_t ad = __vabsdiffu4(gp[k], gq[c]);
                        const float cdf = __uint_as_float(__dp4a(ad, ad, mq[c])) - 8388608.0f;
                        const float e = dsh - delta[k];
                        const float f = ex2_approx(fmaf(-e, e, fmaf(cdf, nkc, lj)));
                        const f32x2 ff = v0 ? pack2(f, 0.f) : pack2(0.f, f);
                        const f32x2 en = v0 ? pack2(-e, 0.f) : pack2(0.f, -e);
                        rnumP[pr] = fma2(ff, en, rnumP[pr]);
                        rdenP[pr] = add2(rdenP[pr], ff);
                    }
                }
            }
#pragma unroll
            for (int pr = 0; pr < 2; ++pr) {
                    if (PSEL != 0 && pr != PSEL - 1) continue;   /* compile time */ numP[pr] = add2(numP[pr], rnumP[pr]); denP[pr] = add2(denP[pr], rdenP[pr]); }
        }
        unpack2(numP[0], num[0], num[1]); unpack2(numP[1], num[2], num[3]);
        unpack2(denP[0], den[0], den[1]); unpack2(denP[1], den[2], den[3]);
#pragma unroll
        for (int k = 0; k < 4; ++k) num[k] = -num[k];
    } else
    {
        const f32x2 ndelP[2] = {pack2(-delta[0], -delta[1]), pack2(-delta[2], -delta[3])};
        const float e_thr = p.e_thr;
        f32x2 numP[2] = {0ull, 0ull}, denP[2] = {0ull, 0ull};
#pragma unroll 1
        for (int i = 0; i < WS; ++i) {
            KDME_LOAD_ROW(sL2)
            f32x2 rnumP[2] = {0ull, 0ull}, rdenP[2] = {0ull, 0ull};
#pragma unroll
            for (int c = C0; c < C0 + WS + 3; ++c) {
                const float dsh = fmaf(dq[c], sq, ncO);
                const f32x2 dsh2 = pack2(dsh, dsh);
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                    if (PSEL != 0 && pr != PSEL - 1) continue;   /* compile time */
                    const int j0 = c - C0 - 2 * pr;
                    const bool v0 = (j0 >= 0 && j0 < WS), v1 = (j0 - 1 >= 0 && j0 - 1 < WS);
                    if (v0 && v1) {
                        const uint32_t ad0 = __vabsdiffu4(gp[2 * pr], gq[c]), ad1 = __vabsdiffu4(gp[2 * pr + 1], gq[c]);
                        const f32x2 xx = pack2(__uint_as_float(__dp4a(ad0, ad0, mq[c])),
                                               __uint_as_float(__dp4a(ad1, ad1, mq[c])));
                        const f32x2 ar = fma2(add2(xx, kNeg23), nkc2, LPr[j0 - 1]);
                        const f32x2 ee = add2(dsh2, ndelP[pr]);
                        float a0, a1, e0, e1;
                        unpack2(ar, a0, a1);
                        unpack2(ee, e0, e1);
                        // fp32 expf(-(d-m)^2/(2 sd^2)) == 0  <=>  factor skipped (.cu:67-68)
                        if (!(fabsf(e0) > e_thr)) a0 = fmaf(-e0, e0, a0);
                        if (!(fabsf(e1) > e_thr)) a1 = fmaf(-e1, e1, a1);
                        const f32x2 ff = pack2(ex2_approx(a0), ex2_approx(a1));
                        rnumP[pr] = fma2(ff, ee, rnumP[pr]);
                        rdenP[pr] = add2(rdenP[pr], ff);
                    } else if (v0 || v1) {
                        const int k = v0 ? 2 * pr : 2 * pr + 1;
                        const int j = v0 ? j0 : j0 - 1;
                        float l_lo, l_hi;
                        unpack2(LPr[(j == 0) ? 0 : j - 1], l_lo, l_hi);
                        const float lj = (j == 0) ? l_hi : l_lo;
                        const uint32_t ad = __vabsdiffu4(gp[k], gq[c]);
                        const float cdf = __uint_as_float(__dp4a(ad, ad, mq[c])) - 8388608.0f;
                        float arg = fmaf(cdf, nkc, lj);
                        const float e = dsh - delta[k];
                        if (!(fabsf(e) > e_thr)) arg = fmaf(-e, e, arg);
                        const float f = ex2_approx(arg);
                        const f32x2 ff = v0 ? pack2(f, 0.f) : pack2(0.f, f);
                        const f32x2 ee = v0 ? pack2(e, 0.f) : pack2(0.f, e);
                        rnumP[pr] = fma2(ff, ee, rnumP[pr]);
                        rdenP[pr] = add2(rdenP[pr], ff);
                    }
                }
            }
#pragma unroll
            for (int pr = 0; pr < 2; ++pr) {
                    if (PSEL != 0 && pr != PSEL - 1) continue;   /* compile time */ numP[pr] = add2(numP[pr], rnumP[pr]); denP[pr] = add2(denP[pr], rdenP[pr]); }
        }
        unpack2(numP[0], num[0], num[1]); unpack2(numP[1], num[2], num[3]);
        unpack2(denP[0], den[0], den[1]); unpack2(denP[1], den[2], den[3]);
    }
#undef KDME_LOAD_ROW

    // ---------------- epilogue: back to millimetres
    float o[4];
    bool flag[4];
    bool anyflag = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        // den > 0 whenever any tap is valid (pass-2 weights are biased into the normal range)
        const float t = (delta[k] + num[k] / den[k]) - c_err;
        o[k] = any[k] ? fmaf(t, p.inv_sq, d0) : 0.f;
        // den / wsum = mean range weight of the window.  When it is tiny, no sample lies near the pass-1
        // mean (a pixel between two surfaces): the output then amplifies the rounding of that mean by
        // (distance / sigma_d)^2, beyond what fp32 sums can absorb -> such pixels are re-evaluated in fp64.
        flag[k] = any[k] && !(den[k] >= wsum[k] * p.flag_scale);
        anyflag |= flag[k];
    }
    const int gy = y0 + ly, gx = x0 + 4 * lx;
    const int oy = gy - p.y_off;
    if (__any_sync(0xffffffffu, anyflag)) {
        // queue the flagged pixels of this warp (one atomic per warp)
        const int lane = tid & 31;
        unsigned m[4];
        int total = 0, before = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            m[k] = __ballot_sync(0xffffffffu, flag[k] && oy < p.out_rows && gx + k < p.width);
            before += __popc(m[k] & ((1u << lane) - 1u));
            total += __popc(m[k]);
        }
        unsigned base = 0;
        if (lane == 0 && total > 0) base = atomicAdd(p.q_count, (unsigned)total);
        base = __shfl_sync(0xffffffffu, base, 0);
        // slots: lane-major (all flagged pixels of lane 0, then lane 1, ...)
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if ((m[k] >> lane) & 1u) {
                const unsigned slot = base + (unsigned)before;
                ++before;
                if (slot < p.q_capacity)
                    p.q_items[slot] = (unsigned)(((long long)frame * p.out_rows + oy) * p.width + gx + k);
            }
    }
    if (oy < p.out_rows && gx < p.width) {
        const long long pix = (long long)frame * p.width * p.out_rows + (long long)oy * p.width + gx;
        float* dst = p.out + pix;
        constexpr int K0 = (PSEL == 2) ? 2 : 0, K1 = (PSEL == 1) ? 2 : 4;   // the pixels this instantiation owns
        if (PSEL == 0 && gx + 3 < p.width && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
            stg_stream_f4(reinterpret_cast<float4*>(dst), make_float4(o[0], o[1], o[2], o[3]));
        } else {
#pragma unroll
            for (int k = K0; k < K1; ++k)
                if (gx + k < p.width) dst[k] = o[k];
        }
        if (p.xyz != nullptr) {
            // DimensionConvertor::projectiveToReal (DimensionConvertor.h:34-48): x = (u - cx)/fx * z,
            // y = (cy - v)/fy * z, IEEE division and un-fused ops in the reference functor's order
            float v3[12];
            const float py = __fdiv_rn(__fsub_rn((float)p.cy, (float)(p.y_img0 + gy)), p.fy);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float px = __fdiv_rn(__fsub_rn((float)(gx + k), (float)p.cx), p.fx);
                v3[3 * k + 0] = __fmul_rn(px, o[k]);
                v3[3 * k + 1] = __fmul_rn(py, o[k]);
                v3[3 * k + 2] = o[k];
            }
            float* xdst = p.xyz + 3 * pix;
            if (PSEL == 0 && gx + 3 < p.width && ((reinterpret_cast<uintptr_t>(xdst) & 15) == 0)) {
#pragma unroll
                for (int q = 0; q < 3; ++q)
                    stg_stream_f4(reinterpret_cast<float4*>(xdst) + q,
                                  make_float4(v3[4 * q], v3[4 * q + 1], v3[4 * q + 2], v3[4 * q + 3]));
            } else {
#pragma unroll
                for (int k = K0; k < K1; ++k)
                    if (gx + k < p.width) { xdst[3 * k] = v3[3 * k]; xdst[3 * k + 1] = v3[3 * k + 1]; xdst[3 * k + 2] = v3[3 * k + 2]; }
            }
        }
    }
}

template <int R, int TW, int TH, int MINB, class DT>
__global__ void __launch_bounds__((TW / 4) * TH, MINB)
jbf_fast_kernel(const __grid_constant__ CUtensorMap tm_depth, const __grid_constant__ CUtensorMap tm_guide,
                const JbfParams p) {
    // CTA-uniform dispatch: whole tiles and whole small tiles run the full body, half units one pair each.  The 64x16
    // instantiations (large launches) carry the full body only: the hot kernel's code is exactly the single-body one.
    if constexpr (TH >= 16) {
        jbf_fast_body<R, TW, TH, 0, DT>(tm_depth, tm_guide, p);
    } else {
        if (!p.half_units || (int)blockIdx.y < p.nbig_rows) jbf_fast_body<R, TW, TH, 0, DT>(tm_depth, tm_guide, p);
        else if ((((int)blockIdx.y - p.nbig_rows) & 1) == 0) jbf_fast_body<R, TW, TH, 1, DT>(tm_depth, tm_guide, p);
        else jbf_fast_body<R, TW, TH, 2, DT>(tm_depth, tm_guide, p);
    }
}

// -----------------------------------------------------------------------------
// Upsampling in gather form (SURVEY.md 8(d) config 3; declared only in the reference,
// JointBilateralFilter.h:14).  The sparse high-res depth image is never materialised: a low-res sample
// (xl, yl) lives at high-res site (floor((2 xl + 1) W / (2 wl)), floor((2 yl + 1) H / (2 hl))), and a
// pixel's window only meets the ~(2r+1)^2 wl hl / (W H) sites of that lattice.  One CTA stages the sites
// its tile can see (low-res depth + the smoothed guide AT the site); each thread owns 4 adjacent pixels and
// sweeps site rows x site columns.  The arithmetic per pixel is the dense kernel's, tap for tap and in the
// same order (taps that are not sites have weight exactly 0 there and add nothing), so the result equals
// jbf_fast_kernel on the materialised sparse image BIT FOR BIT -- including the accumulation origin rule,
// the 2Sum row partials and the fp64 refinement queue.  Frames of a batch are blockIdx.z; every frame shares the
// lattice tables, and its low-res depth is read through upsample_sample (float or uint16).
// padding of a pair-table row of the gather kernel: entries for window columns -2 .. WS+4 (WS + 7 is even, so a
// table is a whole number of 16-byte words)
constexpr int kUpsPad = 7;

struct UpsampleGeom {
    int ncol_max, nrow_max;      // staged site columns / rows per tile (host-computed bound)
    int radius;
    const float* ltab1;          // padded pair table [(2r+1)][(2r+1) + kUpsPad][2], bias1 (pass 1); see the kernel
    const float* ltab2;          // same, bias kWeightBias (pass 2)
    // the lattice, tabulated once per (wl, hl) on the host (no 64-bit divisions in the kernel):
    const int* site_x;           // [wl] high-res x of low-res column xl
    const int* site_y;           // [hl]
    const int* tile_xl;          // [tiles_x][2] = first low-res column with site >= x0 - r, first with site > x0 + TW - 1 + r
    const int* tile_yl;          // [tiles_y][2]
};

// first low-res index whose site is >= x (wl when every site lies below x)
__host__ __device__ __forceinline__ int upsample_first_site_at_or_after(int x, int W, int wl) {
    if (x <= 0) return 0;
    long long num = 2LL * wl * x - W;                       // site(xl) >= x  <=>  (2xl+1) W >= 2 wl x  (floor is monotone)
    int xl = (num <= 0) ? 0 : (int)((num + 2LL * W - 1) / (2LL * W));
    while (xl > 0 && (int)(((2LL * (xl - 1) + 1) * W) / (2LL * wl)) >= x) --xl;
    while (xl < wl && (int)(((2LL * xl + 1) * W) / (2LL * wl)) < x) ++xl;
    return xl < wl ? xl : wl;   // wl: no such site
}

// One site seen by a thread's two pixel pairs, pass 1 / pass 2 (the dense kernel's packed tap, LUT pair from the
// padded table; lp points at pair 0's entry, pair 1's is two entries below)
__device__ __forceinline__ void gather_site_p1(const uint32_t (&gp)[4], float d, uint32_t gq, const float2* lp, float sq,
                                               float ncO, f32x2 nkc2, f32x2 (&raccP)[2], f32x2 (&rwsP)[2]) {
    const f32x2 kNeg23 = pack2(-8388608.0f, -8388608.0f);
    const uint32_t mq = (d != 0.f) ? kMagicValid : kMagicInvalid;
    const float dsh = fmaf(d, sq, ncO);
    const f32x2 dsh2 = pack2(dsh, dsh);
#pragma unroll
    for (int pr = 0; pr < 2; ++pr) {
        const float2 l2 = lp[-2 * pr];
        const uint32_t ad0 = __vabsdiffu4(gp[2 * pr], gq), ad1 = __vabsdiffu4(gp[2 * pr + 1], gq);
        const f32x2 xx = pack2(__uint_as_float(__dp4a(ad0, ad0, mq)), __uint_as_float(__dp4a(ad1, ad1, mq)));
        const f32x2 ar = fma2(add2(xx, kNeg23), nkc2, pack2(l2.x, l2.y));
        float a0, a1;
        unpack2(ar, a0, a1);
        const f32x2 ff = pack2(ex2_approx(a0), ex2_approx(a1));
        raccP[pr] = fma2(ff, dsh2, raccP[pr]);
        rwsP[pr] = add2(rwsP[pr], ff);
    }
}
__device__ __forceinline__ void gather_site_p2(const uint32_t (&gp)[4], float d, uint32_t gq, const float2* lp, float sq,
                                               float ncO, f32x2 nkc2, const f32x2 (&ndelP)[2], float e_thr,
                                               f32x2 (&rnumP)[2], f32x2 (&rdenP)[2]) {
    const f32x2 kNeg23 = pack2(-8388608.0f, -8388608.0f);
    const uint32_t mq = (d != 0.f) ? kMagicValid : kMagicInvalid;
    const float dsh = fmaf(d, sq, ncO);
    const f32x2 dsh2 = pack2(dsh, dsh);
#pragma unroll
    for (int pr = 0; pr < 2; ++pr) {
        const float2 l2 = lp[-2 * pr];
        const uint32_t ad0 = __vabsdiffu4(gp[2 * pr], gq), ad1 = __vabsdiffu4(gp[2 * pr + 1], gq);
        const f32x2 xx = pack2(__uint_as_float(__dp4a(ad0, ad0, mq)), __uint_as_float(__dp4a(ad1, ad1, mq)));
        const f32x2 ar = fma2(add2(xx, kNeg23), nkc2, pack2(l2.x, l2.y));
        const f32x2 ee = add2(dsh2, ndelP[pr]);
        float a0, a1, e0, e1;
        unpack2(ar, a0, a1);
        unpack2(ee, e0, e1);
        if (!(fabsf(e0) > e_thr)) a0 = fmaf(-e0, e0, a0);
        if (!(fabsf(e1) > e_thr)) a1 = fmaf(-e1, e1, a1);
        const f32x2 ff = pack2(ex2_approx(a0), ex2_approx(a1));
        rnumP[pr] = fma2(ff, ee, rnumP[pr]);
        rdenP[pr] = add2(rdenP[pr], ff);
    }
}

// MAXC > 0: no thread sees more than MAXC site columns (host-computed: ceil((2r+4) wl / W)); the columns are then
// resolved once per thread into registers and every site row is a straight-line body of MAXC sites (a missing
// column reads a staged site with an out-of-window table entry: weight exactly 0).  MAXC == 0: runtime column loop.
template <int TW, int TH, int MAXC>
__global__ void __launch_bounds__((TW / 4) * TH, 3)
jbf_upsample_gather_kernel(const JbfParams p, const UpsampleGeom g) {
    constexpr int NT = (TW / 4) * TH;
    const int R = g.radius, WS = 2 * R + 1;
    // pair tables, one row per window row: entry e = jj + 2 holds {Lx[jj], Lx[jj-1]} for jj = -2 .. WS+4, where
    // Lx[j] = log2 spatial weight for 0 <= j < WS and -3e38 outside the window (2^(-3e38 + ...) == 0 exactly under
    // ex2.approx.ftz): a lane whose column falls outside the window gets weight 0 from the table itself, so the tap
    // needs neither a clamp nor a predicate.  Built once per handle on the host (kUpsPad), copied here 16 bytes at a time.
    const int LPW = WS + kUpsPad;
    extern __shared__ __align__(16) uint8_t smem_up[];
    float* sL1 = reinterpret_cast<float*>(smem_up);                      // [WS][LPW][2], WS * LPW * 2 is a multiple of 4
    float* sL2 = sL1 + WS * LPW * 2;
    float* sSd = sL2 + WS * LPW * 2;                                     // [nrow_max][ncol_max] sample depth (0 = hole)
    uint32_t* sSg = reinterpret_cast<uint32_t*>(sSd + g.nrow_max * g.ncol_max);   // guide word at the site
    int* sXs = reinterpret_cast<int*>(sSg + g.nrow_max * g.ncol_max);    // [ncol_max] site x
    int* sYs = sXs + g.ncol_max;                                         // [nrow_max] site y

    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH, frame = blockIdx.z;
    const uint32_t* gsrc = p.guide4 + (long long)frame * p.guide_frame_stride;
    const long long fpix = (long long)frame * p.width * p.out_rows;   // first output pixel of the frame
    for (int idx = tid; idx < WS * LPW / 2; idx += NT) {
        reinterpret_cast<float4*>(sL1)[idx] = __ldg(reinterpret_cast<const float4*>(g.ltab1) + idx);
        reinterpret_cast<float4*>(sL2)[idx] = __ldg(reinterpret_cast<const float4*>(g.ltab2) + idx);
    }
    grid_dependency_wait();
    if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) *p.q_count_prev = 0u;
    // site columns with x in [x0 - R, x0 + TW - 1 + R], site rows with y in [y0 - R, y0 + TH - 1 + R]
    const int xl0 = __ldg(g.tile_xl + 2 * blockIdx.x), yl0 = __ldg(g.tile_yl + 2 * blockIdx.y);
    const int ncol = min(__ldg(g.tile_xl + 2 * blockIdx.x + 1) - xl0, g.ncol_max);
    const int nrow = min(__ldg(g.tile_yl + 2 * blockIdx.y + 1) - yl0, g.nrow_max);
    for (int t = tid; t < ncol + nrow; t += NT) {
        if (t < ncol) sXs[t] = __ldg(g.site_x + xl0 + t);
        else sYs[t - ncol] = __ldg(g.site_y + yl0 + (t - ncol));
    }
    __syncthreads();
    for (int idx = tid; idx < ncol * nrow; idx += NT) {
        const int sr = idx / ncol, sc = idx - sr * ncol;
        const float d = upsample_sample(p, frame, xl0 + sc, yl0 + sr);
        sSd[sr * g.ncol_max + sc] = (d > kValidDepth) ? d : 0.f;
        sSg[sr * g.ncol_max + sc] = __ldg(gsrc + (long long)sYs[sr] * p.guide_pitch + sXs[sc]);
    }
    __syncthreads();

    const int lx = tid % (TW / 4), ly = tid / (TW / 4);
    const int gy = y0 + ly, gx = x0 + 4 * lx;
    uint32_t gp[4] = {0u, 0u, 0u, 0u};
    if (gy < p.height) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (gx + k < p.width) gp[k] = __ldg(gsrc + (long long)gy * p.guide_pitch + gx + k);
    }
    // this thread's site rows [r_lo, r_hi) and site columns [c_lo, c_hi) (union over its 4 pixels)
    // (the lattice is near-uniform: start from the proportional guess and correct by a step or two instead of
    // scanning the staged lists from their first entry)
    int r_lo = 0, r_hi = 0, c_lo = 0, c_hi = 0;
    if (nrow > 0) r_lo = min(max((int)floorf((float)(gy - R - sYs[0]) * ((float)p.hl / (float)p.height)), 0), nrow);
    if (ncol > 0) c_lo = min(max((int)floorf((float)(gx - R - sXs[0]) * ((float)p.wl / (float)p.width)), 0), ncol);
    while (r_lo > 0 && sYs[r_lo - 1] >= gy - R) --r_lo;
    while (r_lo < nrow && sYs[r_lo] < gy - R) ++r_lo;
    r_hi = r_lo;
    while (r_hi < nrow && sYs[r_hi] <= gy + R) ++r_hi;
    while (c_lo > 0 && sXs[c_lo - 1] >= gx - R) --c_lo;
    while (c_lo < ncol && sXs[c_lo] < gx - R) ++c_lo;
    c_hi = c_lo;
    while (c_hi < ncol && sXs[c_hi] <= gx + 3 + R) ++c_hi;

    // accumulation origin, the dense kernel's rule: first valid own pixel, else the first valid sample of the
    // thread's windows -- own row first, then top to bottom, columns ascending
    float d0 = 0.f;
    {
        bool has = false;
        int own = -1;
        for (int sr = r_lo; sr < r_hi; ++sr) if (sYs[sr] == gy) own = sr;
        if (own >= 0)
            for (int sc = c_lo; sc < c_hi && !has; ++sc)
                if (sXs[sc] >= gx && sXs[sc] <= gx + 3 && sSd[own * g.ncol_max + sc] != 0.f) { d0 = sSd[own * g.ncol_max + sc]; has = true; }
        if (!has && own >= 0)
            for (int sc = c_lo; sc < c_hi && !has; ++sc)
                if (sSd[own * g.ncol_max + sc] != 0.f) { d0 = sSd[own * g.ncol_max + sc]; has = true; }
        for (int sr = r_lo; sr < r_hi && !has; ++sr)
            for (int sc = c_lo; sc < c_hi && !has; ++sc)
                if (sSd[sr * g.ncol_max + sc] != 0.f) { d0 = sSd[sr * g.ncol_max + sc]; has = true; }
    }
    const float sq = p.sq;
    const float cO = __fmul_rn(d0, sq);
    const float c_err = fmaf(d0, sq, -cO);
    const float ncO = -cO;
    const float nkc = p.nkc;

    // Branch-free taps in the dense kernel's packed form: pixels (0,1) and (2,3) share a site, lane 0 of a pair
    // sees it at window column j0 and lane 1 at j0 - 1.  A lane whose column falls outside the window reads -3e38
    // from the padded table, a site that is a hole carries the invalid magic in the IDP.4A accumulator (as in the
    // dense kernel): either way the weight is exactly 0 and adds nothing -- the sums are the dense kernel's, bit for bit.
    const f32x2 nkc2 = pack2(nkc, nkc);
    const int ncm = g.ncol_max;
    const int jofs = R + 2 - gx;              // table entry of pair 0 for a site at x: x + jofs; pair 1: two less
    // the thread's site columns, resolved once: staged column and table entry (a missing column: any staged
    // column -- its data is finite -- with the all-out-of-window entry WS + 5, whose pair-1 partner WS + 3 is too)
    int scol[MAXC > 0 ? MAXC : 1], eoff[MAXC > 0 ? MAXC : 1];
    if constexpr (MAXC > 0) {
        if (ncol == 0) r_hi = r_lo;           // no staged site at all: nothing to sweep
#pragma unroll
        for (int c = 0; c < MAXC; ++c) {
            const int sc = c_lo + c;
            const bool ok = sc < c_hi;
            scol[c] = ok ? sc : min(c_lo, max(ncol - 1, 0));
            eoff[c] = ok ? sXs[ok ? sc : 0] + jofs : WS + 5;   // entries WS + 5 and WS + 3: all four columns outside
        }
    }
    float wsum[4], delta[4];
    bool any[4];
    {
        f32x2 accP[2] = {0ull, 0ull}, wsP[2] = {0ull, 0ull}, accL[2] = {0ull, 0ull}, wsL[2] = {0ull, 0ull};
        f32x2 gaccP[2] = {0ull, 0ull}, gwsP[2] = {0ull, 0ull};
        for (int sr = r_lo; sr < r_hi; ++sr) {
            const int wrow = sYs[sr] - gy + R;
            const float2* lrow = reinterpret_cast<const float2*>(sL1) + wrow * LPW;
            const float* drow = sSd + sr * ncm;
            const uint32_t* grow = sSg + sr * ncm;
            f32x2 raccP[2] = {0ull, 0ull}, rwsP[2] = {0ull, 0ull};
            if constexpr (MAXC > 0) {
#pragma unroll
                for (int c = 0; c < MAXC; ++c)
                    gather_site_p1(gp, drow[scol[c]], grow[scol[c]], lrow + eoff[c], sq, ncO, nkc2, raccP, rwsP);
            } else {
#pragma unroll 2
                for (int sc = c_lo; sc < c_hi; ++sc)
                    gather_site_p1(gp, drow[sc], grow[sc], lrow + sXs[sc] + jofs, sq, ncO, nkc2, raccP, rwsP);
            }
            // the dense kernel's grouping: rows of the same group of kRowsPer2Sum window rows are added plainly,
            // group sums are combined with 2Sum (groups without sites add nothing either way)
#pragma unroll
            for (int pr = 0; pr < 2; ++pr) { gaccP[pr] = add2(gaccP[pr], raccP[pr]); gwsP[pr] = add2(gwsP[pr], rwsP[pr]); }
            const int grp = wrow / kRowsPer2Sum;
            const int grp_next = (sr + 1 < r_hi) ? (sYs[sr + 1] - gy + R) / kRowsPer2Sum : -1;
            if (grp_next != grp) {
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                    two_sum2(accP[pr], gaccP[pr], accL[pr]);
                    two_sum2(wsP[pr], gwsP[pr], wsL[pr]);
                    gaccP[pr] = 0ull; gwsP[pr] = 0ull;
                }
            }
        }
        float acc[4], accl[4], wsl[4];
        unpack2(accP[0], acc[0], acc[1]); unpack2(accP[1], acc[2], acc[3]);
        unpack2(wsP[0], wsum[0], wsum[1]); unpack2(wsP[1], wsum[2], wsum[3]);
        unpack2(accL[0], accl[0], accl[1]); unpack2(accL[1], accl[2], accl[3]);
        unpack2(wsL[0], wsl[0], wsl[1]); unpack2(wsL[1], wsl[2], wsl[3]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            any[k] = wsum[k] > 0.f;
            const float dh = acc[k] / wsum[k];
            float res = fmaf(-dh, wsum[k], acc[k]);
            res += accl[k];
            res = fmaf(-dh, wsl[k], res);
            delta[k] = any[k] ? (dh + res / wsum[k]) : 0.f;
        }
    }
    float num[4], den[4];
    {
        const f32x2 ndelP[2] = {pack2(-delta[0], -delta[1]), pack2(-delta[2], -delta[3])};
        const float e_thr = p.e_thr;
        f32x2 numP[2] = {0ull, 0ull}, denP[2] = {0ull, 0ull};
        for (int sr = r_lo; sr < r_hi; ++sr) {
            const float2* lrow = reinterpret_cast<const float2*>(sL2) + (sYs[sr] - gy + R) * LPW;
            const float* drow = sSd + sr * ncm;
            const uint32_t* grow = sSg + sr * ncm;
            f32x2 rnumP[2] = {0ull, 0ull}, rdenP[2] = {0ull, 0ull};
            if constexpr (MAXC > 0) {
#pragma unroll
                for (int c = 0; c < MAXC; ++c)
                    gather_site_p2(gp, drow[scol[c]], grow[scol[c]], lrow + eoff[c], sq, ncO, nkc2, ndelP, e_thr, rnumP, rdenP);
            } else {
#pragma unroll 2
                for (int sc = c_lo; sc < c_hi; ++sc)
                    gather_site_p2(gp, drow[sc], grow[sc], lrow + sXs[sc] + jofs, sq, ncO, nkc2, ndelP, e_thr, rnumP, rdenP);
            }
#pragma unroll
            for (int pr = 0; pr < 2; ++pr) { numP[pr] = add2(numP[pr], rnumP[pr]); denP[pr] = add2(denP[pr], rdenP[pr]); }
        }
        unpack2(numP[0], num[0], num[1]); unpack2(numP[1], num[2], num[3]);
        unpack2(denP[0], den[0], den[1]); unpack2(denP[1], den[2], den[3]);
    }

    float o[4];
    bool flag[4];
    bool anyflag = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float t = (delta[k] + num[k] / den[k]) - c_err;
        o[k] = any[k] ? fmaf(t, p.inv_sq, d0) : 0.f;
        flag[k] = any[k] && !(den[k] >= wsum[k] * p.flag_scale);
        anyflag |= flag[k];
    }
    if (__any_sync(0xffffffffu, anyflag)) {
        const int lane = tid & 31;
        unsigned m[4];
        int total = 0, before = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            m[k] = __ballot_sync(0xffffffffu, flag[k] && gy < p.height && gx + k < p.width);
            before += __popc(m[k] & ((1u << lane) - 1u));
            total += __popc(m[k]);
        }
        unsigned base = 0;
        if (lane == 0 && total > 0) base = atomicAdd(p.q_count, (unsigned)total);
        base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if ((m[k] >> lane) & 1u) {
                const unsigned slot = base + (unsigned)before;
                ++before;
                if (slot < p.q_capacity) p.q_items[slot] = (unsigned)(fpix + (long long)gy * p.width + gx + k);
            }
    }
    if (gy < p.height && gx < p.width) {
        float* dst = p.out + fpix + (long long)gy * p.width + gx;
        if (gx + 3 < p.width && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
            stg_stream_f4(reinterpret_cast<float4*>(dst), make_float4(o[0], o[1], o[2], o[3]));
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (gx + k < p.width) dst[k] = o[k];
        }
    }
}

// -----------------------------------------------------------------------------
// fp64 refinement of the queued (ill-conditioned) pixels.  One warp per pixel: the taps of its window are
// split across the 32 lanes and the four sums are combined with warp shuffles.  This is the reference
// formula (JointBilateralFilter.cu:16-78) with exact exponentials, fp32 only where the reference's
// skip-if-zero guards are decided.  Reads the frame from global memory (just filtered: L2-resident), so
// it is independent of the filter kernel's tiling; the whole GPU shares the queue, so a frame whose
// ill-conditioned pixels cluster in one place (a hole between two surfaces) costs no tail.
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return __shfl_sync(0xffffffffu, v, 0);
}

// two sums reduced in lockstep (their shuffles interleave: half the latency of two separate reductions)
__device__ __forceinline__ void warp_sum2_f64(double& a, double& b) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ta = __shfl_xor_sync(0xffffffffu, a, o), tb = __shfl_xor_sync(0xffffffffu, b, o);
        a += ta;
        b += tb;
    }
    a = __shfl_sync(0xffffffffu, a, 0);
    b = __shfl_sync(0xffffffffu, b, 0);
}

__device__ __forceinline__ float jbf_sample_depth(const JbfParams& p, int frame, int gx, int gy) {
    if (p.mode == kStageUpsample) {
        const int xl = p.ups_inv_x ? __ldg(p.ups_inv_x + gx) : upsample_site(gx, p.width, p.wl);
        const int yl = p.ups_inv_y ? __ldg(p.ups_inv_y + gy) : upsample_site(gy, p.height, p.hl);
        return ((xl >= 0) & (yl >= 0)) ? upsample_sample(p, frame, xl, yl) : 0.f;
    }
    const float* row = static_cast<const float*>(p.depth) + (long long)frame * p.depth_frame_stride + (long long)gy * p.width;
    if (p.depth_up != nullptr && gy < p.band0) row = p.depth_up + (long long)gy * p.width;
    else if (p.depth_dn != nullptr && gy >= p.band1) row = p.depth_dn + (long long)(gy - p.band1) * p.width;
    return load_depth<float>(row, gx);
}

// exp(-x) for x >= 0 in fp64 without the library's special-case handling: 2^(-x log2e) by Cody-Waite
// reduction (n = nearest integer, |f| <= 0.5) and the degree-11 Taylor polynomial of e^(f ln2) (truncation
// < 1e-14 relative), exponent attached by integer add.  Arguments beyond the double range return 0.
__device__ __forceinline__ double exp_neg_f64(double x) {
    // branch-free (the out-of-range case is a clamp + select): the caller's unrolled taps then form independent
    // straight-line chains the scheduler can interleave -- the kernel is bound by the latency of these chains
    const double t0 = -x * 1.4426950408889634;                // log2 domain, <= 0
    const bool tiny = t0 < -1000.0;
    const double t = tiny ? -1000.0 : t0;
    const double kMagic = 6755399441055744.0;                 // 1.5 * 2^52: rounds to nearest integer
    const double tn = t + kMagic;
    const int n = __double2loint(tn);
    const double f = (t - (tn - kMagic)) * 0.6931471805599453; // natural-log units, |f| <= 0.3466
    // Estrin evaluation of sum_{k=0..11} f^k / k! (dependency depth 5 instead of 11)
    const double f2 = f * f, f4 = f2 * f2, f8 = f4 * f4;
    const double q0 = fma(f, 1.0, 1.0);                                            // 1/0! + f/1!
    const double q1 = fma(f, 1.666666666666667e-01, 0.5);                          // 1/2! + f/3!
    const double q2 = fma(f, 8.333333333333333e-03, 4.166666666666666e-02);        // 1/4! + f/5!
    const double q3 = fma(f, 1.984126984126984e-04, 1.388888888888889e-03);        // 1/6! + f/7!
    const double q4 = fma(f, 2.755731922398589e-06, 2.48015873015873e-05);         // 1/8! + f/9!
    const double q5 = fma(f, 2.505210838544172e-08, 2.755731922398589e-07);        // 1/10! + f/11!
    const double r0 = fma(q1, f2, q0), r1 = fma(q3, f2, q2), r2 = fma(q5, f2, q4);
    double p = fma(r1, f4, r0);
    p = fma(r2, f8, p);
    const double r = __hiloint2double(__double2hiint(p) + (n << 20), __double2loint(p));
    return tiny ? 0.0 : r;
}

// KMAX = taps per lane the instantiation can hold: (2r+1)^2 <= 32 * KMAX
// PLAIN = whole-frame / local-band depth plane (no upsampling lattice, no peer-memory halos): direct loads, of
// float32 or (DT = uint16_t, PLAIN only) uint16 depth
template <int KMAX, bool PLAIN, class DT>
__global__ void __launch_bounds__(128) jbf_refine_kernel(const JbfParams p, const int radius) {
    const int lane = threadIdx.x & 31;
    const int ws = 2 * radius + 1, ntap = ws * ws;
    // the lane's taps t = lane + 32 u -> window offsets and spatial weights, once per warp (not per pixel)
    int tdx[KMAX], tdy[KMAX];
    double tsw[KMAX];
    {
        int ti = lane / ws, tj = lane - ti * ws;
        const int di = 32 / ws, dj = 32 - di * ws;
#pragma unroll
        for (int u = 0; u < KMAX; ++u) {
            const int t = lane + 32 * u;
            tdx[u] = tj - radius;
            tdy[u] = (t < ntap) ? ti - radius : (1 << 28);    // beyond the window: fails the bounds test below
            const float s = (t < ntap) ? __ldg(p.slut + t) : 0.f;
            tsw[u] = (s != 0.0f) ? (double)s : 1.0;           // skip-if-zero guard on the spatial factor (.cu:30-31)
            ti += di; tj += dj;
            if (tj >= ws) { tj -= ws; ++ti; }
        }
    }
    grid_dependency_wait();   // the queue is complete only when the filter kernel has finished
    const unsigned nwarps = gridDim.x * (blockDim.x >> 5);
    const unsigned first = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const unsigned total_px = (unsigned)p.out_rows * (unsigned)p.width * (unsigned)p.n_frames;
    // the count and this warp's first item are fetched together (one round trip); a slot beyond the count holds a
    // stale index, which is clamped into the frame and never used
    unsigned idx_next = (first < p.q_capacity) ? p.q_items[first] : 0u;
    const unsigned pushed = *reinterpret_cast<volatile unsigned int*>(p.q_count);
    const unsigned count = pushed < p.q_capacity ? pushed : p.q_capacity;
    const unsigned per_frame = (unsigned)p.out_rows * (unsigned)p.width;
    for (unsigned item = first; item < count; item += nwarps) {
        unsigned idx = idx_next;
        if (idx >= total_px) idx = total_px - 1;
        if (item + nwarps < count) idx_next = p.q_items[item + nwarps];
        const int frame = (int)(idx / per_frame);
        const unsigned rem = idx - (unsigned)frame * per_frame;
        const int oy = (int)(rem / (unsigned)p.width), x = (int)(rem - (unsigned)oy * (unsigned)p.width);
        const int y = oy + p.y_off;
        const uint32_t* gsrc = p.guide4 + (long long)frame * p.guide_frame_stride;
        const DT* dsrc = static_cast<const DT*>(p.depth) + (long long)frame * p.depth_frame_stride;
        // all of the lane's loads are issued before the first use (the taps are independent: one round trip
        // to L2 per pixel instead of two per tap); out-of-window taps read the centre and are masked
        float dfl[KMAX];
        uint32_t gql[KMAX];
        const uint32_t gpix = __ldg(gsrc + (long long)y * p.guide_pitch + x);   // same batch of loads as the taps
#pragma unroll
        for (int u = 0; u < KMAX; ++u) {
            const int ty = y + tdy[u], tx = x + tdx[u];
            const bool in = tx >= 0 && tx < p.width && ty >= 0 && ty < p.height;
            const int cy_ = in ? ty : y, cx_ = in ? tx : x;
            const float df = PLAIN ? load_depth<DT>(dsrc, (long long)cy_ * p.width + cx_) : jbf_sample_depth(p, frame, cx_, cy_);
            gql[u] = __ldg(gsrc + (long long)cy_ * p.guide_pitch + cx_);
            dfl[u] = in ? df : 0.f;
        }
        // each lane keeps its taps in registers between the two passes: depth and the spatial x colour weight.
        // Both passes are straight-line per tap (selects, no branches), so the KMAX exponentials of a lane are
        // independent chains in flight together.
        double dl[KMAX], fl[KMAX];
        double a = 0.0, wt = 0.0;
#pragma unroll
        for (int u = 0; u < KMAX; ++u) {
            const bool v = dfl[u] > kValidDepth;
            const uint32_t ad = __vabsdiffu4(gpix, gql[u]);
            const double cd = (double)__dp4a(ad, ad, 0u);
            const double w = tsw[u] * exp_neg_f64(cd * p.kc);
            const double f = v ? w : 0.0;
            dl[u] = v ? (double)dfl[u] : 0.0;
            fl[u] = f;
            a = fma(dl[u], f, a);
            wt += f;
        }
        warp_sum2_f64(a, wt);
        // wt == 0 (no valid tap): every fl is 0, the pass below yields den == 0 -> output 0 (m is unused garbage-free)
        const double m = (wt > 0.0) ? a / wt : 0.0;
        double num = 0.0, den = 0.0;
#pragma unroll
        for (int u = 0; u < KMAX; ++u) {
            const double e = dl[u] - m;
            const double q = e * e * p.kd;
            const bool keep = q <= kExpZeroArg;               // else fp32 expf() == 0: factor skipped (.cu:67-68)
            const double g = exp_neg_f64(keep ? q : 0.0);
            const double f = keep ? fl[u] * g : fl[u];
            num = fma(dl[u], f, num);
            den += f;
        }
        warp_sum2_f64(num, den);
        const float r = (den == 0.0) ? 0.f : (float)(num / den);
        if (lane == 0) {
            p.out[idx] = r;
            if (p.xyz != nullptr) {
                const float px = __fdiv_rn(__fsub_rn((float)x, (float)p.cx), p.fx);
                const float py = __fdiv_rn(__fsub_rn((float)p.cy, (float)(p.y_img0 + y)), p.fy);
                float* xd = p.xyz + 3ll * idx;
                xd[0] = __fmul_rn(px, r); xd[1] = __fmul_rn(py, r); xd[2] = r;
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && p.stats != nullptr && pushed != 0u) {
        atomicAdd(p.stats, (unsigned long long)count);
        atomicAdd(p.stats + 1, (unsigned long long)(pushed - count));
    }
}

// -----------------------------------------------------------------------------
// Generic kernel: any radius <= KDME_MAX_RADIUS, any sigmas (including those for
// which the colour skip-if-zero guard can fire, sigma_c == 0 and sigma_d == 0).
// One pixel per thread, same staging and the same shifted accumulation; the
// guards are evaluated explicitly per tap.  Used when the fast path's
// preconditions do not hold; slower by design.
struct JbfGenericParams {
    JbfParams base;
    int radius;
    int cd_skip;      // colour factor skipped when cd > cd_skip (fp32 expf == 0); INT_MAX = never
    int use_color;    // 0 when sigma_c == 0 (factor is 0 -> skipped, .cu:26-27,32-33)
    int use_depth;    // 0 when sigma_d == 0 (depth_filter uninitialised in the reference -> skipped)
};

template <int TW, int TH, class DT>
__global__ void __launch_bounds__(TW * TH)
jbf_generic_kernel(const JbfGenericParams gp_) {
    const JbfParams& p = gp_.base;
    const int R = gp_.radius, WS = 2 * R + 1;
    const int SP = TW + 2 * R, SH = TH + 2 * R;
    extern __shared__ __align__(128) uint8_t smem_gen[];
    float* sD = reinterpret_cast<float*>(smem_gen);
    uint32_t* sG = reinterpret_cast<uint32_t*>(sD + SP * SH);
    float* sL = reinterpret_cast<float*>(sG + SP * SH);
    __shared__ float sRed[32];
    constexpr int NT = TW * TH;
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TW, y0 = p.y_off + blockIdx.y * TH, frame = blockIdx.z;
    const uint32_t* gsrc = p.guide4 + (long long)frame * p.guide_frame_stride;
    const DT* dsrc = static_cast<const DT*>(p.depth) + (long long)frame * p.depth_frame_stride;
    for (int idx = tid; idx < SP * SH; idx += NT) {
        int sy = idx / SP, sx = idx - sy * SP;
        int gx = x0 - R + sx, gy = y0 - R + sy;
        bool in = (gx >= 0) & (gx < p.width) & (gy >= 0) & (gy < p.height);
        float d = 0.f;
        uint32_t g = 0u;
        if (in) {
            g = __ldg(gsrc + (long long)gy * p.guide_pitch + gx);
            if (p.mode == kStageUpsample) {
                int xl = upsample_site(gx, p.width, p.wl);
                int yl = upsample_site(gy, p.height, p.hl);
                if ((xl >= 0) & (yl >= 0)) d = upsample_sample(p, frame, xl, yl);
            } else {
                d = load_depth<DT>(dsrc, (long long)gy * p.width + gx);
            }
        }
        sD[idx] = d;
        sG[idx] = g;
    }
    for (int idx = tid; idx < WS * WS; idx += NT) sL[idx] = __ldg(p.ltab + idx);
    __syncthreads();
    float lmin = 3.0e38f;
    for (int idx = tid; idx < SP * SH; idx += NT) {
        float d = sD[idx];
        if (d > kValidDepth) lmin = fminf(lmin, d);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lmin = fminf(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
    if ((tid & 31) == 0) sRed[tid >> 5] = lmin;
    __syncthreads();
    float dref = 3.0e38f;
    for (int w = 0; w < NT / 32; ++w) dref = fminf(dref, sRed[w]);
    if (dref > 1.0e38f) dref = 0.f;
    __syncthreads();
    for (int idx = tid; idx < SP * SH; idx += NT) {
        float d = sD[idx];
        // invalid samples are flagged with NaN-free sentinel: negative infinity never occurs in input
        sD[idx] = (d > kValidDepth) ? (d - dref) * p.sq : -3.0e38f;
    }
    __syncthreads();

    const int lx = tid % TW, ly = tid / TW;
    const int pc = (ly + R) * SP + lx + R;
    const uint32_t gpix = sG[pc];
    // accumulation origin: the centre sample, else the first sample of the window
    float d0 = sD[pc];
    if (!(d0 > -1.0e38f)) {
        d0 = 0.f;
        for (int t = 0; t < WS * WS; ++t) {
            const int i = t / WS, j = t - i * WS;
            const float d = sD[(ly + i) * SP + lx + j];
            if (d > -1.0e38f) { d0 = d; break; }
        }
    }
    float acc = 0.f, wsum = 0.f;
    for (int i = 0; i < WS; ++i) {
        float racc = 0.f, rws = 0.f;
        for (int j = 0; j < WS; ++j) {
            const int q = (ly + i) * SP + lx + j;
            const float d = sD[q];
            if (!(d > -1.0e38f)) continue;
            const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
            const int cd = (int)__dp4a(ad, ad, 0u);
            float arg = sL[i * WS + j];
            if (gp_.use_color && cd <= gp_.cd_skip) arg = fmaf((float)cd, p.nkc, arg);
            const float f = ex2_approx(arg);
            racc = fmaf(f, d - d0, racc);
            rws += f;
        }
        acc += racc;
        wsum += rws;
    }
    float o = 0.f;
    if (wsum > 0.f) {
        const float delta = acc / wsum;  // mean = d0 + delta
        float num = 0.f, den = 0.f;
        for (int i = 0; i < WS; ++i) {
            float rnum = 0.f, rden = 0.f;
            for (int j = 0; j < WS; ++j) {
                const int q = (ly + i) * SP + lx + j;
                const float d = sD[q];
                if (!(d > -1.0e38f)) continue;
                const uint32_t ad = __vabsdiffu4(gpix, sG[q]);
                const int cd = (int)__dp4a(ad, ad, 0u);
                float arg = sL[i * WS + j];
                if (gp_.use_color && cd <= gp_.cd_skip) arg = fmaf((float)cd, p.nkc, arg);
                const float e = (d - d0) - delta;
                if (gp_.use_depth && !(fabsf(e) > p.e_thr)) arg = fmaf(-e, e, arg);
                const float f = ex2_approx(arg);
                rnum = fmaf(f, e, rnum);
                rden += f;
            }
            num += rnum;
            den += rden;
        }
        o = (den > 0.f) ? dref + ((delta + num / den) + d0) * p.inv_sq : 0.f;
    }
    const int gx = x0 + lx, oy = y0 + ly - p.y_off;
    if (gx < p.width && oy < p.out_rows)
        p.out[(long long)frame * p.width * p.out_rows + (long long)oy * p.width + gx] = o;
}

}  // namespace kdme
