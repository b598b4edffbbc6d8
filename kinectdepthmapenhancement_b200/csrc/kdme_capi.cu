// kdme_capi.cu -- extern "C" boundary (include/kdme_b200.h) over the sm_100a kernels.
//
// Host-side logic only: argument validation, LUT construction (the reference's
// calcSpatialFilter, JointBilateralFilter.cpp:31-40), kernel selection, TMA
// descriptor encoding, launch.  There is no CPU fallback: every entry point
// either launches a CUDA kernel or returns an error.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <type_traits>
#include <vector>

#include "../../include/kdme_b200.h"
#include "buffer2d_kernels.cuh"
#include "guided_kernels.cuh"
#include "jbf_kernels.cuh"
#include "presmooth_kernels.cuh"

using namespace kdme;

// ------------------------------------------------------------------ errors
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CK(expr)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(-(int)e_, std::string(#expr) + ": " + cudaGetErrorString(e_));             \
    } while (0)

extern "C" const char* kdme_last_error(void) { return g_err.c_str(); }
extern "C" const char* kdme_version(void) { return "kdme_b200 0.1.0 sm_100a"; }

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// ------------------------------------------------------------------ TMA descriptors
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

// The handle-less entry points (kdme_guided_*, kdme_depth_bilateral_xyz, kdme_mean_3d_error,
// kdme_projective_to_real) launch on the CURRENT device: their pointers must live there.
static int check_pointer_device(const void* ptr, const char* who) {
    cudaPointerAttributes a;
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess) return fail(KDME_EINVAL, std::string(who) + ": no current CUDA device");
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return fail(KDME_EINVAL, std::string(who) + ": not a CUDA pointer"); }
    if (a.type == cudaMemoryTypeDevice && a.device != cur)
        return fail(KDME_EINVAL, std::string(who) + ": pointer lives on device " + std::to_string(a.device) +
                                 " but the current device is " + std::to_string(cur) + " (call cudaSetDevice first)");
    static std::atomic<unsigned long long> ok_devs{0}, bad_devs{0};   // compute capability, looked up once per device
    const unsigned long long bit = 1ull << (cur & 63);
    if (!((ok_devs.load(std::memory_order_acquire) | bad_devs.load(std::memory_order_acquire)) & bit)) {
        int major = 0;
        cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, cur);
        (major == 10 ? ok_devs : bad_devs).fetch_or(bit, std::memory_order_release);
    }
    if (bad_devs.load(std::memory_order_acquire) & bit)
        return fail(KDME_ENOTSUP, std::string(who) + ": this library is built for sm_100a (B200) only");
    return KDME_OK;
}

// 3-D map over [n][rows][pitch_elems] 4-byte elements, box {bx, by, 1}, zero OOB fill.
static bool encode_map(CUtensorMap* map, CUtensorMapDataType dt, const void* base, int width, int height, int n,
                       long long row_pitch_bytes, long long frame_pitch_bytes, int bx, int by) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[3] = {(cuuint64_t)width, (cuuint64_t)height, (cuuint64_t)n};
    cuuint64_t strides[2] = {(cuuint64_t)row_pitch_bytes, (cuuint64_t)frame_pitch_bytes};
    cuuint32_t box[3] = {(cuuint32_t)bx, (cuuint32_t)by, 1u};
    cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = fn(map, dt, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

// ------------------------------------------------------------------ JBF handle
constexpr int kPipeDepth = 3;  // device slots of the host pipeline (jbf_process_host)
struct jbf_handle {
    int width = 0, height = 0, radius = 0, max_batch = 1, device = 0;
    float sigma_s = 0, sigma_c = 0, sigma_d = 0;
    // pre-smooth (JointBilateralFilter.cu:285)
    int ps_ksize = 5;
    float ps_sigma_c = 30.f, ps_sigma_s = 30.f;
    float *ps_space_dev = nullptr, *ps_color_dev = nullptr;
    // owned buffers
    float* filtered_dev = nullptr;   // Filtered_Device
    float* filtered_host = nullptr;  // Filtered_Host (pinned, lazy)
    int guide_pitch = 0;             // words per row of a lane's guide4
    uint8_t* smooth_bgr = nullptr;   // copy in the guide's format for getSmoothImage_Device (lazy)
    size_t smooth_bytes = 0;         // its size
    int guide_channels = 3;          // bytes per pixel of every raw guide the handle reads (1, 3 or 4)
    float* ltab_pairs_dev = nullptr; // packed-math layout [WS][LPP][2] = {L[i][j], L[i][j-1]}, j = 1..WS-1 (pass 2, bias 32)
    float* ltab_pairs1_dev = nullptr;// same layout for pass 1, bias `bias1`
    float* slut_dev = nullptr;       // the raw fp32 LUT of calcSpatialFilter [WS][WS] (fp64 refinement path)
    unsigned long long* stats_dev = nullptr;  // [0] pixels refined in fp64, [1] dropped (queue full), since the last jbf_refine_stats
    float bias1 = 0.f, flag_scale = 0.f;
    double kc = 0, kd = 0;
    float* ltab_generic_dev = nullptr;  // [WS][WS], bias kWeightBias
    float *ltab_ups1_dev = nullptr, *ltab_ups2_dev = nullptr;   // padded pair tables of the gather-form upsampling
    // derived
    bool fast = false;
    float nkc = 0, sq = 1, inv_sq = 1, e_thr = 0;
    int cd_skip = INT_MAX, use_color = 1, use_depth = 1;
    bool force_no_tma = false, no_refine = false;
    int force_tile_h = 0;
    int last_variant = 0;
    // What a stream of launches owns; every launch is given the lane it runs on.  lanes[0] is the caller's stream
    // with the buffers jbf_create allocates.  lanes[1] is the internal lane of the chunk loops (run_chunks),
    // allocated on first use: odd chunks run there with their own guide buffer, refinement queue and TMA
    // descriptors, so that a chunk's pre-smooth fills the tail of the previous chunk's filter and the fp64
    // refinement launch hides behind the next filter.
    struct MapKey { const void* depth = nullptr; const void* guide = nullptr; int rows = 0, n = 0, gp = 0, bx = 0, by = 0; };
    struct Lane {
        cudaStream_t stream = nullptr;
        uint32_t* guide4 = nullptr;            // smooth_Device in the internal u8x4 layout, max_batch frames
        unsigned int* q_count_dev = nullptr;   // refinement queue (see JbfParams): two alternating counters
        int q_cur = 0;
        unsigned int* q_items_dev = nullptr;
        size_t q_capacity = 0;
        // TMA descriptors of the lane's last fast launch, reused while (pointers, rows, frames, box) are unchanged
        MapKey map_key;
        CUtensorMap map_depth, map_guide;
    } lanes[2];
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // gather-form upsampling: the site lattice tabulated for (ups_wl, ups_hl, ups_rows): site_x[wl], site_y[hl],
    // tile_xl[tiles_x][2], tile_yl[tiles_y][2]
    int* ups_tab_dev = nullptr; int ups_wl = 0, ups_hl = 0, ups_rows = 0;
    bool one_lane = false;
    // host pipeline (jbf_process_host)
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_in[kPipeDepth] = {}, ev_done[kPipeDepth] = {}, ev_free[kPipeDepth] = {};
    float* pipe_depth[kPipeDepth] = {};
    uint16_t* pipe_depth16[kPipeDepth] = {};   // u16 sensor depth staging (jbf_process_host_u16), lazy
    uint8_t* pipe_bgr[kPipeDepth] = {};
    float* pipe_out[kPipeDepth] = {};
    size_t pipe_bgr_step = 0;
    int pipe_chunk = 1;
};

using Lane = jbf_handle::Lane;

static bool fast_radius_available(int r);
static int buf_blocks(long long n);

static int ensure_alt_lane(jbf_handle* h) {
    Lane& a = h->lanes[1];
    if (a.stream) return KDME_OK;
    cudaStream_t s = nullptr;
    CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    cudaError_t e = cudaMalloc(&a.guide4, (size_t)h->max_batch * h->height * h->guide_pitch * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&a.q_count_dev, 2 * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemset(a.q_count_dev, 0, 2 * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        cudaFree(a.guide4); cudaFree(a.q_count_dev); cudaStreamDestroy(s);
        a.guide4 = nullptr; a.q_count_dev = nullptr;
        return fail(-(int)e, std::string("second chunk lane: ") + cudaGetErrorString(e));
    }
    a.stream = s;
    return KDME_OK;
}

// calcSpatialFilter -- JointBilateralFilter.cpp:31-40, fp32 on the host as the reference does.
static void host_spatial_lut(std::vector<float>& lut, int ws, float sigma_s) {
    lut.resize((size_t)ws * ws);
    for (int i = 0; i < ws; i++)
        for (int j = 0; j < ws; j++) {
            float dx = (float)(j - ws / 2), dy = (float)(i - ws / 2);
            float dis_x = dx * dx, dis_y = dy * dy;
            lut[(size_t)i * ws + j] = expf(-(dis_x + dis_y) / (2.0f * (sigma_s * sigma_s)));
        }
}

// A spatial weight s in the log2 domain, plus the exponent bias; s == 0 contributes the bias alone (the skip-if-zero
// guard on the spatial factor, JointBilateralFilter.cu:30-31,63-64).
static float log2_weight(float s, float bias) {
    return (s != 0.0f && std::isfinite(s)) ? (float)(std::log2((double)s) + (double)bias) : bias;
}

// [ws][ws] log2 weights: the generic kernel's table.
static std::vector<float> generic_table(const std::vector<float>& lut, int ws, float bias) {
    std::vector<float> t(lut.size());
    for (size_t i = 0; i < lut.size(); i++) t[i] = log2_weight(lut[i], bias);
    return t;
}

// Packed-math pair table of the fast kernel: [ws][ws - 1][2] = {L[i][j], L[i][j-1]}, j = 1..ws-1.
static std::vector<float> pair_table(const std::vector<float>& lut, int ws, float bias) {
    const int lpp = ws - 1;
    std::vector<float> t((size_t)ws * std::max(lpp, 1) * 2, 0.f);
    for (int i = 0; i < ws; i++)
        for (int j = 1; j < ws; j++) {
            t[((size_t)i * lpp + (j - 1)) * 2 + 0] = log2_weight(lut[(size_t)i * ws + j], bias);
            t[((size_t)i * lpp + (j - 1)) * 2 + 1] = log2_weight(lut[(size_t)i * ws + j - 1], bias);
        }
    return t;
}

// Padded pair table of the gather-form upsampling (see jbf_upsample_gather_kernel): [ws][ws + kUpsPad][2] =
// {L[i][e-2], L[i][e-3]}, -3e38 where the column lies outside the window.
static std::vector<float> ups_pair_table(const std::vector<float>& lut, int ws, float bias) {
    const int lpw = ws + kUpsPad;
    const float kOut = -3.0e38f;
    std::vector<float> t((size_t)ws * lpw * 2);
    for (int i = 0; i < ws; i++)
        for (int e = 0; e < lpw; e++) {
            const int jj = e - 2;
            t[((size_t)i * lpw + e) * 2 + 0] = (jj >= 0 && jj < ws) ? log2_weight(lut[(size_t)i * ws + jj], bias) : kOut;
            t[((size_t)i * lpw + e) * 2 + 1] = (jj >= 1 && jj <= ws) ? log2_weight(lut[(size_t)i * ws + jj - 1], bias) : kOut;
        }
    return t;
}

// cudaMalloc + an upload on `st`; the caller synchronises `st` before `v` goes away.
static cudaError_t upload(float** dev, const std::vector<float>& v, cudaStream_t st) {
    const cudaError_t e = cudaMalloc(dev, v.size() * sizeof(float));
    return e != cudaSuccess ? e : cudaMemcpyAsync(*dev, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice, st);
}

static int build_tables(jbf_handle* h) {
    cudaStream_t st = h->lanes[0].stream;
    const int ws = 2 * h->radius + 1;
    std::vector<float> lut;
    host_spatial_lut(lut, ws, h->sigma_s);
    // pass 1 evaluates 2^(arg + bias1): with bias1 = 0 the heavy taps' arguments are rounded near 0
    // (ulp ~1e-8) instead of near 32 (ulp 3.8e-6), which is what the pass-1 mean's accuracy needs.  The
    // bias is only kept when some pass-1 weight could otherwise flush to zero under ex2.approx.ftz.
    double lmin = 0.0;
    for (size_t i = 0; i < lut.size(); i++)
        if (lut[i] != 0.0f && std::isfinite(lut[i])) lmin = std::min(lmin, std::log2((double)lut[i]));
    const double cmin = (h->sigma_c != 0.0f) ? -kLog2e * 3.0 * 255.0 * 255.0 / (2.0 * (double)h->sigma_c * (double)h->sigma_c) : 0.0;
    h->bias1 = (lmin + cmin > -120.0) ? 0.f : kWeightBias;
    const std::vector<float> pairs = pair_table(lut, ws, kWeightBias), pairs1 = pair_table(lut, ws, h->bias1),
                             generic = generic_table(lut, ws, kWeightBias), ups1 = ups_pair_table(lut, ws, h->bias1),
                             ups2 = ups_pair_table(lut, ws, kWeightBias);
    CK(upload(&h->ltab_pairs_dev, pairs, st));
    CK(upload(&h->ltab_pairs1_dev, pairs1, st));
    CK(upload(&h->ltab_generic_dev, generic, st));
    CK(upload(&h->ltab_ups1_dev, ups1, st));
    CK(upload(&h->ltab_ups2_dev, ups2, st));
    CK(upload(&h->slut_dev, lut, st));
    CK(cudaMalloc(&h->stats_dev, 2 * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(h->stats_dev, 0, 2 * sizeof(unsigned long long), st));
    CK(cudaMalloc(&h->lanes[0].q_count_dev, 2 * sizeof(unsigned int)));
    CK(cudaMemsetAsync(h->lanes[0].q_count_dev, 0, 2 * sizeof(unsigned int), st));
    CK(cudaStreamSynchronize(st));

    // colour factor: exp(-cd/(2 sc^2)); cd is an integer in [0, 3*255^2]
    h->use_color = (h->sigma_c != 0.0f);
    h->use_depth = (h->sigma_d != 0.0f);
    h->cd_skip = INT_MAX;
    if (h->use_color) {
        const float den = 2 * (h->sigma_c * h->sigma_c);
        h->nkc = (float)(-kLog2e / (2.0 * (double)h->sigma_c * (double)h->sigma_c));
        // largest cd whose fp32 expf() is still non-zero (monotone): binary search
        int lo = 0, hi = 3 * 255 * 255;
        if (expf(-(float)hi / den) == 0.0f) {
            while (lo < hi) {
                int mid = (lo + hi + 1) / 2;
                if (expf(-(float)mid / den) != 0.0f) lo = mid; else hi = mid - 1;
            }
            h->cd_skip = lo;
        }
    } else {
        h->nkc = 0.f;
    }
    if (h->use_depth) {
        const double k = kLog2e / (2.0 * (double)h->sigma_d * (double)h->sigma_d);
        h->sq = (float)std::sqrt(k);
        h->inv_sq = (float)(1.0 / std::sqrt(k));
        h->e_thr = (float)std::sqrt(kExpZeroArg * kLog2e);  // == sqrt(150) in scaled units
    } else {
        h->sq = 1.f; h->inv_sq = 1.f; h->e_thr = 3.0e38f;
    }
    // fast path: colour guard can never fire, all factors present, kernel instantiated, and the
    // invalid-tap marker (1.7e38 * nkc) must still drive the exponent to -inf.
    h->fast = h->use_color && h->use_depth && h->cd_skip == INT_MAX && std::isfinite(h->nkc) &&
              (h->nkc < -1e-20f) && std::isfinite(h->sq) && h->sq > 0.f && fast_radius_available(h->radius);
    if (getenv("KDME_FORCE_GENERIC")) h->fast = false;
    h->force_no_tma = getenv("KDME_NO_TMA") != nullptr;
    h->no_refine = getenv("KDME_NO_REFINE") != nullptr;
    h->one_lane = getenv("KDME_ONE_LANE") != nullptr;
    if (const char* th = getenv("KDME_TILE_H")) h->force_tile_h = atoi(th);
    h->kc = h->use_color ? 1.0 / (2.0 * (double)h->sigma_c * (double)h->sigma_c) : 0.0;
    h->kd = h->use_depth ? 1.0 / (2.0 * (double)h->sigma_d * (double)h->sigma_d) : 0.0;
    // refine in fp64 when the mean range weight den/wsum (biases removed) is below 2^-8
    h->flag_scale = h->no_refine ? 0.f : (float)std::exp2((double)kWeightBias - (double)h->bias1 - 8.0);
    return KDME_OK;
}

static int build_presmooth_luts(jbf_handle* h) {
    if (h->ps_ksize == 0) return KDME_OK;
    cudaStream_t st = h->lanes[0].stream;
    const int k = h->ps_ksize, r = k / 2;
    std::vector<float> sp((size_t)k * k), col(766);
    const float ss = -0.5f / (h->ps_sigma_s * h->ps_sigma_s);
    const float sc = -0.5f / (h->ps_sigma_c * h->ps_sigma_c);
    for (int dy = -r; dy <= r; dy++)
        for (int dx = -r; dx <= r; dx++) {
            int s2 = dx * dx + dy * dy;
            sp[(size_t)(dy + r) * k + (dx + r)] = (s2 > r * r) ? -1.0f : expf((float)s2 * ss);
        }
    for (int n = 0; n <= 765; n++) col[n] = expf((float)(n * n) * sc);
    if (!h->ps_space_dev) CK(cudaMalloc(&h->ps_space_dev, kPsMaxK * kPsMaxK * sizeof(float)));
    if (!h->ps_color_dev) CK(cudaMalloc(&h->ps_color_dev, 768 * sizeof(float)));
    CK(cudaMemcpyAsync(h->ps_space_dev, sp.data(), sp.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->ps_color_dev, col.data(), col.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    return KDME_OK;
}

extern "C" int jbf_create(jbf_handle** out, int width, int height, float sigma_spatial, float sigma_color,
                          float sigma_depth, int window_radius, int max_batch, int device, void* stream) {
    if (!out) return fail(KDME_EINVAL, "jbf_create: out is NULL");
    *out = nullptr;
    if (width <= 0 || height <= 0) return fail(KDME_EINVAL, "jbf_create: width/height must be positive");
    if (window_radius < 0 || window_radius > KDME_MAX_RADIUS)
        return fail(KDME_EINVAL, "jbf_create: window_radius must be in [0, 15]");
    if (max_batch < 1 || max_batch > 65535)
        return fail(KDME_EINVAL, "jbf_create: max_batch must be in [1, 65535] (frames are grid.z of one launch)");
    if (!(sigma_spatial == sigma_spatial) || !(sigma_color == sigma_color) || !(sigma_depth == sigma_depth) ||
        sigma_spatial < 0 || sigma_color < 0 || sigma_depth < 0)
        return fail(KDME_EINVAL, "jbf_create: sigmas must be non-negative numbers");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(KDME_EINVAL, "jbf_create: no such CUDA device");
    DeviceGuard g(device);
    if (!g.ok) return fail(KDME_EINVAL, "jbf_create: cudaSetDevice failed");
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(KDME_ENOTSUP, "jbf_create: this library is built for sm_100a (B200) only");
    jbf_handle* h = new jbf_handle();
    h->width = width; h->height = height; h->radius = window_radius; h->max_batch = max_batch;
    h->device = device; h->lanes[0].stream = (cudaStream_t)stream;
    h->sigma_s = sigma_spatial; h->sigma_c = sigma_color; h->sigma_d = sigma_depth;
    h->guide_pitch = (width + 3) & ~3;
    int rc = KDME_OK;
    auto cleanup = [&](int code) { jbf_destroy(h); return code; };
    cudaError_t e;
    if ((e = cudaMalloc(&h->filtered_dev, (size_t)width * height * sizeof(float))) != cudaSuccess)
        return cleanup(fail(-(int)e, "jbf_create: cudaMalloc(Filtered_Device) failed"));
    if ((e = cudaMalloc(&h->lanes[0].guide4, (size_t)max_batch * height * h->guide_pitch * sizeof(uint32_t))) != cudaSuccess)
        return cleanup(fail(-(int)e, "jbf_create: cudaMalloc(smooth_Device) failed"));
    if ((rc = build_tables(h)) != KDME_OK) return cleanup(rc);
    if ((rc = build_presmooth_luts(h)) != KDME_OK) return cleanup(rc);
    *out = h;
    return KDME_OK;
}

extern "C" void jbf_destroy(jbf_handle* h) {
    if (!h) return;
    DeviceGuard g(h->device);
    cudaFree(h->filtered_dev);
    if (h->filtered_host) cudaFreeHost(h->filtered_host);
    cudaFree(h->smooth_bgr);
    cudaFree(h->ltab_pairs_dev);
    cudaFree(h->ltab_pairs1_dev);
    cudaFree(h->slut_dev);
    cudaFree(h->stats_dev);
    cudaFree(h->ups_tab_dev);
    cudaFree(h->ltab_ups1_dev);
    cudaFree(h->ltab_ups2_dev);
    for (Lane& l : h->lanes) {
        cudaFree(l.guide4);
        cudaFree(l.q_count_dev);
        cudaFree(l.q_items_dev);
    }
    if (h->lanes[1].stream) cudaStreamDestroy(h->lanes[1].stream);   // lanes[0] runs on the caller's stream
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    cudaFree(h->ltab_generic_dev);
    cudaFree(h->ps_space_dev);
    cudaFree(h->ps_color_dev);
    for (int b = 0; b < kPipeDepth; b++) {
        cudaFree(h->pipe_depth[b]); cudaFree(h->pipe_bgr[b]); cudaFree(h->pipe_out[b]); cudaFree(h->pipe_depth16[b]);
        if (h->ev_in[b]) cudaEventDestroy(h->ev_in[b]);
        if (h->ev_done[b]) cudaEventDestroy(h->ev_done[b]);
        if (h->ev_free[b]) cudaEventDestroy(h->ev_free[b]);
    }
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
    delete h;
}

extern "C" int jbf_set_presmooth(jbf_handle* h, int ksize, float sigma_color, float sigma_spatial) {
    if (!h) return fail(KDME_EINVAL, "jbf_set_presmooth: NULL handle");
    if (ksize != 0 && (ksize < 1 || ksize > kPsMaxK || (ksize & 1) == 0))
        return fail(KDME_EINVAL, "jbf_set_presmooth: ksize must be 0 (off) or odd in [1, 9]");
    if (ksize != 0 && (!(sigma_color > 0) || !(sigma_spatial > 0)))
        return fail(KDME_EINVAL, "jbf_set_presmooth: sigmas must be positive");
    DeviceGuard g(h->device);
    h->ps_ksize = ksize; h->ps_sigma_c = sigma_color; h->ps_sigma_s = sigma_spatial;
    return build_presmooth_luts(h);
}

extern "C" int jbf_set_guide_channels(jbf_handle* h, int channels) {
    if (!h) return fail(KDME_EINVAL, "jbf_set_guide_channels: NULL handle");
    if (channels != KDME_GUIDE_GRAY && channels != KDME_GUIDE_BGR && channels != KDME_GUIDE_BGRX)
        return fail(KDME_EINVAL, "jbf_set_guide_channels: channels must be 1 (GRAY), 3 (BGR) or 4 (BGRX)");
    h->guide_channels = channels;
    return KDME_OK;
}

// Default (0) and minimum row step of a raw guide of `channels` bytes per pixel.
static int check_guide_step(int channels, int width, size_t* step, const char* who) {
    const size_t row = (size_t)channels * width;
    if (*step == 0) *step = row;
    if (*step < row)
        return fail(KDME_EINVAL, std::string(who) + ": guide step smaller than " + std::to_string(channels) + "*width");
    return KDME_OK;
}

// The same for a raw guide of the handle's format.
static int guide_step(const jbf_handle* h, size_t* step, const char* who) {
    return check_guide_step(h->guide_channels, h->width, step, who);
}

// Default (0) and checks of the row step of a caller's internal u8x4 guide; *pitch_words is the step in words.
static int guide4_step(const jbf_handle* h, size_t* step, int* pitch_words, const char* who) {
    if (*step == 0) *step = (size_t)h->guide_pitch * 4;
    if (*step % 4 != 0 || *step < (size_t)h->width * 4)
        return fail(KDME_EINVAL, std::string(who) + ": guide_step must be a multiple of 4 and >= 4*width");
    *pitch_words = (int)(*step / 4);
    return KDME_OK;
}

// ------------------------------------------------------------------ launches
// fn(std::integral_constant<int, C>{}) for a guide of c = 1, 3 or 4 channels (validated by the caller).
template <class Fn>
static auto with_channels(int c, Fn&& fn) {
    switch (c) {
        case 1: return fn(std::integral_constant<int, 1>{});
        case 4: return fn(std::integral_constant<int, 4>{});
        default: return fn(std::integral_constant<int, 3>{});
    }
}

// cudaLaunchKernelEx, with programmatic stream serialisation when `pdl`: the kernel may launch before the previous
// kernel on the stream has finished, and waits for it on the device.
template <class Kern, class... Args>
static int launch_ex(Kern kern, dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, const Args&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    CK(cudaLaunchKernelEx(&cfg, kern, args...));
    return KDME_OK;
}

// Lets Kern use up to `bytes` of dynamic shared memory on `device`; set once per device (one bit each).
template <auto Kern>
static int allow_dyn_smem(int device, int bytes) {
    static std::atomic<unsigned long long> done{0};
    const unsigned long long bit = 1ull << (device & 63);
    if (!(done.load(std::memory_order_acquire) & bit)) {
        CK(cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        done.fetch_or(bit, std::memory_order_release);
    }
    return KDME_OK;
}

// The raw guide in the handle's format -> the internal u8x4 guide, without smoothing.
static void launch_guide4_convert(jbf_handle* h, Lane& lane, const uint8_t* bgr, size_t bgr_step,
                                  long long bgr_frame_stride, uint32_t* guide4, int guide_pitch,
                                  long long guide_frame_stride, int rows, int n) {
    dim3 blk(128), grd((h->width + 127) / 128, rows, n);
    with_channels(h->guide_channels, [&](auto c) {
        bgr_to_guide4_kernel<decltype(c)::value><<<grd, blk, 0, lane.stream>>>(
            bgr, (long long)bgr_step, bgr_frame_stride, guide4, guide_pitch, guide_frame_stride, h->width, rows);
    });
}

template <int C>
static void launch_presmooth_c(jbf_handle* h, Lane& lane, const PresmoothParams& p, int rows, int n) {
    if (h->ps_ksize == 5) {
        // 64x16 tiles, 128 threads, 4x2 pixels per thread; a launch too small to fill the GPU with them (one
        // Kinect frame is 300) uses 64x8 tiles of 128 threads with 4x1 pixels: four times the warps
        constexpr int TW = 64;
        const long long ctas16 = (long long)((h->width + TW - 1) / TW) * ((rows + 15) / 16) * n;
        if (ctas16 >= 148LL * 6) {
            dim3 grd((h->width + TW - 1) / TW, (rows + 15) / 16, n);
            presmooth5_kernel<TW, 16, 2, C><<<grd, (TW / 4) * 8, 0, lane.stream>>>(p);
        } else {
            dim3 grd((h->width + TW - 1) / TW, (rows + 7) / 8, n);
            presmooth5_kernel<TW, 8, 1, C><<<grd, (TW / 4) * 8, 0, lane.stream>>>(p);
        }
    } else {
        constexpr int TW = 32, TH = 8;
        dim3 grd((h->width + TW - 1) / TW, (rows + TH - 1) / TH, n);
        presmooth_kernel<TW, TH, C><<<grd, TW * TH, 0, lane.stream>>>(p);
    }
}

static int launch_presmooth(jbf_handle* h, Lane& lane, const uint8_t* bgr, size_t bgr_step, uint32_t* guide4,
                            int guide_pitch, int n, int rows = -1, const uint8_t* bgr_up = nullptr,
                            const uint8_t* bgr_dn = nullptr, int band0 = 0, int band1 = 0) {
    if (rows < 0) rows = h->height;
    { int rc = guide_step(h, &bgr_step, "pre-smooth"); if (rc != KDME_OK) return rc; }
    if (h->ps_ksize == 0) {
        if (bgr_up || bgr_dn) return fail(KDME_ENOTSUP, "peer-memory halos need the guide pre-smooth enabled");
        launch_guide4_convert(h, lane, bgr, bgr_step, (long long)bgr_step * rows, guide4, guide_pitch,
                              (long long)guide_pitch * rows, rows, n);
    } else {
        PresmoothParams p;
        p.width = h->width; p.height = rows; p.n_frames = n;
        p.bgr = bgr; p.bgr_step = (long long)bgr_step; p.bgr_frame_stride = (long long)bgr_step * rows;
        p.guide4 = guide4; p.guide_pitch = guide_pitch; p.guide_frame_stride = (long long)guide_pitch * rows;
        p.ksize = h->ps_ksize; p.space_lut = h->ps_space_dev; p.color_lut = h->ps_color_dev;
        p.bgr_up = bgr_up; p.bgr_dn = bgr_dn; p.band0 = band0; p.band1 = band1;
        with_channels(h->guide_channels, [&](auto c) { launch_presmooth_c<decltype(c)::value>(h, lane, p, rows, n); });
    }
    CK(cudaGetLastError());
    return KDME_OK;
}

// One (radius, tile height) instantiation: encode (or reuse) the TMA maps for its box and launch.
template <int R, int TH>
static int launch_fast_rt(jbf_handle* h, Lane& lane, JbfParams p, bool want_tma, bool pdl) {
    constexpr int TW = 64;
    const int rows = p.height;
    using T = JbfTile<R, TW, TH>;
    // resident CTAs per SM, by registers and by shared memory.  Registers: r <= 5 runs best at 80, r = 6..9 at 64
    // (one more resident CTA of 256 threads, +2.5 % measured), larger windows need 128 (the row segment alone is
    // 3 x (2r + 8) registers)
    constexpr int kByRegs = (R <= 5 ? 65536 / 80 : R <= 9 ? 65536 / 64 : 65536 / 128) / T::NT;
    constexpr int kBySmem = (227 * 1024) / (T::SMEM + 1024);
    constexpr int MINB = (kByRegs < kBySmem ? kByRegs : kBySmem) < 1 ? 1 : (kByRegs < kBySmem ? kByRegs : kBySmem);
    constexpr int kSmemCap = 226 * 1024;
    { int rc = allow_dyn_smem<jbf_fast_kernel<R, TW, TH, MINB>>(h->device, kSmemCap); if (rc != KDME_OK) return rc; }
    if (want_tma) {
        jbf_handle::MapKey& k = lane.map_key;
        if (k.depth != p.depth || k.guide != p.guide4 || k.rows != rows || k.n != p.n_frames || k.gp != p.guide_pitch ||
            k.bx != T::SP || k.by != T::SH) {
            bool ok = encode_map(&lane.map_depth, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, p.depth, p.width, rows, p.n_frames,
                                 (long long)p.width * 4, (long long)p.width * rows * 4, T::SP, T::SH) &&
                      encode_map(&lane.map_guide, CU_TENSOR_MAP_DATA_TYPE_UINT32, p.guide4, p.width, rows, p.n_frames,
                                 (long long)p.guide_pitch * 4, (long long)p.guide_pitch * rows * 4, T::SP, T::SH);
            if (ok) {
                k.depth = p.depth; k.guide = p.guide4; k.rows = rows; k.n = p.n_frames; k.gp = p.guide_pitch;
                k.bx = T::SP; k.by = T::SH;
            } else {
                k = jbf_handle::MapKey();
                want_tma = false;
            }
        }
        if (want_tma) p.mode = kStageTma;
    }
    h->last_variant = (p.mode == kStageTma ? 0x100 : 0) | (TH == 8 ? 0x200 : 0) | (TH == 4 ? 0x800 : 0) | 0x400;
    const int tx = (p.width + TW - 1) / TW;
    int tile_rows = (p.out_rows + TH - 1) / TH;
    p.nbig_rows = INT_MAX; p.ts = 2; p.half_units = 0;
    const long long ctas = (long long)tx * tile_rows * p.n_frames;
    const long long slots = 148LL * MINB;   // CTAs of this instantiation the GPU holds at once
    if (TH > 2 && TH < 16 && ctas <= slots && 2 * ctas > 148) {   // (64x16 kernels: full body only)
        // Less than one wave of tiles (one Kinect frame: 600 tiles of 64x8 on 1184 slots): every SM sub-partition
        // would hold ~4 warps, and at that occupancy a warp's run time is set by the length of its own instruction
        // stream (latency-bound: 61 % issue slots against 72 % with the 8 warps of batch mode).  Every tile goes out
        // as two HALF units instead (jbf_fast_body's PSEL: one pixel pair each; the tile is staged twice, the
        // instruction streams are halves): twice the warps, each half as long -- 72.6 -> 67.9 us per Kinect frame at
        // r = 7.  (Keeping a few tiles whole so that the launch fits one wave is worse, 100 us: a whole tile then
        // takes twice as long as everything around it.)
        p.nbig_rows = 0; p.ts = TH; p.half_units = 1;
        tile_rows = 2 * tile_rows;
    } else if (TH > 2 && ctas < 148LL * 12 && ctas % 148 != 0) {
        // A few waves: keep a whole number of TH-row tiles per SM and cut the image rows left over into 2-row tiles
        // (one warp each), so the surplus spreads over many SMs instead of giving a few SMs one more big tile.
        const long long per_sm = ctas / 148;
        const int nbig = (int)std::min<long long>(tile_rows, (per_sm * 148) / ((long long)tx * p.n_frames));
        const int rem = p.out_rows - nbig * TH;
        if (nbig >= 1 && rem > 0) { p.nbig_rows = nbig; tile_rows = nbig + (rem + p.ts - 1) / p.ts; }
    }
    // A launch of less than one full wave: the block scheduler packs CTAs onto SMs up to the residency limit
    // and leaves the other SMs idle, so the limit is lowered to what the launch needs (ceil(CTAs / 148)) by
    // padding the dynamic shared memory request -- every SM then gets its share.
    size_t smem_bytes = T::SMEM;
    {
        const long long grid_ctas = (long long)tx * tile_rows * p.n_frames;
        int want_res = (int)((grid_ctas + 147) / 148);
        if (want_res < 1) want_res = 1;
        if (want_res < MINB) {
            const size_t padded = (size_t)(228 * 1024) / (size_t)want_res - 1024 - 512;   // 1 KB per CTA is reserved by the system
            if (padded > smem_bytes) smem_bytes = padded > (size_t)kSmemCap ? (size_t)kSmemCap : padded;
        }
    }
    return launch_ex(jbf_fast_kernel<R, TW, TH, MINB>, dim3(tx, tile_rows, p.n_frames), dim3(T::NT), smem_bytes,
                     lane.stream, pdl, lane.map_depth, lane.map_guide, p);
}

#define KDME_FAST_RADII(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15)

static bool fast_radius_available(int r) {
    switch (r) {
#define X(R) case R:
        KDME_FAST_RADII(X)
#undef X
        return true;
        default: return false;
    }
}

// Upsampling runs in gather form (jbf_upsample_gather_kernel, tiles kUpsTW x kUpsTH) on the fast path unless the
// dense form is asked for (KDME_UPSAMPLE_DENSE) or the staged sites of a tile would not fit in shared memory.
// Fills the launch geometry except the lattice pointers.
constexpr int kUpsTW = 64, kUpsTH = 16;
static bool ups_gather_form(const jbf_handle* h, int wl, int hl, int rows, UpsampleGeom* g, size_t* smem) {
    if (!h->fast || getenv("KDME_UPSAMPLE_DENSE")) return false;
    g->radius = h->radius;
    g->ncol_max = (int)(((long long)(kUpsTW + 2 * h->radius) * wl + h->width - 1) / h->width) + 2;
    g->nrow_max = (int)(((long long)(kUpsTH + 2 * h->radius) * hl + rows - 1) / rows) + 2;
    g->ltab1 = h->ltab_ups1_dev;
    g->ltab2 = h->ltab_ups2_dev;
    const int ws = 2 * h->radius + 1;
    *smem = (size_t)g->ncol_max * g->nrow_max * 8 + (size_t)(g->ncol_max + g->nrow_max + 1) * 4 +
            (size_t)ws * (ws + kUpsPad) * 16 + 16;
    return *smem <= 200 * 1024;
}

// The site lattice of (wl, hl) in frames of `rows` rows for the gather form, tabulated once (no 64-bit division is
// left in the kernel): site_x[wl], site_y[hl], tile_xl[tiles_x][2], tile_yl[tiles_y][2], then the inverse maps of
// the fp64 refinement.  Shared by both chunk lanes: a rebuild synchronises the caller's stream (lanes[0]) before it
// frees the old table, so it runs before any chunk is forked to the internal lane.
static int ensure_ups_table(jbf_handle* h, int wl, int hl, int rows) {
    if (h->ups_tab_dev && h->ups_wl == wl && h->ups_hl == hl && h->ups_rows == rows) return KDME_OK;
    const int W = h->width, ntx = (W + kUpsTW - 1) / kUpsTW, nty = (rows + kUpsTH - 1) / kUpsTH;
    std::vector<int> tab((size_t)wl + hl + 2 * (size_t)(ntx + nty) + (size_t)W + rows, -1);
    for (int x = 0; x < wl; ++x) tab[x] = (int)(((2LL * x + 1) * W) / (2LL * wl));
    for (int y = 0; y < hl; ++y) tab[(size_t)wl + y] = (int)(((2LL * y + 1) * rows) / (2LL * hl));
    int* tx = tab.data() + wl + hl;
    int* ty = tx + 2 * ntx;
    for (int b = 0; b < ntx; ++b) {
        tx[2 * b] = upsample_first_site_at_or_after(b * kUpsTW - h->radius, W, wl);
        tx[2 * b + 1] = upsample_first_site_at_or_after(b * kUpsTW + kUpsTW + h->radius, W, wl);
    }
    for (int b = 0; b < nty; ++b) {
        ty[2 * b] = upsample_first_site_at_or_after(b * kUpsTH - h->radius, rows, hl);
        ty[2 * b + 1] = upsample_first_site_at_or_after(b * kUpsTH + kUpsTH + h->radius, rows, hl);
    }
    int* ix = ty + 2 * nty;      // inverse maps (fp64 refinement of upsampled pixels): column -> xl or -1
    int* iy = ix + W;
    for (int x = 0; x < wl; ++x) ix[tab[x]] = x;
    for (int y = 0; y < hl; ++y) iy[tab[(size_t)wl + y]] = y;
    CK(cudaStreamSynchronize(h->lanes[0].stream));
    cudaFree(h->ups_tab_dev);
    h->ups_tab_dev = nullptr;
    CK(cudaMalloc(&h->ups_tab_dev, tab.size() * sizeof(int)));
    CK(cudaMemcpy(h->ups_tab_dev, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice));
    h->ups_wl = wl; h->ups_hl = hl; h->ups_rows = rows;
    return KDME_OK;
}

// The request of a filter launch over n whole frames: rows = out_rows = height, no halos, no low-res input, no
// back-projection, plain mode.  Callers set what their call differs in; launch_filter fills the rest.
static JbfParams filter_request(const jbf_handle* h, const float* depth, const uint32_t* guide4, int guide_pitch,
                                float* out, int n) {
    JbfParams p = {};
    p.width = h->width; p.height = h->height; p.out_rows = h->height; p.n_frames = n;
    p.depth = depth; p.guide4 = guide4; p.guide_pitch = guide_pitch; p.out = out;
    p.mode = kStagePlain;
    return p;
}

// The generic kernel: runtime radius, one pixel per thread (exotic sigmas, radius 0).
static int launch_generic(jbf_handle* h, Lane& lane, const JbfParams& p) {
    JbfGenericParams gp;
    gp.base = p;
    gp.base.ltab = h->ltab_generic_dev;
    gp.radius = h->radius; gp.cd_skip = h->cd_skip; gp.use_color = h->use_color; gp.use_depth = h->use_depth;
    constexpr int TW = 32, TH = 8;
    const int SP = TW + 2 * h->radius, SH = TH + 2 * h->radius, ws = 2 * h->radius + 1;
    size_t smem = (size_t)SP * SH * 8 + (size_t)ws * ws * 4;
    { int rc = allow_dyn_smem<jbf_generic_kernel<TW, TH>>(h->device, 64 * 1024); if (rc != KDME_OK) return rc; }
    dim3 grd((p.width + TW - 1) / TW, (p.out_rows + TH - 1) / TH, p.n_frames);
    jbf_generic_kernel<TW, TH><<<grd, TW * TH, smem, lane.stream>>>(gp);
    CK(cudaGetLastError());
    h->last_variant = 1;
    return KDME_OK;
}

// The fast kernel of the handle's radius, staged by TMA where the buffers allow it.
static int launch_fast(jbf_handle* h, Lane& lane, const JbfParams& p, bool pdl) {
    const bool want_tma = p.mode == kStagePlain && !h->force_no_tma && (h->width % 4 == 0) &&
                          (p.guide_pitch % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.depth) & 15) == 0) &&
                          ((reinterpret_cast<uintptr_t>(p.guide4) & 15) == 0);
    // Tile height: the arithmetic of a pixel does not depend on the tile it falls in, so the choice is
    // purely a scheduling one.  Large launches use 64x16 tiles (least halo per pixel); a launch of only
    // a few waves (one Kinect frame is 300 such tiles on 148 SMs) is cut finer so that the most loaded
    // SM holds as little more than the average as possible.
    const int tx = (h->width + 63) / 64;
    int best_th = 16;
    double best_cost = 1e300;
    const int cand[3] = {16, 8, 4};
    for (int ci = 0; ci < 3; ++ci) {
        const int th = cand[ci];
        const long long ctas = (long long)tx * ((p.out_rows + th - 1) / th) * p.n_frames;
        const long long per_sm = (ctas + 147) / 148;
        const double cost = (double)per_sm * (th + 0.06 * (th + 2 * h->radius) + 0.25);
        if (cost < best_cost * 0.97) { best_cost = cost; best_th = th; }
    }
    if (h->force_tile_h == 16 || h->force_tile_h == 8 || h->force_tile_h == 4) best_th = h->force_tile_h;
    switch (h->radius) {
#define X(R) case R: return best_th == 16 ? launch_fast_rt<R, 16>(h, lane, p, want_tma, pdl)                  \
                          : best_th == 8 ? launch_fast_rt<R, 8>(h, lane, p, want_tma, pdl)                    \
                                         : launch_fast_rt<R, 4>(h, lane, p, want_tma, pdl);
        KDME_FAST_RADII(X)
#undef X
        default: return fail(KDME_ENOTSUP, "no fast kernel for this radius");
    }
}

template <int MAXC>
static int launch_gather_k(const jbf_handle* h, Lane& lane, const JbfParams& p, const UpsampleGeom& g, size_t smem,
                           bool pdl) {
    constexpr int TW = kUpsTW, TH = kUpsTH;
    { int rc = allow_dyn_smem<jbf_upsample_gather_kernel<TW, TH, MAXC>>(h->device, 200 * 1024); if (rc != KDME_OK) return rc; }
    return launch_ex(jbf_upsample_gather_kernel<TW, TH, MAXC>, dim3((p.width + TW - 1) / TW, (p.height + TH - 1) / TH, p.n_frames),
                     dim3((TW / 4) * TH), smem, lane.stream, pdl, p, g);
}

// Upsampling in gather form: only the sites of the low-res lattice are visited (bit-identical to the dense form).
// Also points p at the lattice's inverse maps, which the refinement reads.
static int launch_gather(jbf_handle* h, Lane& lane, JbfParams& p, UpsampleGeom g, size_t smem, bool pdl) {
    const int rows = p.height, wl = p.wl, hl = p.hl;
    const int ntx = (p.width + kUpsTW - 1) / kUpsTW, nty = (rows + kUpsTH - 1) / kUpsTH;
    // built by the caller, on its own stream, before any chunk went to the internal lane
    if (!h->ups_tab_dev || h->ups_wl != wl || h->ups_hl != hl || h->ups_rows != rows)
        return fail(KDME_EINVAL, "upsampling: the site lattice was not built for this size");
    g.site_x = h->ups_tab_dev; g.site_y = h->ups_tab_dev + wl;
    g.tile_xl = h->ups_tab_dev + wl + hl; g.tile_yl = g.tile_xl + 2 * ntx;
    p.ups_inv_x = g.tile_yl + 2 * nty; p.ups_inv_y = p.ups_inv_x + p.width;
    // site columns any thread can see: lattice points in 2r + 4 consecutive pixels
    const int maxc = (int)(((long long)(2 * h->radius + 4) * wl + h->width - 1) / h->width);
    const bool loop = getenv("KDME_GATHER_GENERIC") != nullptr;   // the runtime column loop at any maxc
    const int rc = !loop && maxc <= 5 ? launch_gather_k<5>(h, lane, p, g, smem, pdl)
                 : !loop && maxc <= 8 ? launch_gather_k<8>(h, lane, p, g, smem, pdl)
                                      : launch_gather_k<0>(h, lane, p, g, smem, pdl);
    if (rc != KDME_OK) return rc;
    h->last_variant = 0x1000 | 0x400;
    return KDME_OK;
}

// fp64 re-evaluation of the queued pixels; launched with programmatic stream serialisation so its launch latency
// hides behind the filter (it waits for the filter's completion on the device).
static int launch_refine(const jbf_handle* h, Lane& lane, const JbfParams& p) {
    const bool plain = p.mode != kStageUpsample && !p.depth_up && !p.depth_dn;
    auto launch = [&](auto kern) { return launch_ex(kern, dim3(148 * 5), dim3(128), 0, lane.stream, true, p, h->radius); };
    if (h->radius <= 7) return plain ? launch(jbf_refine_kernel<8, true>) : launch(jbf_refine_kernel<8, false>);
    if (h->radius <= 10) return plain ? launch(jbf_refine_kernel<16, true>) : launch(jbf_refine_kernel<16, false>);
    return plain ? launch(jbf_refine_kernel<31, true>) : launch(jbf_refine_kernel<31, false>);
}

// Launches request p on `lane`: its stream, refinement queue and TMA descriptors.
static int launch_filter(jbf_handle* h, Lane& lane, JbfParams p, bool pdl) {
    if ((p.depth_up || p.depth_dn) && !h->fast)
        return fail(KDME_ENOTSUP, "peer-memory halos are implemented for the fast kernel (default sigmas, r = 1..15)");
    if (p.xyz && !h->fast) return fail(KDME_ENOTSUP, "the fused back-projection needs the fast kernel (default sigmas, r = 1..15)");
    const int rows = p.height, wl = p.wl, hl = p.hl;
    p.depth_frame_stride = (long long)h->width * rows;
    p.guide_frame_stride = (long long)p.guide_pitch * rows;
    p.lo_frame_stride = (long long)wl * hl;
    p.nkc = h->nkc; p.sq = h->sq; p.inv_sq = h->inv_sq; p.e_thr = h->e_thr;
    p.flag_scale = h->flag_scale; p.kc = h->kc; p.kd = h->kd; p.slut = h->slut_dev; p.stats = h->stats_dev;
    p.q_count = lane.q_count_dev + lane.q_cur; p.q_count_prev = lane.q_count_dev + (lane.q_cur ^ 1);
    p.q_items = lane.q_items_dev; p.q_capacity = (unsigned)lane.q_capacity;
    if (!h->fast) return launch_generic(h, lane, p);
    p.ltab_pairs = h->ltab_pairs_dev;
    p.ltab_pairs1 = h->ltab_pairs1_dev;
    // queue of ill-conditioned pixels: a quarter of the launch's pixels (at least 64 K entries); pixels
    // beyond it keep their fp32 value and are counted (jbf_refine_stats)
    const unsigned long long px = (unsigned long long)h->width * p.out_rows * p.n_frames;
    if (px > 0xFFFFFFFFull) return fail(KDME_ENOTSUP, "more than 2^32 pixels in one launch");
    size_t want = (size_t)std::min<unsigned long long>(std::max<unsigned long long>(px / 4, 65536ull), px);
    if (h->flag_scale > 0.f && want > lane.q_capacity) {
        CK(cudaStreamSynchronize(lane.stream));
        cudaFree(lane.q_items_dev);
        lane.q_items_dev = nullptr; lane.q_capacity = 0;
        CK(cudaMalloc(&lane.q_items_dev, want * sizeof(unsigned int)));
        lane.q_capacity = want;
    }
    p.q_items = lane.q_items_dev; p.q_capacity = (unsigned)lane.q_capacity;
    UpsampleGeom g;
    size_t smem = 0;
    const int rc = p.mode == kStageUpsample && ups_gather_form(h, wl, hl, rows, &g, &smem)
                       ? launch_gather(h, lane, p, g, smem, pdl) : launch_fast(h, lane, p, pdl);
    if (rc != KDME_OK) return rc;
    lane.q_cur ^= 1;
    return h->flag_scale > 0.f ? launch_refine(h, lane, p) : KDME_OK;
}

extern "C" int jbf_presmooth(jbf_handle* h, const uint8_t* bgr_dev, size_t bgr_step, uint8_t* guide4_dev,
                             size_t guide_step, int n_frames) {
    if (!h || !bgr_dev || !guide4_dev) return fail(KDME_EINVAL, "jbf_presmooth: NULL argument");
    if (n_frames < 1) return fail(KDME_EINVAL, "jbf_presmooth: n_frames must be >= 1");
    int pitch = 0;
    { int rc = guide4_step(h, &guide_step, &pitch, "jbf_presmooth"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    return launch_presmooth(h, h->lanes[0], bgr_dev, bgr_step, reinterpret_cast<uint32_t*>(guide4_dev), pitch, n_frames);
}

extern "C" int jbf_filter_guide4(jbf_handle* h, const float* depth_dev, const uint8_t* guide4_dev, size_t guide_step,
                                 float* out_dev, int n_frames) {
    if (!h || !depth_dev || !guide4_dev || !out_dev) return fail(KDME_EINVAL, "jbf_filter_guide4: NULL argument");
    if (n_frames < 1 || n_frames > 65535) return fail(KDME_EINVAL, "jbf_filter_guide4: n_frames must be in [1, 65535] (frames are grid.z of one launch)");
    if (depth_dev == out_dev) return fail(KDME_EINVAL, "jbf_filter_guide4: in-place operation is not supported");
    int pitch = 0;
    { int rc = guide4_step(h, &guide_step, &pitch, "jbf_filter_guide4"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    return launch_filter(h, h->lanes[0],
                         filter_request(h, depth_dev, reinterpret_cast<const uint32_t*>(guide4_dev), pitch, out_dev, n_frames),
                         /*pdl=*/false);
}

extern "C" int jbf_presmooth_rows(jbf_handle* h, const uint8_t* bgr_dev, size_t bgr_step, uint8_t* guide4_dev,
                                  size_t guide_step, int rows) {
    if (!h || !bgr_dev || !guide4_dev) return fail(KDME_EINVAL, "jbf_presmooth_rows: NULL argument");
    if (rows < 1) return fail(KDME_EINVAL, "jbf_presmooth_rows: rows must be >= 1");
    int pitch = 0;
    { int rc = guide4_step(h, &guide_step, &pitch, "jbf_presmooth_rows"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    return launch_presmooth(h, h->lanes[0], bgr_dev, bgr_step, reinterpret_cast<uint32_t*>(guide4_dev), pitch, 1, rows);
}

extern "C" int jbf_filter_rows(jbf_handle* h, const float* depth_dev, const uint8_t* guide4_dev, size_t guide_step,
                               float* out_dev, int rows, int y_off, int out_rows) {
    if (!h || !depth_dev || !guide4_dev || !out_dev) return fail(KDME_EINVAL, "jbf_filter_rows: NULL argument");
    if (rows < 1 || y_off < 0 || out_rows < 1 || y_off + out_rows > rows)
        return fail(KDME_EINVAL, "jbf_filter_rows: need 0 <= y_off and y_off + out_rows <= rows");
    int pitch = 0;
    { int rc = guide4_step(h, &guide_step, &pitch, "jbf_filter_rows"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    JbfParams p = filter_request(h, depth_dev, reinterpret_cast<const uint32_t*>(guide4_dev), pitch, out_dev, 1);
    p.height = rows; p.y_off = y_off; p.out_rows = out_rows;
    return launch_filter(h, h->lanes[0], p, /*pdl=*/false);
}

// Row bands with the halos read from the neighbour GPUs' memory inside the kernels (NVLink peer loads):
// the arrays hold `rows` rows of which [band0, band1) are this rank's own; *_up / *_dn are peer-mapped
// pointers positioned so that row r < band0 is  up + r * pitch  and row r >= band1 is  dn + (r - band1) * pitch.
extern "C" int jbf_presmooth_rows_p2p(jbf_handle* h, const uint8_t* bgr_dev, size_t bgr_step, uint8_t* guide4_dev,
                                      size_t guide_step, int rows, int band0, int band1, const uint8_t* bgr_up,
                                      const uint8_t* bgr_dn) {
    if (!h || !bgr_dev || !guide4_dev) return fail(KDME_EINVAL, "jbf_presmooth_rows_p2p: NULL argument");
    if (rows < 1 || band0 < 0 || band1 > rows || band0 >= band1)
        return fail(KDME_EINVAL, "jbf_presmooth_rows_p2p: need 0 <= band0 < band1 <= rows");
    int pitch = 0;
    { int rc = guide4_step(h, &guide_step, &pitch, "jbf_presmooth_rows_p2p"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    return launch_presmooth(h, h->lanes[0], bgr_dev, bgr_step, reinterpret_cast<uint32_t*>(guide4_dev), pitch, 1, rows,
                            bgr_up, bgr_dn, band0, band1);
}

extern "C" int jbf_filter_rows_p2p(jbf_handle* h, const float* depth_dev, const uint8_t* guide4_dev, size_t guide_step,
                                   float* out_dev, int rows, int y_off, int out_rows, int band0, int band1,
                                   const float* depth_up, const float* depth_dn) {
    if (!h || !depth_dev || !guide4_dev || !out_dev) return fail(KDME_EINVAL, "jbf_filter_rows_p2p: NULL argument");
    if (rows < 1 || y_off < 0 || out_rows < 1 || y_off + out_rows > rows || band0 < 0 || band1 > rows || band0 >= band1)
        return fail(KDME_EINVAL, "jbf_filter_rows_p2p: bad row ranges");
    int pitch = 0;
    { int rc = guide4_step(h, &guide_step, &pitch, "jbf_filter_rows_p2p"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    JbfParams p = filter_request(h, depth_dev, reinterpret_cast<const uint32_t*>(guide4_dev), pitch, out_dev, 1);
    p.height = rows; p.y_off = y_off; p.out_rows = out_rows;
    p.depth_up = depth_up; p.depth_dn = depth_dn; p.band0 = band0; p.band1 = band1;
    return launch_filter(h, h->lanes[0], p, /*pdl=*/false);
}

// The chunk loop of the batched calls: chunks of `chunk` frames, fn(lane, c, f0, n) enqueues chunk c, frames
// [f0, f0 + n), on `lane`.  With more than one chunk on the fast path, the chunks alternate between the caller's
// stream (lanes[0]) and the internal lane (lanes[1]), which is forked from the caller's stream before the first
// chunk and joined back into it after the last, so the call keeps the caller's stream semantics.
template <class Fn>
static int run_chunks(jbf_handle* h, int n_frames, int chunk, Fn&& fn) {
    const bool two = n_frames > chunk && !h->one_lane && h->fast;
    Lane &l0 = h->lanes[0], &l1 = h->lanes[1];
    if (two) {
        int rc = ensure_alt_lane(h);
        if (rc != KDME_OK) return rc;
        CK(cudaEventRecord(h->ev_fork, l0.stream));
        CK(cudaStreamWaitEvent(l1.stream, h->ev_fork, 0));
    }
    for (int c = 0, f0 = 0; f0 < n_frames; f0 += chunk, ++c) {
        int rc = fn(two && (c & 1) ? l1 : l0, c, f0, std::min(chunk, n_frames - f0));
        if (rc != KDME_OK) return rc;
    }
    if (two) {
        CK(cudaEventRecord(h->ev_join, l1.stream));
        CK(cudaStreamWaitEvent(l0.stream, h->ev_join, 0));
    }
    return KDME_OK;
}

extern "C" int jbf_process_batch(jbf_handle* h, const float* depth_dev, const uint8_t* bgr_dev, size_t bgr_step,
                                 float* out_dev, int n_frames) {
    if (!h || !depth_dev || !bgr_dev || !out_dev) return fail(KDME_EINVAL, "jbf_process_batch: NULL argument");
    if (n_frames < 1) return fail(KDME_EINVAL, "jbf_process_batch: n_frames must be >= 1");
    { int rc = guide_step(h, &bgr_step, "jbf_process_batch"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    const size_t plane = (size_t)h->width * h->height;
    return run_chunks(h, n_frames, h->max_batch, [&](Lane& lane, int, int f0, int n) {
        int rc = launch_presmooth(h, lane, bgr_dev + (size_t)f0 * bgr_step * h->height, bgr_step, lane.guide4,
                                  h->guide_pitch, n);
        if (rc != KDME_OK) return rc;
        return launch_filter(h, lane, filter_request(h, depth_dev + (size_t)f0 * plane, lane.guide4, h->guide_pitch,
                                                     out_dev + (size_t)f0 * plane, n), /*pdl=*/true);
    });
}

extern "C" int jbf_process(jbf_handle* h, const float* depth_dev, const uint8_t* bgr_dev, size_t bgr_step) {
    if (!h) return fail(KDME_EINVAL, "jbf_process: NULL handle");
    return jbf_process_batch(h, depth_dev, bgr_dev, bgr_step, h->filtered_dev, 1);
}

// Process + DimensionConvertor::projectiveToReal in one launch pair (main.cpp:179 + :182,
// KinectDepthEnhancement.cpp:59-60): the filter's epilogue writes the float3 cloud beside the depth plane.
extern "C" int jbf_process_xyz(jbf_handle* h, const float* depth_dev, const uint8_t* bgr_dev, size_t bgr_step,
                               float* xyz_dev, float fx, float fy, int cx, int cy) {
    if (!h || !depth_dev || !bgr_dev || !xyz_dev) return fail(KDME_EINVAL, "jbf_process_xyz: NULL argument");
    if (!(fx != 0.f) || !(fy != 0.f)) return fail(KDME_EINVAL, "jbf_process_xyz: focal lengths must be non-zero");
    if (!h->fast) {   // exotic sigmas / radius 0 (generic kernel): the two calls the reference makes, back to back
        int rc2 = jbf_process_batch(h, depth_dev, bgr_dev, bgr_step, h->filtered_dev, 1);
        if (rc2 != KDME_OK) return rc2;
        DeviceGuard g(h->device);
        return kdme_projective_to_real(h->filtered_dev, xyz_dev, h->width, h->height, fx, fy, cx, cy, h->lanes[0].stream);
    }
    { int rc = guide_step(h, &bgr_step, "jbf_process_xyz"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    Lane& lane = h->lanes[0];   // one frame: one chunk, on the caller's stream
    int rc = launch_presmooth(h, lane, bgr_dev, bgr_step, lane.guide4, h->guide_pitch, 1);
    if (rc != KDME_OK) return rc;
    JbfParams p = filter_request(h, depth_dev, lane.guide4, h->guide_pitch, h->filtered_dev, 1);
    p.xyz = xyz_dev; p.fx = fx; p.fy = fy; p.cx = cx; p.cy = cy;
    return launch_filter(h, lane, p, /*pdl=*/true);
}

// Pixels re-evaluated in fp64 (ill-conditioned: no sample near the pass-1 mean) and pixels dropped because
// the queue was full, since the previous call.  Synchronises the handle's stream.
extern "C" int jbf_refine_stats(jbf_handle* h, unsigned long long* refined, unsigned long long* dropped) {
    if (!h) return fail(KDME_EINVAL, "jbf_refine_stats: NULL handle");
    DeviceGuard g(h->device);
    unsigned long long v[2] = {0, 0};
    CK(cudaMemcpyAsync(v, h->stats_dev, sizeof(v), cudaMemcpyDeviceToHost, h->lanes[0].stream));
    CK(cudaMemsetAsync(h->stats_dev, 0, sizeof(v), h->lanes[0].stream));
    CK(cudaStreamSynchronize(h->lanes[0].stream));
    if (refined) *refined = v[0];
    if (dropped) *dropped = v[1];
    return KDME_OK;
}

// n_frames Upsampling calls; the low-res depth is float (depth_lo) or uint16 (depth_lo16), the other one is NULL
static int upsample_batch(jbf_handle* h, const float* depth_lo, const uint16_t* depth_lo16, int wl, int hl,
                          const uint8_t* bgr_dev, size_t bgr_step, float* out_dev, int n_frames, const char* who) {
    if (!h || !(depth_lo || depth_lo16) || !bgr_dev || !out_dev) return fail(KDME_EINVAL, std::string(who) + ": NULL argument");
    if (n_frames < 1) return fail(KDME_EINVAL, std::string(who) + ": n_frames must be >= 1");
    if (wl <= 0 || hl <= 0 || wl > h->width || hl > h->height)
        return fail(KDME_EINVAL, std::string(who) + ": low-res size must be positive and <= the handle's size");
    { int rc = guide_step(h, &bgr_step, who); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    UpsampleGeom geom;
    size_t smem = 0;
    if (ups_gather_form(h, wl, hl, h->height, &geom, &smem)) {
        int rc = ensure_ups_table(h, wl, hl, h->height);
        if (rc != KDME_OK) return rc;
    }
    const size_t plane = (size_t)h->width * h->height, lo_plane = (size_t)wl * hl;
    return run_chunks(h, n_frames, h->max_batch, [&](Lane& lane, int, int f0, int n) {
        int rc = launch_presmooth(h, lane, bgr_dev + (size_t)f0 * bgr_step * h->height, bgr_step, lane.guide4,
                                  h->guide_pitch, n);
        if (rc != KDME_OK) return rc;
        JbfParams p = filter_request(h, nullptr, lane.guide4, h->guide_pitch, out_dev + (size_t)f0 * plane, n);
        p.mode = kStageUpsample; p.wl = wl; p.hl = hl;
        p.depth_lo = depth_lo ? depth_lo + (size_t)f0 * lo_plane : nullptr;
        p.depth_lo16 = depth_lo16 ? depth_lo16 + (size_t)f0 * lo_plane : nullptr;
        return launch_filter(h, lane, p, /*pdl=*/true);
    });
}

extern "C" int jbf_upsample_batch(jbf_handle* h, const float* depth_lo_dev, int wl, int hl, const uint8_t* bgr_hi_dev,
                                  size_t bgr_step, float* out_hi_dev, int n_frames) {
    return upsample_batch(h, depth_lo_dev, nullptr, wl, hl, bgr_hi_dev, bgr_step, out_hi_dev, n_frames,
                          "jbf_upsample_batch");
}

extern "C" int jbf_upsample_batch_u16(jbf_handle* h, const uint16_t* depth_lo_dev, int wl, int hl,
                                      const uint8_t* bgr_hi_dev, size_t bgr_step, float* out_hi_dev, int n_frames) {
    return upsample_batch(h, nullptr, depth_lo_dev, wl, hl, bgr_hi_dev, bgr_step, out_hi_dev, n_frames,
                          "jbf_upsample_batch_u16");
}

extern "C" int jbf_upsample(jbf_handle* h, const float* depth_lo_dev, int wl, int hl, const uint8_t* bgr_hi_dev,
                            size_t bgr_step, float* out_hi_dev) {
    return jbf_upsample_batch(h, depth_lo_dev, wl, hl, bgr_hi_dev, bgr_step, out_hi_dev, 1);
}

// Host pipeline: kPipeDepth device slots of pipe_chunk frames each; H2D, compute and D2H run on three
// streams so that, in steady state, the upload of chunk c+1 and the download of chunk c-1 overlap the
// filter of chunk c.  Small chunks keep the fill/drain bubble short.
static int ensure_pipe(jbf_handle* h, size_t bgr_step) {
    if (h->s_h2d && h->pipe_bgr_step == bgr_step) return KDME_OK;
    if (h->s_h2d && h->pipe_bgr_step != bgr_step) {
        for (int b = 0; b < kPipeDepth; b++) { cudaFree(h->pipe_bgr[b]); h->pipe_bgr[b] = nullptr; }
    }
    const size_t plane = (size_t)h->width * h->height;
    if (!h->s_h2d) {
        // ~5 Mpixel per chunk (16 Kinect frames): enough CTAs to fill the GPU, short pipeline bubble
        long long want = (5LL << 20) / (long long)plane;
        if (want < 1) want = 1;
        h->pipe_chunk = (int)((want < h->max_batch) ? want : h->max_batch);
        CK(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
        for (int b = 0; b < kPipeDepth; b++) {
            CK(cudaEventCreateWithFlags(&h->ev_in[b], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->ev_done[b], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->ev_free[b], cudaEventDisableTiming));
            CK(cudaMalloc(&h->pipe_depth[b], plane * h->pipe_chunk * sizeof(float)));
            CK(cudaMalloc(&h->pipe_out[b], plane * h->pipe_chunk * sizeof(float)));
        }
    }
    for (int b = 0; b < kPipeDepth; b++) CK(cudaMalloc(&h->pipe_bgr[b], bgr_step * h->height * h->pipe_chunk));
    h->pipe_bgr_step = bgr_step;
    return KDME_OK;
}

static int process_host_impl(jbf_handle* h, const float* depth_host, const uint16_t* depth16_host,
                             const uint8_t* bgr_host, size_t bgr_step, float* out_host, int n_frames) {
    { int rc = guide_step(h, &bgr_step, "jbf_process_host"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    int rc = ensure_pipe(h, bgr_step);   // re-sizes the guide slots when the guide's row bytes change
    if (rc != KDME_OK) return rc;
    const size_t plane = (size_t)h->width * h->height;
    const size_t bgr_frame = bgr_step * h->height;
    if (depth16_host)
        for (int b = 0; b < kPipeDepth; b++)
            if (!h->pipe_depth16[b]) CK(cudaMalloc(&h->pipe_depth16[b], plane * h->pipe_chunk * sizeof(uint16_t)));
    rc = run_chunks(h, n_frames, h->pipe_chunk, [&](Lane& lane, int c, int f0, int n) {
        const int b = c % kPipeDepth;
        if (c >= kPipeDepth) CK(cudaStreamWaitEvent(h->s_h2d, h->ev_done[b], 0));  // slot inputs consumed
        if (depth16_host)
            CK(cudaMemcpyAsync(h->pipe_depth16[b], depth16_host + (size_t)f0 * plane, plane * n * sizeof(uint16_t),
                               cudaMemcpyHostToDevice, h->s_h2d));
        else
            CK(cudaMemcpyAsync(h->pipe_depth[b], depth_host + (size_t)f0 * plane, plane * n * sizeof(float),
                               cudaMemcpyHostToDevice, h->s_h2d));
        CK(cudaMemcpyAsync(h->pipe_bgr[b], bgr_host + (size_t)f0 * bgr_frame, bgr_frame * n, cudaMemcpyHostToDevice,
                           h->s_h2d));
        CK(cudaEventRecord(h->ev_in[b], h->s_h2d));
        CK(cudaStreamWaitEvent(lane.stream, h->ev_in[b], 0));
        if (c >= kPipeDepth) CK(cudaStreamWaitEvent(lane.stream, h->ev_free[b], 0));  // slot output drained
        if (depth16_host) {   // sensor millimetres -> float, as Buffer2D::insertData(xn::DepthMetaData*) does (Buffer2D.cpp:18-32)
            const long long cnt = (long long)plane * n;
            u16_to_f32_kernel<<<buf_blocks(cnt), 256, 0, lane.stream>>>(h->pipe_depth16[b], h->pipe_depth[b], cnt);
            CK(cudaGetLastError());
        }
        int rc = launch_presmooth(h, lane, h->pipe_bgr[b], bgr_step, lane.guide4, h->guide_pitch, n);
        if (rc != KDME_OK) return rc;
        rc = launch_filter(h, lane, filter_request(h, h->pipe_depth[b], lane.guide4, h->guide_pitch, h->pipe_out[b], n),
                           /*pdl=*/true);
        if (rc != KDME_OK) return rc;
        CK(cudaEventRecord(h->ev_done[b], lane.stream));
        CK(cudaStreamWaitEvent(h->s_d2h, h->ev_done[b], 0));
        CK(cudaMemcpyAsync(out_host + (size_t)f0 * plane, h->pipe_out[b], plane * n * sizeof(float),
                           cudaMemcpyDeviceToHost, h->s_d2h));
        CK(cudaEventRecord(h->ev_free[b], h->s_d2h));
        return KDME_OK;
    });
    if (rc != KDME_OK) return rc;
    CK(cudaStreamSynchronize(h->s_d2h));
    CK(cudaStreamSynchronize(h->lanes[0].stream));
    return KDME_OK;
}

extern "C" int jbf_process_host(jbf_handle* h, const float* depth_host, const uint8_t* bgr_host, size_t bgr_step,
                                float* out_host, int n_frames) {
    if (!h || !depth_host || !bgr_host || !out_host) return fail(KDME_EINVAL, "jbf_process_host: NULL argument");
    if (n_frames < 1) return fail(KDME_EINVAL, "jbf_process_host: n_frames must be >= 1");
    return process_host_impl(h, depth_host, nullptr, bgr_host, bgr_step, out_host, n_frames);
}

extern "C" int jbf_process_host_u16(jbf_handle* h, const uint16_t* depth_host, const uint8_t* bgr_host, size_t bgr_step,
                                    float* out_host, int n_frames) {
    if (!h || !depth_host || !bgr_host || !out_host) return fail(KDME_EINVAL, "jbf_process_host_u16: NULL argument");
    if (n_frames < 1) return fail(KDME_EINVAL, "jbf_process_host_u16: n_frames must be >= 1");
    return process_host_impl(h, nullptr, depth_host, bgr_host, bgr_step, out_host, n_frames);
}

// Page-locked host memory for the buffers of jbf_process_host*: write-combined memory is read by the copy
// engine without snooping the CPU caches (for buffers the CPU only writes, front to back: sensor frames);
// the result buffer must be ordinary pinned memory (the CPU reads it).
extern "C" void* kdme_host_alloc(size_t bytes, int write_combined) {
    void* p = nullptr;
    const unsigned flags = cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0u);
    cudaError_t e = cudaHostAlloc(&p, bytes, flags);
    if (e != cudaSuccess) { fail(-(int)e, std::string("kdme_host_alloc: ") + cudaGetErrorString(e)); return nullptr; }
    return p;
}
extern "C" void kdme_host_free(void* p) { if (p) cudaFreeHost(p); }

extern "C" float* jbf_filtered_device(jbf_handle* h) { return h ? h->filtered_dev : nullptr; }

extern "C" const float* jbf_filtered_host(jbf_handle* h) {
    if (!h) { fail(KDME_EINVAL, "jbf_filtered_host: NULL handle"); return nullptr; }
    DeviceGuard g(h->device);
    const size_t bytes = (size_t)h->width * h->height * sizeof(float);
    if (!h->filtered_host && cudaMallocHost(&h->filtered_host, bytes) != cudaSuccess) {
        fail(KDME_EINVAL, "jbf_filtered_host: cudaMallocHost failed");
        return nullptr;
    }
    cudaStream_t st = h->lanes[0].stream;
    if (cudaMemcpyAsync(h->filtered_host, h->filtered_dev, bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
        fail(KDME_EINVAL, "jbf_filtered_host: D2H copy failed");
        return nullptr;
    }
    return h->filtered_host;
}

extern "C" const uint8_t* jbf_guide4_device(jbf_handle* h, size_t* step) {
    if (!h) return nullptr;
    if (step) *step = (size_t)h->guide_pitch * 4;
    return reinterpret_cast<const uint8_t*>(h->lanes[0].guide4);
}

extern "C" const uint8_t* jbf_smooth_device(jbf_handle* h, size_t* step) {
    if (!h) return nullptr;
    DeviceGuard g(h->device);
    const Lane& l0 = h->lanes[0];   // the guide of the last jbf_process
    const int C = h->guide_channels;
    const size_t bytes = (size_t)h->width * h->height * C;
    if (h->smooth_bytes != bytes) {
        if (h->smooth_bgr && cudaStreamSynchronize(l0.stream) != cudaSuccess) {
            fail(KDME_EINVAL, "jbf_smooth_device: stream synchronisation failed");
            return nullptr;
        }
        cudaFree(h->smooth_bgr);
        h->smooth_bgr = nullptr; h->smooth_bytes = 0;
        if (cudaMalloc(&h->smooth_bgr, bytes) != cudaSuccess) {
            fail(KDME_EINVAL, "jbf_smooth_device: cudaMalloc failed");
            return nullptr;
        }
        h->smooth_bytes = bytes;
    }
    dim3 blk(128), grd((h->width + 127) / 128, h->height);
    with_channels(C, [&](auto c) {
        guide4_to_image_kernel<decltype(c)::value><<<grd, blk, 0, l0.stream>>>(l0.guide4, h->guide_pitch, h->smooth_bgr,
                                                                              h->width, h->height);
    });
    if (step) *step = (size_t)h->width * C;
    return h->smooth_bgr;
}

extern "C" int jbf_kernel_variant(jbf_handle* h) { return h ? ((h->fast ? 0 : 1) | (h->last_variant & 0x1F00)) : -1; }

// ------------------------------------------------------------------ MRF (next row f1)
extern "C" int jbf_mrf(jbf_handle* h, const float* depth_dev, const uint8_t* bgr_dev, size_t bgr_step, float* out_dev,
                       int window_radius, float color_sigma, float smooth_sigma) {
    if (!h || !depth_dev || !bgr_dev || !out_dev) return fail(KDME_EINVAL, "jbf_mrf: NULL argument");
    if (window_radius < 0 || window_radius > KDME_MAX_RADIUS) return fail(KDME_EINVAL, "jbf_mrf: bad radius");
    if (depth_dev == out_dev) return fail(KDME_EINVAL, "jbf_mrf: in-place operation is not supported");
    { int rc = guide_step(h, &bgr_step, "jbf_mrf"); if (rc != KDME_OK) return rc; }
    DeviceGuard g(h->device);
    Lane& l0 = h->lanes[0];
    launch_guide4_convert(h, l0, bgr_dev, bgr_step, 0, l0.guide4, h->guide_pitch, 0, h->height, 1);
    CK(cudaGetLastError());
    constexpr int TW = 32, TH = 8;
    const int SP = TW + 2 * window_radius, SH = TH + 2 * window_radius;
    dim3 g2((h->width + TW - 1) / TW, (h->height + TH - 1) / TH);
    mrf_kernel<TW, TH><<<g2, TW * TH, (size_t)SP * SH * 8, l0.stream>>>(depth_dev, l0.guide4, h->guide_pitch, out_dev,
                                                                        h->width, h->height, window_radius,
                                                                        color_sigma, smooth_sigma);
    CK(cudaGetLastError());
    return KDME_OK;
}

extern "C" int kdme_projective_to_real(const float* depth_dev, float* xyz_dev, int width, int height, float fx,
                                       float fy, int cx, int cy, void* stream) {
    if (!depth_dev || !xyz_dev || width <= 0 || height <= 0) return fail(KDME_EINVAL, "projective_to_real: bad argument");
    { int rcd = check_pointer_device(depth_dev, "kdme_projective_to_real"); if (rcd != KDME_OK) return rcd; }
    const long long n = (long long)width * height;
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    projective_to_real_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(depth_dev, xyz_dev, width, height, fx, fy, cx, cy);
    CK(cudaGetLastError());
    return KDME_OK;
}

// ------------------------------------------------------------------ next rows f2, f4
extern "C" int kdme_depth_bilateral_xyz(const float* normalized_dev, const float* in_dev, float* out_dev, int width,
                                        int height, int window_radius, float sigma_spatial, float sigma_depth,
                                        void* stream) {
    if (!normalized_dev || !in_dev || !out_dev) return fail(KDME_EINVAL, "kdme_depth_bilateral_xyz: NULL argument");
    if (in_dev == out_dev) return fail(KDME_EINVAL, "kdme_depth_bilateral_xyz: in-place operation is not supported");
    if (width <= 0 || height <= 0 || window_radius < 0 || window_radius > KDME_MAX_RADIUS || !(sigma_spatial > 0) ||
        !(sigma_depth > 0))
        return fail(KDME_EINVAL, "kdme_depth_bilateral_xyz: bad size, radius or sigma");
    int rcd = check_pointer_device(in_dev, "kdme_depth_bilateral_xyz");
    if (rcd != KDME_OK) return rcd;
    const int ws = 2 * window_radius + 1;
    cudaStream_t st = (cudaStream_t)stream;
    // spatial LUT, cached per (device, window, sigma): built and uploaded once
    static std::mutex mu;
    static std::map<std::tuple<int, int, float>, float*> cache;
    float* stab = nullptr;
    {
        int cur = 0;
        CK(cudaGetDevice(&cur));
        std::lock_guard<std::mutex> lk(mu);
        auto key = std::make_tuple(cur, ws, sigma_spatial);
        auto it = cache.find(key);
        if (it == cache.end()) {
            std::vector<float> lut;
            host_spatial_lut(lut, ws, sigma_spatial);
            CK(cudaMalloc(&stab, lut.size() * sizeof(float)));
            CK(cudaMemcpy(stab, lut.data(), lut.size() * sizeof(float), cudaMemcpyHostToDevice));
            cache[key] = stab;
        } else {
            stab = it->second;
        }
    }
    constexpr int TW = 32, TH = 8;
    const int SP = TW + 2 * window_radius, SH = TH + 2 * window_radius;
    dim3 grd((width + TW - 1) / TW, (height + TH - 1) / TH);
    const double nkd = -kLog2e / (2.0 * (double)sigma_depth * (double)sigma_depth);
    depth_bilateral_xyz_kernel<TW, TH><<<grd, TW * TH, (size_t)SP * SH * 12 + (size_t)ws * ws * 8, st>>>(
        normalized_dev, in_dev, out_dev, stab, width, height, window_radius, (float)nkd, (float)(nkd - (float)nkd),
        (float)(std::sqrt(2.0 * kExpZeroArg) * (double)sigma_depth));
    CK(cudaGetLastError());
    return KDME_OK;
}

extern "C" int kdme_mean_3d_error(const float* points_dev, const float* truth_dev, long long n_points,
                                  double* mean_out, long long* count_out, void* stream) {
    if (!points_dev || !truth_dev || !mean_out || n_points <= 0)
        return fail(KDME_EINVAL, "kdme_mean_3d_error: bad argument");
    { int rcd = check_pointer_device(points_dev, "kdme_mean_3d_error"); if (rcd != KDME_OK) return rcd; }
    cudaStream_t st = (cudaStream_t)stream;
    double* acc = nullptr;
    CK(cudaMallocAsync(&acc, 2 * sizeof(double), st));
    CK(cudaMemsetAsync(acc, 0, 2 * sizeof(double), st));
    long long blocks = (n_points + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    mean_3d_error_kernel<<<(int)blocks, 256, 0, st>>>(points_dev, truth_dev, n_points, acc);
    CK(cudaGetLastError());
    double host[2] = {0, 0};
    CK(cudaMemcpyAsync(host, acc, sizeof(host), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaFreeAsync(acc, st));
    *mean_out = (host[1] > 0) ? host[0] / host[1] : 0.0;
    if (count_out) *count_out = (long long)host[1];
    return KDME_OK;
}

// ------------------------------------------------------------------ guided fill
// One guided call over n_frames frames stored back to back.  The depth is exactly one of depth / depth16 (the fill:
// width x height samples per frame) or depth_lo / depth_lo16 (the upsampling: wl x hl samples per frame).
struct GuidedCall {
    const float* depth; const uint16_t* depth16;
    const float* depth_lo; const uint16_t* depth_lo16; int wl, hl;
    const int32_t* labels; const uint8_t* bgr; size_t bgr_step;
    float* out; int width, height, n_frames, radius;
    float sigma_s, sigma_c, sigma_d;
};

constexpr int kGuidedTW = 32, kGuidedTH = 8;
constexpr int kMaxGridZ = 65535;   // gridDim.z limit: frames per launch

template <class T>
static T* advance(T* ptr, long long n) { return ptr ? ptr + n : ptr; }

// 1 / (2 sigma^2) in double, as the fp64 oracle forms it; 0 for sigma = 0, where the reference skips the factor.
static double guided_k(float sigma) { return (sigma != 0.0f) ? 1.0 / (2.0 * (double)sigma * (double)sigma) : 0.0; }

// The kernel's parameters for the whole call: image, pointers, per-frame strides, sigmas and spatial factors.
template <int WS_CT>
static GuidedParams<WS_CT> guided_params(const GuidedCall& c) {
    static_assert(2 * KDME_MAX_RADIUS + 1 <= 31, "GuidedParams<0> holds a window of at most 31 x 31 factors");
    GuidedParams<WS_CT> p;
    const long long plane = (long long)c.width * c.height;
    p.width = c.width; p.height = c.height;
    p.depth = c.depth; p.depth16 = c.depth16; p.depth_lo = c.depth_lo; p.depth_lo16 = c.depth_lo16;
    p.wl = c.wl; p.hl = c.hl;
    p.labels = c.labels; p.bgr = c.bgr; p.bgr_step = (long long)c.bgr_step; p.out = c.out;
    p.depth_stride = (c.depth_lo || c.depth_lo16) ? (long long)c.wl * c.hl : plane;
    p.bgr_stride = (long long)c.height * (long long)c.bgr_step;
    p.labels_stride = c.labels ? plane : 0;
    p.out_stride = plane;
    p.sigma_c = c.sigma_c;
    p.radius = c.radius;
    p.kc = guided_k(c.sigma_c);
    p.kd = guided_k(c.sigma_d);
    std::vector<float> lut;
    host_spatial_lut(lut, 2 * c.radius + 1, c.sigma_s);
    for (size_t i = 0; i < lut.size(); i++) p.sfac[i] = (lut[i] != 0.0f) ? lut[i] : 1.0f;
    return p;
}

// Launches `kernel` over the call's frames in slices of at most kMaxGridZ frames (blockIdx.z), in order on one
// stream; each slice's pointers start at its first frame.
template <class P>
static int guided_slices(const P& p0, int n_frames, void (*kernel)(const P), size_t smem, cudaStream_t st) {
    P p = p0;
    for (int f0 = 0; f0 < n_frames; f0 += kMaxGridZ) {
        const long long f = f0;
        p.depth = advance(p0.depth, f * p0.depth_stride);
        p.depth16 = advance(p0.depth16, f * p0.depth_stride);
        p.depth_lo = advance(p0.depth_lo, f * p0.depth_stride);
        p.depth_lo16 = advance(p0.depth_lo16, f * p0.depth_stride);
        p.labels = advance(p0.labels, f * p0.labels_stride);
        p.bgr = p0.bgr + f * p0.bgr_stride;
        p.out = p0.out + f * p0.out_stride;
        const dim3 grd((p.width + kGuidedTW - 1) / kGuidedTW, (p.height + kGuidedTH - 1) / kGuidedTH,
                       std::min(kMaxGridZ, n_frames - f0));
        kernel<<<grd, kGuidedTW * kGuidedTH, smem, st>>>(p);
        CK(cudaGetLastError());
    }
    return KDME_OK;
}

// One launch path for both window forms; the depth type is chosen once per call, whatever the number of frames.
template <int WS_CT, int C>
static int guided_launch(const GuidedCall& c, cudaStream_t stream) {
    const GuidedParams<WS_CT> p = guided_params<WS_CT>(c);
    const size_t smem = (WS_CT > 0) ? 0 : (size_t)(kGuidedTW + 2 * c.radius) * (kGuidedTH + 2 * c.radius) * 12;
    if (c.depth16 || c.depth_lo16)
        return guided_slices(p, c.n_frames, guided_fill_kernel<WS_CT, kGuidedTW, kGuidedTH, C, true>, smem, stream);
    return guided_slices(p, c.n_frames, guided_fill_kernel<WS_CT, kGuidedTW, kGuidedTH, C, false>, smem, stream);
}

// Windows 3..7 run the compile-time-window form, every other window the run-time one; both at any sigmas.
template <int C>
static int guided_launch_c(const GuidedCall& c, cudaStream_t stream) {
    switch (c.radius) {
        case 1: return guided_launch<3, C>(c, stream);
        case 2: return guided_launch<5, C>(c, stream);
        case 3: return guided_launch<7, C>(c, stream);
        default: return guided_launch<0, C>(c, stream);
    }
}

// The kernels read every frame's depth while they write the output: true where the depth input's `in_bytes` and the
// `out_floats` output floats share a byte.
static bool guided_overlap(const void* in, unsigned long long in_bytes, const float* out, unsigned long long out_floats) {
    const uintptr_t i0 = (uintptr_t)in, i1 = i0 + in_bytes;
    const uintptr_t o0 = (uintptr_t)out, o1 = o0 + out_floats * sizeof(float);
    return i0 < o1 && o0 < i1;
}

// Every guided entry point: the checks in order, then the launch.  The call is a fill when its depth is depth or
// depth16, an upsampling when it is depth_lo or depth_lo16; the other three are NULL.
static int guided_batch(GuidedCall c, int channels, void* stream, const char* who) {
    const void* lo = c.depth_lo ? (const void*)c.depth_lo : (const void*)c.depth_lo16;
    const void* in = lo ? lo : c.depth ? (const void*)c.depth : (const void*)c.depth16;
    if (!in || !c.bgr || !c.out) return fail(KDME_EINVAL, std::string(who) + ": NULL argument");
    if (c.n_frames < 1) return fail(KDME_EINVAL, std::string(who) + ": n_frames must be >= 1");
    if (!lo && (c.width <= 0 || c.height <= 0)) return fail(KDME_EINVAL, std::string(who) + ": bad size");
    if (lo && (c.width <= 0 || c.height <= 0 || c.wl <= 0 || c.hl <= 0 || c.wl > c.width || c.hl > c.height))
        return fail(KDME_EINVAL, std::string(who) + ": low-res size must be positive and <= the high-res size");
    const unsigned long long plane = (unsigned long long)c.width * c.height;
    const unsigned long long in_samples = lo ? (unsigned long long)c.wl * c.hl : plane;
    const size_t sample_bytes = (c.depth16 || c.depth_lo16) ? sizeof(uint16_t) : sizeof(float);
    if (guided_overlap(in, in_samples * c.n_frames * sample_bytes, c.out, plane * c.n_frames))
        return fail(KDME_EINVAL, std::string(who) + ": the output overlaps the depth input (in-place operation is not supported)");
    if (c.radius < 0 || c.radius > KDME_MAX_RADIUS) return fail(KDME_EINVAL, std::string(who) + ": bad radius");
    if (channels != KDME_GUIDE_GRAY && channels != KDME_GUIDE_BGR && channels != KDME_GUIDE_BGRX)
        return fail(KDME_EINVAL, std::string(who) + ": guide_channels must be 1 (GRAY), 3 (BGR) or 4 (BGRX)");
    { int rc = check_guide_step(channels, c.width, &c.bgr_step, who); if (rc != KDME_OK) return rc; }
    { int rcd = check_pointer_device(in, who); if (rcd != KDME_OK) return rcd; }
    return with_channels(channels, [&](auto ch) { return guided_launch_c<decltype(ch)::value>(c, (cudaStream_t)stream); });
}

extern "C" int kdme_guided_fill_batch(const float* depth_dev, const int32_t* labels_dev, const uint8_t* bgr_dev,
                                      size_t bgr_step, int guide_channels, float* out_dev, int width, int height,
                                      int n_frames, int window_radius, float sigma_spatial, float sigma_color,
                                      float sigma_depth, void* stream) {
    return guided_batch({depth_dev, nullptr, nullptr, nullptr, 0, 0, labels_dev, bgr_dev, bgr_step, out_dev, width,
                         height, n_frames, window_radius, sigma_spatial, sigma_color, sigma_depth},
                        guide_channels, stream, "kdme_guided_fill_batch");
}

extern "C" int kdme_guided_fill_batch_u16(const uint16_t* depth_dev, const int32_t* labels_dev, const uint8_t* bgr_dev,
                                          size_t bgr_step, int guide_channels, float* out_dev, int width, int height,
                                          int n_frames, int window_radius, float sigma_spatial, float sigma_color,
                                          float sigma_depth, void* stream) {
    return guided_batch({nullptr, depth_dev, nullptr, nullptr, 0, 0, labels_dev, bgr_dev, bgr_step, out_dev, width,
                         height, n_frames, window_radius, sigma_spatial, sigma_color, sigma_depth},
                        guide_channels, stream, "kdme_guided_fill_batch_u16");
}

extern "C" int kdme_guided_fill_ex(const float* depth_dev, const int32_t* labels_dev, const uint8_t* bgr_dev,
                                   size_t bgr_step, int guide_channels, float* out_dev, int width, int height,
                                   int window_radius, float sigma_spatial, float sigma_color, float sigma_depth,
                                   void* stream) {
    return guided_batch({depth_dev, nullptr, nullptr, nullptr, 0, 0, labels_dev, bgr_dev, bgr_step, out_dev, width,
                         height, 1, window_radius, sigma_spatial, sigma_color, sigma_depth},
                        guide_channels, stream, "kdme_guided_fill");
}

extern "C" int kdme_guided_fill(const float* depth_dev, const int32_t* labels_dev, const uint8_t* bgr_dev,
                                size_t bgr_step, float* out_dev, int width, int height, int window_radius,
                                float sigma_spatial, float sigma_color, float sigma_depth, void* stream) {
    return kdme_guided_fill_ex(depth_dev, labels_dev, bgr_dev, bgr_step, KDME_GUIDE_BGR, out_dev, width, height,
                               window_radius, sigma_spatial, sigma_color, sigma_depth, stream);
}

extern "C" int kdme_guided_upsample_batch(const float* depth_lo_dev, int wl, int hl, const int32_t* labels_hi_dev,
                                          const uint8_t* bgr_hi_dev, size_t bgr_step, int guide_channels,
                                          float* out_hi_dev, int width, int height, int n_frames, int window_radius,
                                          float sigma_spatial, float sigma_color, float sigma_depth, void* stream) {
    return guided_batch({nullptr, nullptr, depth_lo_dev, nullptr, wl, hl, labels_hi_dev, bgr_hi_dev, bgr_step, out_hi_dev,
                         width, height, n_frames, window_radius, sigma_spatial, sigma_color, sigma_depth},
                        guide_channels, stream, "kdme_guided_upsample_batch");
}

extern "C" int kdme_guided_upsample_batch_u16(const uint16_t* depth_lo_dev, int wl, int hl,
                                              const int32_t* labels_hi_dev, const uint8_t* bgr_hi_dev, size_t bgr_step,
                                              int guide_channels, float* out_hi_dev, int width, int height,
                                              int n_frames, int window_radius, float sigma_spatial, float sigma_color,
                                              float sigma_depth, void* stream) {
    return guided_batch({nullptr, nullptr, nullptr, depth_lo_dev, wl, hl, labels_hi_dev, bgr_hi_dev, bgr_step, out_hi_dev,
                         width, height, n_frames, window_radius, sigma_spatial, sigma_color, sigma_depth},
                        guide_channels, stream, "kdme_guided_upsample_batch_u16");
}

extern "C" int kdme_guided_upsample_ex(const float* depth_lo_dev, int wl, int hl, const int32_t* labels_hi_dev,
                                       const uint8_t* bgr_hi_dev, size_t bgr_step, int guide_channels, float* out_hi_dev,
                                       int width, int height, int window_radius, float sigma_spatial, float sigma_color,
                                       float sigma_depth, void* stream) {
    return guided_batch({nullptr, nullptr, depth_lo_dev, nullptr, wl, hl, labels_hi_dev, bgr_hi_dev, bgr_step, out_hi_dev,
                         width, height, 1, window_radius, sigma_spatial, sigma_color, sigma_depth},
                        guide_channels, stream, "kdme_guided_upsample");
}

extern "C" int kdme_guided_upsample(const float* depth_lo_dev, int wl, int hl, const int32_t* labels_hi_dev,
                                    const uint8_t* bgr_hi_dev, size_t bgr_step, float* out_hi_dev, int width,
                                    int height, int window_radius, float sigma_spatial, float sigma_color,
                                    float sigma_depth, void* stream) {
    return kdme_guided_upsample_ex(depth_lo_dev, wl, hl, labels_hi_dev, bgr_hi_dev, bgr_step, KDME_GUIDE_BGR, out_hi_dev,
                                   width, height, window_radius, sigma_spatial, sigma_color, sigma_depth, stream);
}

// ------------------------------------------------------------------ Buffer2D
struct buf2d_handle {
    int width = 0, height = 0, device = 0;
    cudaStream_t stream = nullptr;
    float* dw = nullptr;        // weighted_d[width*height]
    float* scratch = nullptr;   // lazily allocated (u16 host path)
    uint16_t* scratch16 = nullptr;
};

static int buf_blocks(long long n) {
    long long b = ((n >> 2) + 255) / 256;
    if (b < 1) b = 1;
    if (b > 148LL * 8) b = 148LL * 8;  // grid-stride; 8 CTAs of 256 threads per SM
    return (int)b;
}

template <int OP>
static int buf_launch(buf2d_handle* b, const float* data, float* out, int n_frames) {
    DeviceGuard g(b->device);
    const long long n = (long long)b->width * b->height;
    buf2d_kernel<OP><<<buf_blocks(n), 256, 0, b->stream>>>(b->dw, data, out, n, b->width, n_frames);
    CK(cudaGetLastError());
    return KDME_OK;
}

extern "C" int buf2d_create(buf2d_handle** out, int width, int height, int device, void* stream) {
    if (!out) return fail(KDME_EINVAL, "buf2d_create: out is NULL");
    *out = nullptr;
    if (width <= 0 || height <= 0) return fail(KDME_EINVAL, "buf2d_create: width/height must be positive");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(KDME_EINVAL, "buf2d_create: no such CUDA device");
    DeviceGuard g(device);
    buf2d_handle* b = new buf2d_handle();
    b->width = width; b->height = height; b->device = device; b->stream = (cudaStream_t)stream;
    cudaError_t e = cudaMalloc(&b->dw, (size_t)width * height * 2 * sizeof(float));
    if (e != cudaSuccess) { delete b; return fail(-(int)e, "buf2d_create: cudaMalloc failed"); }
    int rc = buf_launch<kBufInit>(b, nullptr, nullptr, 0);
    if (rc != KDME_OK) { cudaFree(b->dw); delete b; return rc; }
    *out = b;
    return KDME_OK;
}
extern "C" void buf2d_destroy(buf2d_handle* b) {
    if (!b) return;
    DeviceGuard g(b->device);
    cudaFree(b->dw); cudaFree(b->scratch); cudaFree(b->scratch16);
    delete b;
}
extern "C" int buf2d_init(buf2d_handle* b) {
    if (!b) return fail(KDME_EINVAL, "buf2d_init: NULL handle");
    return buf_launch<kBufInit>(b, nullptr, nullptr, 0);
}
extern "C" int buf2d_insert_f32(buf2d_handle* b, const float* data_dev) {
    if (!b || !data_dev) return fail(KDME_EINVAL, "buf2d_insert_f32: NULL argument");
    if (reinterpret_cast<uintptr_t>(data_dev) & 15) return fail(KDME_EINVAL, "buf2d_insert_f32: data must be 16-byte aligned");
    return buf_launch<kBufInsertF32>(b, data_dev, nullptr, 0);
}
extern "C" int buf2d_insert_dw(buf2d_handle* b, const float* dw_dev) {
    if (!b || !dw_dev) return fail(KDME_EINVAL, "buf2d_insert_dw: NULL argument");
    DeviceGuard g(b->device);
    CK(cudaMemcpyAsync(b->dw, dw_dev, (size_t)b->width * b->height * 2 * sizeof(float), cudaMemcpyDeviceToDevice, b->stream));
    return KDME_OK;
}
extern "C" int buf2d_insert_f32x2(buf2d_handle* b, const float* xy_dev) {
    if (!b || !xy_dev) return fail(KDME_EINVAL, "buf2d_insert_f32x2: NULL argument");
    if (reinterpret_cast<uintptr_t>(xy_dev) & 15) return fail(KDME_EINVAL, "buf2d_insert_f32x2: data must be 16-byte aligned");
    return buf_launch<kBufInsertXY>(b, xy_dev, nullptr, 0);
}
extern "C" int buf2d_update_batch_f32(buf2d_handle* b, const float* data_dev, int n_frames) {
    if (!b || !data_dev) return fail(KDME_EINVAL, "buf2d_update: NULL argument");
    if (n_frames < 1) return fail(KDME_EINVAL, "buf2d_update: n_frames must be >= 1");
    if (reinterpret_cast<uintptr_t>(data_dev) & 15) return fail(KDME_EINVAL, "buf2d_update: data must be 16-byte aligned");
    if (n_frames > 1 && (((long long)b->width * b->height) & 3))
        return fail(KDME_EINVAL, "buf2d_update_batch: width*height must be a multiple of 4 for batches");
    const long long n = (long long)b->width * b->height;
    if (n_frames > 1 && n < 148LL * 2048 * 4) {
        // small buffer: one pixel per thread (four times the warps; see buf2d_update_batch_px1_kernel)
        DeviceGuard g(b->device);
        long long blocks = (n + 255) / 256;
        if (blocks > 148LL * 8) blocks = 148LL * 8;
        buf2d_update_batch_px1_kernel<<<(int)blocks, 256, 0, b->stream>>>(b->dw, data_dev, n, n_frames);
        CK(cudaGetLastError());
        return KDME_OK;
    }
    return buf_launch<kBufUpdate>(b, data_dev, nullptr, n_frames);
}
extern "C" int buf2d_update_f32(buf2d_handle* b, const float* data_dev) { return buf2d_update_batch_f32(b, data_dev, 1); }
extern "C" int buf2d_update_u16_host(buf2d_handle* b, const uint16_t* depth_host) {
    if (!b || !depth_host) return fail(KDME_EINVAL, "buf2d_update_u16_host: NULL argument");
    DeviceGuard g(b->device);
    const long long n = (long long)b->width * b->height;
    if (!b->scratch16) CK(cudaMalloc(&b->scratch16, n * sizeof(uint16_t)));
    CK(cudaMemcpyAsync(b->scratch16, depth_host, n * sizeof(uint16_t), cudaMemcpyHostToDevice, b->stream));
    buf2d_update_u16_kernel<<<buf_blocks(n), 256, 0, b->stream>>>(b->dw, b->scratch16, n);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(b->stream));   // depth_host may be pageable: the caller may reuse it on return
    return KDME_OK;
}
extern "C" int buf2d_get_depth(buf2d_handle* b, float* out_dev) {
    if (!b || !out_dev) return fail(KDME_EINVAL, "buf2d_get_depth: NULL argument");
    if (reinterpret_cast<uintptr_t>(out_dev) & 15) return fail(KDME_EINVAL, "buf2d_get_depth: out must be 16-byte aligned");
    return buf_launch<kBufGetDepth>(b, nullptr, out_dev, 0);
}
extern "C" int buf2d_get_weight(buf2d_handle* b, float* out_dev) {
    if (!b || !out_dev) return fail(KDME_EINVAL, "buf2d_get_weight: NULL argument");
    if (reinterpret_cast<uintptr_t>(out_dev) & 15) return fail(KDME_EINVAL, "buf2d_get_weight: out must be 16-byte aligned");
    return buf_launch<kBufGetWeight>(b, nullptr, out_dev, 0);
}
extern "C" float* buf2d_raw(buf2d_handle* b) { return b ? b->dw : nullptr; }
