// common.cuh -- shared helpers for the sm_100a kernels of the joint-bilateral path.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace kdme {

// fp32 expf() returns exactly 0 below -150 ln2 (denormals kept, no FTZ): the
// reference's skip-if-zero guards (JointBilateralFilter.cu:30-33,63-68) fire there.
constexpr double kExpZeroArg = 103.97207708399179;  // natural-log units
constexpr double kLog2e = 1.4426950408889634;
constexpr double kLn2 = 0.6931471805599453;
// All tap weights are evaluated as 2^(arg + kWeightBias): only ratios of weights
// matter, and the bias keeps every weight the reference can represent (down to its
// fp32 denormals, 2^-149) inside the normal range of ex2.approx.ftz.
constexpr float kWeightBias = 32.0f;
// A depth is a sample only when > 50 mm (JointBilateralFilter.cu:21).
constexpr float kValidDepth = 50.0f;

// float bits of 2^23: IDP.4A accumulates the integer colour distance on top of it,
// giving the float 2^23 + cd exactly; an invalid tap carries 0x7F000000 (1.7e38)
// instead, which drives the exponent argument to -inf and the weight to exactly 0.
constexpr uint32_t kMagicValid = 0x4B000000u;
constexpr uint32_t kMagicInvalid = 0x7F000000u;

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ float rcp_approx(float x) {   // MUFU.RCP, max relative error 2^-23
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ float lds_f32(uint32_t addr) {   // ld.shared through a 32-bit shared-window address
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}

// ---- mbarrier + TMA (cp.async.bulk.tensor) primitives -------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    uint32_t done;
    do {
        asm volatile(
            "{\n.reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(phase)
            : "memory");
    } while (!done);
}
// 3-D tiled TMA load: box -> shared memory, completion on an mbarrier (bytes).
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                            int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// ---- programmatic dependent launch (PDL): a kernel launched with
// cudaLaunchAttributeProgrammaticStreamSerialization may start while its predecessor in the stream is
// still running; grid_dependency_wait() blocks until the predecessor's memory is visible, and the
// predecessor calls grid_launch_dependents() once its remaining work no longer gates the successor's
// prologue.  Both are no-ops in an ordinary launch.
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- packed fp32x2 arithmetic (Blackwell FFMA2 / FADD2: one issue slot, two lanes of fp32) ----------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 neg2(f32x2 a) { return a ^ 0x8000000080000000ull; }   // both lanes negated (exact)
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// Depth sample i of a plane of DT (float, or uint16_t millimetres) as a float: every depth read of every kernel goes
// through here.  A uint16 sample s reads as the float (float)s, exactly, so a uint16 frame filters bit for bit like its
// float32 image (s <= 50 is a hole).
template <class DT>
__device__ __forceinline__ float load_depth(const void* base, long long i) {
    return (float)__ldg(static_cast<const DT*>(base) + i);
}

// low-res sample index landing on high-res coordinate x, or -1 (SURVEY.md 8(d) config 3):
// x_hi(xl) = floor((2 xl + 1) * W / (2 wl)); at most one xl per x when W >= wl.
__device__ __forceinline__ int upsample_site(int x, int W, int wl) {
    long long num = 2LL * wl * x - W;
    int xl = (num <= 0) ? 0 : (int)((num + 2LL * W - 1) / (2LL * W));
    if (xl >= wl) return -1;
    return ((int)(((2LL * xl + 1) * W) / (2LL * wl)) == x) ? xl : -1;
}

// 16-byte streaming global accesses (read-once inputs / write-once outputs).
__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ void stg_stream_f4(float4* p, const float4& v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

}  // namespace kdme
