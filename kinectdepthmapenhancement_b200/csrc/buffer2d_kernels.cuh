// buffer2d_kernels.cuh -- ArrayBuffer / Buffer2D device accumulators for sm_100a.
//
// Reference: ArrayBuffer/ArrayBuffer.h:12-15 (weighted_d {float d; float w;}, AoS,
// 8 bytes), ArrayBuffer/ArrayBuffer.cu:9-22 (init), ArrayBuffer/Buffer2D.cu:13-140.
// The reference runs one thread per pixel on a 2-D grid that drops the remainder
// of sizes not divisible by 32x24; these kernels are flat, grid-stride, cover
// every pixel, and move 16 bytes per access (two weighted_d per float4, four
// depths per float4).  They are pure streaming: 8 / 12 / 20 bytes per pixel.
//
// Arithmetic is written with explicit round-to-nearest intrinsics so nvcc cannot
// contract it into FMAs: results are bit-identical to the un-fused fp32
// evaluation in oracle/kdme_oracle.c.
#pragma once
#include "common.cuh"

namespace kdme {

// updateWaitedDepth -- Buffer2D.cu:13-30 (THRESH is passed but unused there).
__device__ __forceinline__ void update_weighted(float& rd, float& rw, float d) {
    if (d > 50.0f) {
        if (rd != 0.0f) {
            if ((float)abs((int)rd - (int)d) < __fmul_rn(d, 0.01f)) {
                const float t1 = __fmul_rn(rd, __fadd_rn(rw, 1.0f));
                const float t2 = __fmul_rn(d, rw);
                rd = __fdiv_rn(__fadd_rn(t1, t2), __fadd_rn(__fmul_rn(rw, 2.0f), 1.0f));
                rw = __fadd_rn(rw, 1.0f);
            }
        } else {
            rd = d;
            rw = 1.0f;
        }
    }
}

enum BufOp : int { kBufInit = 0, kBufInsertF32, kBufInsertXY, kBufUpdate, kBufGetDepth, kBufGetWeight };

// n = number of pixels; buf = {d,w} interleaved; data/out planar (or float2 for InsertXY).
template <int OP>
__global__ void __launch_bounds__(256) buf2d_kernel(float* __restrict__ buf, const float* __restrict__ data,
                                                    float* __restrict__ out, long long n, int width,
                                                    int n_frames) {
    const long long nquad = n >> 2;  // groups of 4 pixels
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long qd = (long long)blockIdx.x * blockDim.x + threadIdx.x; qd < nquad; qd += stride) {
        float4* b4 = reinterpret_cast<float4*>(buf) + 2 * qd;
        if (OP == kBufInit) {
            b4[0] = make_float4(0.f, 0.f, 0.f, 0.f);
            b4[1] = make_float4(0.f, 0.f, 0.f, 0.f);
        } else if (OP == kBufInsertF32) {
            const float4 d = ldg_stream_f4(reinterpret_cast<const float4*>(data) + qd);
            b4[0] = make_float4(d.x, 1.f, d.y, 1.f);
            b4[1] = make_float4(d.z, 1.f, d.w, 1.f);
        } else if (OP == kBufInsertXY) {
            // d = data.x, w = ROW INDEX (Buffer2D.cu:137)
            const float4 a = ldg_stream_f4(reinterpret_cast<const float4*>(data) + 2 * qd);
            const float4 c = ldg_stream_f4(reinterpret_cast<const float4*>(data) + 2 * qd + 1);
            const long long px = 4 * qd;
            b4[0] = make_float4(a.x, (float)((px + 0) / width), a.z, (float)((px + 1) / width));
            b4[1] = make_float4(c.x, (float)((px + 2) / width), c.z, (float)((px + 3) / width));
        } else if (OP == kBufUpdate) {
            float4 a = b4[0], c = b4[1];
            // frames are applied in order (the update is a recurrence per pixel) but their loads are
            // independent: issue 8 at a time so the pass stays bandwidth- rather than latency-bound
            constexpr int PF = 8;
            if (n_frames == 1) {  // the per-frame call of the reference (Buffer2D.cu:116-120): pure streaming
                const float4 d = ldg_stream_f4(reinterpret_cast<const float4*>(data) + qd);
                update_weighted(a.x, a.y, d.x);
                update_weighted(a.z, a.w, d.y);
                update_weighted(c.x, c.y, d.z);
                update_weighted(c.z, c.w, d.w);
            } else
            for (int f0 = 0; f0 < n_frames; f0 += PF) {
                float4 d[PF];
#pragma unroll
                for (int u = 0; u < PF; ++u)
                    if (f0 + u < n_frames)
                        d[u] = ldg_stream_f4(reinterpret_cast<const float4*>(data + (long long)(f0 + u) * n) + qd);
#pragma unroll
                for (int u = 0; u < PF; ++u)
                    if (f0 + u < n_frames) {
                        update_weighted(a.x, a.y, d[u].x);
                        update_weighted(a.z, a.w, d[u].y);
                        update_weighted(c.x, c.y, d[u].z);
                        update_weighted(c.z, c.w, d[u].w);
                    }
            }
            b4[0] = a;
            b4[1] = c;
        } else if (OP == kBufGetDepth) {
            const float4 a = b4[0], c = b4[1];
            stg_stream_f4(reinterpret_cast<float4*>(out) + qd, make_float4(a.x, a.z, c.x, c.z));
        } else {
            const float4 a = b4[0], c = b4[1];
            stg_stream_f4(reinterpret_cast<float4*>(out) + qd, make_float4(a.y, a.w, c.y, c.w));
        }
    }
    // tail (n not a multiple of 4): scalar, first threads of block 0
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const long long k = (nquad << 2) + threadIdx.x;
        float rd = buf[2 * k], rw = buf[2 * k + 1];
        if (OP == kBufInit) { rd = 0.f; rw = 0.f; }
        else if (OP == kBufInsertF32) { rd = data[k]; rw = 1.f; }
        else if (OP == kBufInsertXY) { rd = data[2 * k]; rw = (float)(k / width); }
        else if (OP == kBufUpdate) { for (int f = 0; f < n_frames; ++f) update_weighted(rd, rw, data[(long long)f * n + k]); }
        else if (OP == kBufGetDepth) { out[k] = rd; }
        else { out[k] = rw; }
        if (OP <= kBufUpdate) { buf[2 * k] = rd; buf[2 * k + 1] = rw; }
    }
}

// N-frame update of a SMALL buffer (one Kinect frame is 307 200 pixels): the update is a branchy serial recurrence
// per pixel (a division per accepted frame), so with 4 pixels per thread a 640x480 buffer is 76 800 threads whose four
// chains run one after the other -- a quarter of the GPU's thread slots, latency-bound (32 % of HBM).  One pixel per
// thread gives the scheduler four times the warps to hide the chain's latency behind; loads stay coalesced (a warp
// reads 128 contiguous bytes of each frame) and 8 frames are in flight per thread.  Same arithmetic, same order.
__global__ void __launch_bounds__(256) buf2d_update_batch_px1_kernel(float* __restrict__ buf, const float* __restrict__ data,
                                                                     long long n, int n_frames) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        float2 a = reinterpret_cast<float2*>(buf)[k];
        constexpr int PF = 8;
        for (int f0 = 0; f0 < n_frames; f0 += PF) {
            float d[PF];
#pragma unroll
            for (int u = 0; u < PF; ++u)
                if (f0 + u < n_frames) d[u] = __ldg(data + (long long)(f0 + u) * n + k);
#pragma unroll
            for (int u = 0; u < PF; ++u)
                if (f0 + u < n_frames) update_weighted(a.x, a.y, d[u]);
        }
        reinterpret_cast<float2*>(buf)[k] = a;
    }
}

// Buffer2D::insertData(xn::DepthMetaData*) -- Buffer2D.cpp:18-32 (host loop u16 -> float, H2D, updateData)
// as ONE pass: the uint16 frame is read directly and folded into the accumulator (18 B/pixel).
__global__ void __launch_bounds__(256) buf2d_update_u16_kernel(float* __restrict__ buf, const uint16_t* __restrict__ data,
                                                               long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nquad = ((reinterpret_cast<uintptr_t>(data) & 7) == 0) ? (n >> 2) : 0;
    for (long long qd = tid; qd < nquad; qd += stride) {
        float4* b4 = reinterpret_cast<float4*>(buf) + 2 * qd;
        const uint2 v = __ldg(reinterpret_cast<const uint2*>(data) + qd);
        float4 a = b4[0], c = b4[1];
        update_weighted(a.x, a.y, (float)(v.x & 0xffffu));
        update_weighted(a.z, a.w, (float)(v.x >> 16));
        update_weighted(c.x, c.y, (float)(v.y & 0xffffu));
        update_weighted(c.z, c.w, (float)(v.y >> 16));
        b4[0] = a;
        b4[1] = c;
    }
    for (long long k = (nquad << 2) + tid; k < n; k += stride) {
        float rd = buf[2 * k], rw = buf[2 * k + 1];
        update_weighted(rd, rw, (float)data[k]);
        buf[2 * k] = rd;
        buf[2 * k + 1] = rw;
    }
}

// DimensionConvertor::projectiveToReal(float*, float3*) -- DimensionConvertor.h:34-61
// (next row f3).  IEEE division and un-fused ops, same order as the reference functor.  n_frames frames back to
// back: v is the row within the frame.
__global__ void __launch_bounds__(256) projective_to_real_kernel(const float* __restrict__ depth,
                                                                 float* __restrict__ xyz, int width, int height,
                                                                 int n_frames, float fx, float fy, int cx, int cy) {
    const long long n = (long long)width * height * n_frames;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        const float z = depth[k];
        const long long row = k / width;
        const int v = (int)(row % height), u = (int)(k - row * width);
        float py = __fsub_rn((float)cy, (float)v);
        float px = __fsub_rn((float)u, (float)cx);
        px = __fdiv_rn(px, fx);
        py = __fdiv_rn(py, fy);
        xyz[3 * k + 0] = __fmul_rn(px, z);
        xyz[3 * k + 1] = __fmul_rn(py, z);
        xyz[3 * k + 2] = z;
    }
}

}  // namespace kdme
