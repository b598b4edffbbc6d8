/*
 * ref_shim_pre.h -- host shim placed BEFORE the reference's own kernel text.
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/kdme_oracle.c header).
 *
 * oracle/build_ref.py streams this file, then line ranges of the reference's
 * .cu sources read in place from the reference checkout, then ref_shim_post.h, into
 * `g++ -x c++ -` and writes only oracle/_ref/libkdme_ref.so.  No reference
 * source text is copied into this repository.
 *
 * The shim gives the CUDA-isms of the kernel text a host meaning:
 *   __global__/__device__ -> nothing; blockIdx/blockDim/threadIdx -> thread-local
 *   structs set by the driver loop in ref_shim_post.h; cv::gpu::GpuMat -> a
 *   struct with the one member the kernels touch (.data).
 * nvcc folds powf(x, 2.0f) to x*x (SURVEY.md 8(a) [probe]); the shim does the
 * same so the host build evaluates what the GPU build evaluates, un-fused.
 */
#include <math.h>
#include <cmath>
#include <cstdlib>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <vector>
#include <omp.h>

#define __global__
#define __device__
#define __host__

struct ref_dim3 { int x, y, z; };
static thread_local ref_dim3 blockIdx = {0, 0, 0}, blockDim = {1, 1, 1}, threadIdx = {0, 0, 0};

struct float2 { float x, y; };
struct float3 { float x, y, z; };

namespace cv { namespace gpu { struct GpuMat { unsigned char *data; }; } }

struct ArrayBuffer { struct weighted_d { float d; float w; }; };

static inline float ref_powf(float x, float y) { return (y == 2.0f) ? x * x : ::powf(x, y); }
static inline float ref_pow(float x, float y) { return ref_powf(x, y); }
static inline double ref_pow(double x, double y) { return ::pow(x, y); }
#define powf ref_powf
#define pow ref_pow
using std::fabs;
using std::abs;
