/*
 * JointBilateralFilter.h -- header-only C++ drop-in for the reference class of the same name
 * (JointBilateralFilter/JointBilateralFilter.h:9-36), forwarding to the C ABI in kdme_b200.h.
 *
 * A caller written against the reference --
 *     JointBilateralFilter JBF(Kinect::Width, Kinect::Height);            // main.cpp:67
 *     JBF.Process(inputDepth_Device, Color_Device);                        // main.cpp:179
 *     convertor.projectiveToReal(JBF.getFiltered_Device(), points);        // main.cpp:182
 * -- compiles unchanged: same constructor, same Process(float*, GpuMat) signature, same getters.
 * The static consts of the reference (JointBilateralFilter.cpp:3-6) are constructor defaults.
 *
 * cv::gpu::GpuMat is only used for {data, step, rows, cols, channels()}; when OpenCV's gpu module
 * is not available define KDME_NO_OPENCV (default when <opencv2/gpu/gpu.hpp> is not found) and the
 * minimal view type below takes its place.
 *
 * Guide formats: Process, ProcessXYZ and Upsampling take the guide's format from
 * color_image.channels(): CV_8UC3 BGR (the reference's), CV_8UC4 BGRX/BGRA (Kinect v2, Azure
 * Kinect colour frames; the 4th byte is ignored) or CV_8UC1 GRAY/IR (filters as the BGR image
 * (g,0,0)).  The pointer-based ProcessBatch / ProcessHost / UpsamplingBatch read the format set by setGuideChannels
 * (default 3).  getSmoothImage_Device returns the smoothed guide in the format of the last call.
 */
#ifndef KDME_JOINT_BILATERALFILTER_H
#define KDME_JOINT_BILATERALFILTER_H

#include <stdexcept>
#include <string>

#include "kdme_b200.h"

#if !defined(KDME_NO_OPENCV) && defined(__has_include)
#if __has_include(<opencv2/gpu/gpu.hpp>)
#include <opencv2/gpu/gpu.hpp>
#define KDME_HAVE_CV_GPU 1
#endif
#endif

#ifndef KDME_HAVE_CV_GPU
namespace cv { namespace gpu {
/* The members of cv::gpu::GpuMat this path touches (8-bit, 1, 3 or 4 channels, device memory). */
struct GpuMat {
    unsigned char* data;
    size_t step;
    int rows, cols;
    GpuMat() : data(0), step(0), rows(0), cols(0), cn(3) {}
    GpuMat(int rows_, int cols_, unsigned char* data_, size_t step_, int channels_ = 3)
        : data(data_), step(step_), rows(rows_), cols(cols_), cn(channels_) {}
    int channels() const { return cn; }
    int cn;
};
} }
#endif

class JointBilateralFilter {
public:
    /* JointBilateralFilter(int width, int height) -- JointBilateralFilter.cpp:8-20 */
    JointBilateralFilter(int width, int height, float spatial_sigma = 70.0f, float color_sigma = 50.0f,
                         float depth_sigma = 20.0f, int window_radius = 2, int max_batch = 1, int device = 0,
                         void* stream = 0)
        : Width(width), Height(height), Channels(3), h_(0) {
        check(jbf_create(&h_, width, height, spatial_sigma, color_sigma, depth_sigma, window_radius, max_batch,
                         device, stream));
    }
    ~JointBilateralFilter() { jbf_destroy(h_); }

    /* void Process(float* depth_device, cv::gpu::GpuMat color_image) -- JointBilateralFilter.cu:283-290 */
    void Process(float* depth_device, cv::gpu::GpuMat color_image) {
        useGuide(color_image);
        check(jbf_process(h_, depth_device, color_image.data, color_image.step));
    }
    /* Declared in the reference only as a comment (JointBilateralFilter.h:14). */
    void Upsampling(float* depthlow_device, int low_width, int low_height, cv::gpu::GpuMat colorhigh_image,
                    float* out_device = 0) {
        useGuide(colorhigh_image);
        check(jbf_upsample(h_, depthlow_device, low_width, low_height, colorhigh_image.data, colorhigh_image.step,
                           out_device ? out_device : jbf_filtered_device(h_)));
    }
    void ProcessBatch(const float* depth_device, const unsigned char* bgr_device, size_t bgr_step, float* out_device,
                      int n_frames) {
        check(jbf_process_batch(h_, depth_device, bgr_device, bgr_step, out_device, n_frames));
    }
    /* n_frames Upsampling calls: low-res frames back to back (float or uint16 millimetres, the ToF sensor's
     * format), guides height*bgr_step bytes apart, n_frames high-res planes out. */
    void UpsamplingBatch(const float* depthlow_device, int low_width, int low_height, const unsigned char* bgr_device,
                         size_t bgr_step, float* out_device, int n_frames) {
        check(jbf_upsample_batch(h_, depthlow_device, low_width, low_height, bgr_device, bgr_step, out_device, n_frames));
    }
    void UpsamplingBatch(const unsigned short* depthlow_device, int low_width, int low_height,
                         const unsigned char* bgr_device, size_t bgr_step, float* out_device, int n_frames) {
        check(jbf_upsample_batch_u16(h_, depthlow_device, low_width, low_height, bgr_device, bgr_step, out_device,
                                     n_frames));
    }
    /* Process + DimensionConvertor::projectiveToReal fused (main.cpp:179 + :182): xyz_device = float3[W*H]. */
    void ProcessXYZ(float* depth_device, cv::gpu::GpuMat color_image, float* xyz_device, float fx, float fy, int cx, int cy) {
        useGuide(color_image);
        check(jbf_process_xyz(h_, depth_device, color_image.data, color_image.step, xyz_device, fx, fy, cx, cy));
    }
    /* Host buffers end to end; uint16 depth is the sensor's own format (main.cpp:91-95). */
    void ProcessHost(const float* depth_host, const unsigned char* bgr_host, size_t bgr_step, float* out_host, int n_frames) {
        check(jbf_process_host(h_, depth_host, bgr_host, bgr_step, out_host, n_frames));
    }
    void ProcessHost(const unsigned short* depth_host, const unsigned char* bgr_host, size_t bgr_step, float* out_host, int n_frames) {
        check(jbf_process_host_u16(h_, depth_host, bgr_host, bgr_step, out_host, n_frames));
    }
    /* Guide format (1 GRAY, 3 BGR, 4 BGRX) of the pointer-based calls ProcessBatch / ProcessHost / UpsamplingBatch. */
    void setGuideChannels(int channels) {
        if (channels != Channels) { check(jbf_set_guide_channels(h_, channels)); Channels = channels; }
    }
    float* getFiltered_Device() const { return jbf_filtered_device(h_); }                       /* .cpp:41-43 */
    float* getFiltered_Host() const { return const_cast<float*>(jbf_filtered_host(h_)); }        /* .cpp:44-46 */
    cv::gpu::GpuMat getSmoothImage_Device() {                                                    /* .cpp:47-49 */
        size_t step = 0;
        const unsigned char* p = jbf_smooth_device(h_, &step);
#ifdef KDME_HAVE_CV_GPU
        return cv::gpu::GpuMat(Height, Width, CV_8UC(Channels), const_cast<unsigned char*>(p), step);
#else
        return cv::gpu::GpuMat(Height, Width, const_cast<unsigned char*>(p), step, Channels);
#endif
    }
    /* visualize(float*) (JointBilateralFilter.cpp:50-79) is an OpenCV highgui window: not part of this path. */
    jbf_handle* handle() const { return h_; }

private:
    JointBilateralFilter(const JointBilateralFilter&);
    JointBilateralFilter& operator=(const JointBilateralFilter&);
    static void check(int rc) {
        if (rc != KDME_OK) throw std::runtime_error(std::string("kdme_b200: ") + kdme_last_error());
    }
    void useGuide(const cv::gpu::GpuMat& m) { setGuideChannels(m.channels()); }
    int Width, Height, Channels;
    jbf_handle* h_;
};

#endif
