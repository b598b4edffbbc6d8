/*
 * MarkovRandomField.h -- header-only C++ drop-in for the reference class of the same name
 * (MarkovRandomField/MarkovRandomField.h), forwarding to the C ABI in kdme_b200.h.
 *
 * A caller written against the reference --
 *     MarkovRandomField MRF(Kinect::Width, Kinect::Height);
 *     MRF.Process(inputDepth_Device, Color_Device);                         // main.cpp:185-190
 *     float* filtered = MRF.getFiltered_Device();
 * -- compiles unchanged.  The static consts of the reference (MarkovRandomField.cpp:3-6: window 5, ColorSigma 50,
 * SmoothSigma 150) are constructor defaults.
 *
 * The class owns a jbf_handle of its size, which provides the device, the stream and the filtered plane.  Process
 * takes the guide's format from color_image.channels() (CV_8UC3 BGR, CV_8UC4 BGRX, CV_8UC1 GRAY), as
 * JointBilateralFilter::Process does; the pointer-based ProcessBatch reads the format set by setGuideChannels
 * (default 3).  cv::gpu::GpuMat is the one of JointBilateralFilter.h (OpenCV's, or its minimal view type under
 * KDME_NO_OPENCV).
 */
#ifndef KDME_MARKOV_RANDOM_FIELD_H
#define KDME_MARKOV_RANDOM_FIELD_H

#include <stdexcept>
#include <string>

#include "JointBilateralFilter.h"
#include "kdme_b200.h"

class MarkovRandomField {
public:
    /* MarkovRandomField(int width, int height) -- MarkovRandomField.cpp */
    MarkovRandomField(int width, int height, int window_radius = 2, float color_sigma = 50.0f,
                      float smooth_sigma = 150.0f, int device = 0, void* stream = 0)
        : Radius(window_radius), ColorSigma(color_sigma), SmoothSigma(smooth_sigma), Channels(3), h_(0) {
        /* the JBF parameters of the handle are its defaults; the MRF reads only its size, device and stream */
        check(jbf_create(&h_, width, height, 70.0f, 50.0f, 20.0f, 2, 1, device, stream));
    }
    ~MarkovRandomField() { jbf_destroy(h_); }

    /* void Process(float* depth_device, cv::gpu::GpuMat color_image) -- MarkovRandomField.cu:42-49.
     * Result in getFiltered_Device(). */
    void Process(float* depth_device, cv::gpu::GpuMat color_image) {
        setGuideChannels(color_image.channels());
        check(jbf_mrf(h_, depth_device, color_image.data, color_image.step, jbf_filtered_device(h_), Radius,
                      ColorSigma, SmoothSigma));
    }
    /* n_frames Process calls: depth frames back to back (float or uint16 millimetres, the sensor's format, read
     * directly), guides height*bgr_step bytes apart, n_frames filtered planes out. */
    void ProcessBatch(const float* depth_device, const unsigned char* bgr_device, size_t bgr_step, float* out_device,
                      int n_frames) {
        check(jbf_mrf_batch(h_, depth_device, bgr_device, bgr_step, out_device, n_frames, Radius, ColorSigma,
                            SmoothSigma));
    }
    void ProcessBatch(const unsigned short* depth_device, const unsigned char* bgr_device, size_t bgr_step,
                      float* out_device, int n_frames) {
        check(jbf_mrf_batch_u16(h_, depth_device, bgr_device, bgr_step, out_device, n_frames, Radius, ColorSigma,
                                SmoothSigma));
    }
    /* Guide format (1 GRAY, 3 BGR, 4 BGRX) of ProcessBatch. */
    void setGuideChannels(int channels) {
        if (channels != Channels) { check(jbf_set_guide_channels(h_, channels)); Channels = channels; }
    }
    float* getFiltered_Device() const { return jbf_filtered_device(h_); }
    jbf_handle* handle() const { return h_; }

private:
    MarkovRandomField(const MarkovRandomField&);
    MarkovRandomField& operator=(const MarkovRandomField&);
    static void check(int rc) {
        if (rc != KDME_OK) throw std::runtime_error(std::string("kdme_b200: ") + kdme_last_error());
    }
    int Radius;
    float ColorSigma, SmoothSigma;
    int Channels;
    jbf_handle* h_;
};

#endif
