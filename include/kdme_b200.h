/*
 * kdme_b200.h -- C ABI of the B200-native joint-bilateral depth-enhancement path.
 *
 * This is the drop-in boundary (SURVEY.md 8(b)).  Plain pointers and sizes only;
 * no torch / OpenCV types.  Every entry point cites the reference interface it
 * replaces (paths relative to stevesuyao/KinectDepthMapEnhancement).
 *
 * Conventions
 *   - All image pointers are DEVICE pointers unless the name says *_host.
 *   - depth: float32, row-major y*width+x, millimetres, values <= 50 are holes
 *     (JointBilateralFilter.cu:21).
 *   - bgr: the guide image, uint8, C bytes per pixel with row pitch `step` bytes
 *     (cv::gpu::GpuMat::data / ::step).  C is the handle's guide format
 *     (jbf_set_guide_channels) or the guide_channels argument of the *_ex calls:
 *       KDME_GUIDE_BGR  (3, default)  packed B,G,R (CV_8UC3; the reference assumes
 *                       step == 3*width, main.cpp:62 createContinuous);
 *       KDME_GUIDE_BGRX (4)           B,G,R,X (CV_8UC4: Kinect v2 BGRX, Azure Kinect
 *                       BGRA32); the 4th byte is ignored, so (b,g,r,x) filters
 *                       exactly as the BGR pixel (b,g,r);
 *       KDME_GUIDE_GRAY (1)           one intensity byte (CV_8UC1: IR amplitude, mono
 *                       camera); g filters exactly as the BGR pixel (g,0,0), i.e.
 *                       every colour distance becomes the one of g alone.
 *     Every weight sums over the channels, so their order does not matter: RGB and
 *     RGBA images are valid BGR and BGRX guides.  step == 0 means C*width; a step
 *     below C*width is KDME_EINVAL.
 *   - Every function returns 0 on success, KDME_EINVAL for a bad argument,
 *     KDME_ENOTSUP for an unsupported configuration, or -(cudaError_t) for a CUDA
 *     failure; kdme_last_error() returns a thread-local description.  (The
 *     reference checks no return code at all, JointBilateralFilter.cpp:16-18.)
 *   - Work is enqueued on the stream given at create time (0 = legacy default
 *     stream, which preserves the reference's ordering with callers' default-stream
 *     work, main.cpp:179-183).  Calls are asynchronous with respect to the host
 *     unless stated.
 *   - One handle per (device, stream); a handle is not thread-safe.
 */
#ifndef KDME_B200_H
#define KDME_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KDME_OK 0
#define KDME_EINVAL (-100001)
#define KDME_ENOTSUP (-100002)
#define KDME_MAX_RADIUS 15
/* Guide formats: bytes per pixel of the raw guide image (see "bgr" above). */
#define KDME_GUIDE_GRAY 1
#define KDME_GUIDE_BGR 3
#define KDME_GUIDE_BGRX 4

const char *kdme_last_error(void);
/* Library / build identification: "kdme_b200 <version> sm_100a". */
const char *kdme_version(void);

/* ======================= JointBilateralFilter ============================= */
typedef struct jbf_handle jbf_handle;

/* JointBilateralFilter::JointBilateralFilter(int width,int height)
 *   JointBilateralFilter.h:11, JointBilateralFilter.cpp:8-20; the static consts
 *   WindowSize/SpatialSigma/ColorSigma/DepthSigma (.cpp:3-6) become arguments
 *   (reference values: radius 2, 70, 50, 20).  Builds the spatial LUT
 *   (calcSpatialFilter, .cpp:31-40) and owns Filtered_Device / smooth_Device.
 *   max_batch >= 1 sizes the internal smoothed-guide buffer for jbf_process_batch, and with it the
 *   chunks of jbf_upsample_batch / jbf_upsample_batch_u16. */
int jbf_create(jbf_handle **out, int width, int height, float sigma_spatial, float sigma_color,
               float sigma_depth, int window_radius, int max_batch, int device, void *stream);

/* JointBilateralFilter::~JointBilateralFilter -- JointBilateralFilter.cpp:21-30 */
void jbf_destroy(jbf_handle *h);

/* Guide pre-smooth parameters of cv::gpu::bilateralFilter(color, smooth, 5, 30.0f, 30.0f)
 *   JointBilateralFilter.cu:285.  ksize == 0 disables the pre-smooth (guide used raw). */
int jbf_set_presmooth(jbf_handle *h, int ksize, float sigma_color, float sigma_spatial);

/* Format of the raw guide every later call on this handle reads (jbf_process, _batch, _batch_u16, _batch_xyz,
 * _batch_xyz_u16, _xyz, _host,
 * _host_u16, jbf_presmooth, _presmooth_rows, _presmooth_rows_p2p, jbf_upsample, _upsample_batch,
 * _upsample_batch_u16, jbf_mrf, _mrf_batch, _mrf_batch_u16):
 * KDME_GUIDE_GRAY, KDME_GUIDE_BGR (the default) or KDME_GUIDE_BGRX; any other value is KDME_EINVAL.
 * Handle state only: no synchronisation, no allocation (the host pipeline's guide slots and the
 * jbf_smooth_device buffer are re-sized when next used). */
int jbf_set_guide_channels(jbf_handle *h, int channels);

/* void JointBilateralFilter::Process(float* depth_device, cv::gpu::GpuMat color_image)
 *   JointBilateralFilter.h:13, JointBilateralFilter.cu:283-290.  Result in
 *   jbf_filtered_device(h). */
int jbf_process(jbf_handle *h, const float *depth_dev, const uint8_t *bgr_dev, size_t bgr_step);

/* Process followed by DimensionConvertor::projectiveToReal(float*, float3*) -- main.cpp:179 + :182,
 * KinectDepthEnhancement.cpp:59-60, DimensionConvertor.h:34-48, DimensionConvertor.cpp:8-9 (cx, cy are the
 * truncated principal point) -- as ONE launch pair: the filter's epilogue also writes the float3 cloud
 * x = (u - cx)/fx * z, y = (cy - v)/fy * z, z (IEEE, un-fused, the functor's order) to xyz_dev
 * [height][width][3].  The depth plane still lands in jbf_filtered_device(h). */
int jbf_process_xyz(jbf_handle *h, const float *depth_dev, const uint8_t *bgr_dev, size_t bgr_step,
                    float *xyz_dev, float fx, float fy, int cx, int cy);

/* Numerical bookkeeping of the fast path (no reference counterpart): pixels whose window holds no sample
 * near the pass-1 mean (a pixel between two surfaces) amplify the rounding of that mean beyond what fp32
 * sums can absorb; the filter queues them and a second kernel re-evaluates them in fp64.  Returns how many
 * were re-evaluated / dropped (queue full) since the previous call; synchronises the handle's stream. */
int jbf_refine_stats(jbf_handle *h, unsigned long long *refined, unsigned long long *dropped);

/* Same operator over n_frames independent frames stored back to back (frame
 * stride width*height elements / height*bgr_step bytes); out_dev receives
 * n_frames planes.  One launch triple (pre-smooth, filter, fp64 refinement) per chunk
 * of max_batch frames (the B200-native form of calling Process once per captured
 * frame, main.cpp:86-101 loop shape).  With more than one chunk, the chunks alternate
 * between the handle's stream and an internal one, forked and joined by events: the
 * call is ordered after the stream's earlier work, and the stream's later work after
 * all of it (plain stream semantics; results do not depend on the chunking). */
int jbf_process_batch(jbf_handle *h, const float *depth_dev, const uint8_t *bgr_dev, size_t bgr_step,
                      float *out_dev, int n_frames);
/* The same with depth already on the device in the sensor's format: uint16 millimetres (Kinect, Azure Kinect
 * frames from a decoder or a torch pipeline), read directly by the filter (no conversion pass, no float copy); a
 * sample s filters exactly as the float (float)s, so values <= 50 are holes and frame k equals jbf_process of
 * frame k as float, bit for bit.  KDME_EINVAL: n_frames < 1, a NULL pointer, a guide step below C*width, or an
 * output whose bytes overlap the depth input's. */
int jbf_process_batch_u16(jbf_handle *h, const uint16_t *depth_dev, const uint8_t *bgr_dev, size_t bgr_step,
                          float *out_dev, int n_frames);
/* jbf_process_xyz over n_frames frames: the filtered planes land in out_dev (n_frames planes), their clouds in
 * xyz_dev (n_frames x height x width x 3 floats, v the row within the frame).  Stream semantics as
 * jbf_process_batch; frame k of both outputs equals jbf_process_xyz on frame k alone (its depth plane and its
 * cloud), bit for bit.  On a handle off the fast kernel (exotic sigmas, radius 0) each chunk is filtered and then
 * back-projected by kdme_projective_to_real_batch on the same stream.  KDME_EINVAL: as jbf_process_batch_u16, plus
 * a zero fx / fy and an xyz_dev that overlaps the depth input or out_dev. */
int jbf_process_batch_xyz(jbf_handle *h, const float *depth_dev, const uint8_t *bgr_dev, size_t bgr_step,
                          float *out_dev, float *xyz_dev, int n_frames, float fx, float fy, int cx, int cy);
/* The same with uint16 millimetre depth (see jbf_process_batch_u16). */
int jbf_process_batch_xyz_u16(jbf_handle *h, const uint16_t *depth_dev, const uint8_t *bgr_dev, size_t bgr_step,
                              float *out_dev, float *xyz_dev, int n_frames, float fx, float fy, int cx, int cy);

/* Filter only (JointBilateralFilter.cu:289-290): guide4_dev is an ALREADY smoothed
 * guide in the internal layout u8x4 {B,G,R,0}, row pitch guide_step bytes
 * (multiple of 16).  Used by the row-band path and by stage-isolated parity tests. */
int jbf_filter_guide4(jbf_handle *h, const float *depth_dev, const uint8_t *guide4_dev,
                      size_t guide_step, float *out_dev, int n_frames);

/* Pre-smooth only: raw guide -> internal u8x4 guide (JointBilateralFilter.cu:285); GRAY g gives {g,0,0,0}. */
int jbf_presmooth(jbf_handle *h, const uint8_t *bgr_dev, size_t bgr_step, uint8_t *guide4_dev,
                  size_t guide_step, int n_frames);

/* Row-band forms (one very large frame split into row bands across GPUs, SURVEY.md 8(e)).  The
 * arrays hold `rows` rows = the band plus whatever halo rows exist on each side (image borders
 * have none); jbf_filter_rows writes only rows [y_off, y_off + out_rows) into out_dev (out_rows
 * rows).  A pixel's arithmetic depends only on the image around it, never on the tile or band it
 * falls in, so any band split equals the single-GPU result bit for bit (whatever tile height either
 * launch picks).  `rows` comes from the arguments (the handle's height is not used by these calls). */
int jbf_presmooth_rows(jbf_handle *h, const uint8_t *bgr_dev, size_t bgr_step, uint8_t *guide4_dev,
                       size_t guide_step, int rows);
int jbf_filter_rows(jbf_handle *h, const float *depth_dev, const uint8_t *guide4_dev, size_t guide_step,
                    float *out_dev, int rows, int y_off, int out_rows);

/* Row bands with the halo rows read from the neighbour GPUs' memory INSIDE the kernels (NVLink peer
 * loads on peer-mapped pointers, e.g. torch symmetric memory / CUDA IPC) -- no exchange step.  The arrays
 * hold `rows` rows of which [band0, band1) are this rank's own; a row r < band0 is read from
 * *_up + r * pitch and a row r >= band1 from *_dn + (r - band1) * pitch (either may be NULL at an image
 * border).  Interior tiles keep TMA staging; the two seam tile-rows stage with plain loads.  Results are
 * bit-identical to jbf_presmooth_rows / jbf_filter_rows on arrays whose halo rows were copied in. */
int jbf_presmooth_rows_p2p(jbf_handle *h, const uint8_t *bgr_dev, size_t bgr_step, uint8_t *guide4_dev,
                           size_t guide_step, int rows, int band0, int band1, const uint8_t *bgr_up,
                           const uint8_t *bgr_dn);
int jbf_filter_rows_p2p(jbf_handle *h, const float *depth_dev, const uint8_t *guide4_dev, size_t guide_step,
                        float *out_dev, int rows, int y_off, int out_rows, int band0, int band1,
                        const float *depth_up, const float *depth_dn);

/* Host-buffer convenience used for end-to-end timing: pinned or pageable HOST
 * depth/bgr in, HOST filtered depth out; H2D, Process, D2H are pipelined in
 * chunks of at most max_batch frames.  Synchronous (returns when out_host is
 * complete).  Mirrors main.cpp:160-163 (upload) + :179 (Process) + :183 (download). */
int jbf_process_host(jbf_handle *h, const float *depth_host, const uint8_t *bgr_host, size_t bgr_step,
                     float *out_host, int n_frames);

/* Same pipeline with the depth in the sensor's own format: uint16 millimetres, as xn::DepthMetaData holds it
 * (main.cpp:91-95; Buffer2D::insertData(xn::DepthMetaData*) converts it to float on the host before the
 * upload, Buffer2D.cpp:18-32).  Here the 2-byte samples are uploaded and the filter reads them directly
 * (as jbf_process_batch_u16): 5 instead of 7 bytes per pixel cross PCIe. */
int jbf_process_host_u16(jbf_handle *h, const uint16_t *depth_host, const uint8_t *bgr_host, size_t bgr_step,
                         float *out_host, int n_frames);

/* Page-locked host memory for those buffers (cudaHostAlloc, portable).  write_combined != 0: for buffers the
 * CPU only writes front to back (sensor frames); never for the result buffer.  NULL on failure. */
void *kdme_host_alloc(size_t bytes, int write_combined);
void kdme_host_free(void *p);

/* float* JointBilateralFilter::getFiltered_Device() const -- JointBilateralFilter.cpp:41-43.
 * Borrowed pointer, valid until the next jbf_process / jbf_destroy. */
float *jbf_filtered_device(jbf_handle *h);

/* float* JointBilateralFilter::getFiltered_Host() const -- JointBilateralFilter.cpp:44-46.
 * Performs the D2H copy the reference only does inside visualize() (.cpp:52) and
 * synchronises the stream.  Pinned memory owned by the handle. */
const float *jbf_filtered_host(jbf_handle *h);

/* cv::gpu::GpuMat JointBilateralFilter::getSmoothImage_Device() -- .cpp:47-49.
 * Returns the smoothed guide in the handle's guide format, continuous, materialised from the
 * internal u8x4 guide of the last jbf_process: packed BGR (CV_8UC3, *step = 3*width), GRAY
 * (CV_8UC1, *step = width) or BGRX (CV_8UC4, *step = 4*width, 4th byte 255). */
const uint8_t *jbf_smooth_device(jbf_handle *h, size_t *step);

/* The internal u8x4 smoothed guide of the last process call and its pitch. */
const uint8_t *jbf_guide4_device(jbf_handle *h, size_t *step);

/* void Upsampling(float* depthlow_device, cv::gpu::GpuMat colorhigh_image) --
 * declared but never implemented in the reference (JointBilateralFilter.h:14,
 * MarkovRandomField.h:14); defined by SURVEY.md 8(d) config 3: low-res sample
 * (xl,yl) sits at high-res pixel (floor((xl+.5)*W/wl), floor((yl+.5)*H/hl)), all
 * other pixels are holes, then the Process formula runs at the handle's
 * (high-res) size and radius.  The sparse image is never materialised in HBM as
 * an input: the scatter happens while staging tiles. */
int jbf_upsample(jbf_handle *h, const float *depth_lo_dev, int wl, int hl, const uint8_t *bgr_hi_dev,
                 size_t bgr_step, float *out_hi_dev);

/* n_frames independent Upsampling calls (a recorded ToF sequence in one call).  Frame strides: wl*hl depth
 * samples, height*bgr_step guide bytes, width*height output floats.  Chunks of max_batch frames; with more
 * than one chunk the chunks alternate between the handle's stream and the internal lane, with
 * jbf_process_batch's stream semantics.  Frame k of the result equals jbf_upsample of frame k alone, bit for
 * bit.  KDME_EINVAL: n_frames < 1, a NULL pointer, wl / hl outside [1, width] / [1, height], a guide step
 * below C*width. */
int jbf_upsample_batch(jbf_handle *h, const float *depth_lo_dev, int wl, int hl, const uint8_t *bgr_hi_dev,
                       size_t bgr_step, float *out_hi_dev, int n_frames);
/* The same with sensor depth: uint16 millimetres (Kinect v2, Azure Kinect), read directly by the kernels
 * (no conversion pass); a sample s filters exactly as the float (float)s, so values <= 50 are holes as
 * before. */
int jbf_upsample_batch_u16(jbf_handle *h, const uint16_t *depth_lo_dev, int wl, int hl, const uint8_t *bgr_hi_dev,
                           size_t bgr_step, float *out_hi_dev, int n_frames);

/* Which kernel the handle selected: 0 = register-tiled fast path, 1 = generic path
 * (exotic sigmas / radius); bit 8 (0x100) set when the last launch staged tiles by TMA
 * (uint16 depth too: needs width % 8 == 0 and a 16-byte aligned depth base, else plain loads),
 * bit 9 (0x200) when it used 64x8 tiles (small launches) instead of 64x16. */
int jbf_kernel_variant(jbf_handle *h);

/* "Next" row f1: MarkovRandomField::Process (MarkovRandomField.cu:4-49), raw guide.  Reference constants
 * (MarkovRandomField.cpp:3-6): radius 2, color_sigma 50, smooth_sigma 150.  The handle provides the size, the guide
 * format, the device and the stream; the call leaves the handle's buffers (jbf_filtered_device, jbf_guide4_device,
 * jbf_smooth_device) as they were.  The batch of one of jbf_mrf_batch. */
int jbf_mrf(jbf_handle *h, const float *depth_dev, const uint8_t *bgr_dev, size_t bgr_step,
            float *out_dev, int window_radius, float color_sigma, float smooth_sigma);
/* n_frames independent MarkovRandomField::Process calls in one call (a recorded Kinect sequence).  Frame strides:
 * width*height depth samples, height*bgr_step guide bytes, width*height output floats.  Frame k of the result
 * equals jbf_mrf on frame k alone, bit for bit.  Nothing is staged in HBM, so there is no max_batch chunking.
 * KDME_EINVAL: n_frames < 1, a NULL pointer, a radius outside [0, KDME_MAX_RADIUS], a guide step below C*width, or
 * an output whose bytes overlap the depth input's. */
int jbf_mrf_batch(jbf_handle *h, const float *depth_dev, const uint8_t *bgr_dev, size_t bgr_step, float *out_dev,
                  int n_frames, int window_radius, float color_sigma, float smooth_sigma);
/* The same with sensor depth: uint16 millimetres, read directly by the kernel (no conversion pass); a sample s
 * filters exactly as the float (float)s. */
int jbf_mrf_batch_u16(jbf_handle *h, const uint16_t *depth_dev, const uint8_t *bgr_dev, size_t bgr_step,
                      float *out_dev, int n_frames, int window_radius, float color_sigma, float smooth_sigma);

/* "Next" row f3: DimensionConvertor::projectiveToReal(float*, float3*)
 * (DimensionConvertor.cu:3-23, DimensionConvertor.h:34-61); cx, cy truncated to
 * int as DimensionConvertor.cpp:8-9 does.  The batch of one of kdme_projective_to_real_batch, with its
 * original checks (KDME_EINVAL for a NULL pointer or a non-positive size only). */
int kdme_projective_to_real(const float *depth_dev, float *xyz_dev, int width, int height, float fx,
                            float fy, int cx, int cy, void *stream);
/* n_frames depth planes stored back to back -> n_frames clouds [height][width][3]; v is the row within each
 * frame, so frame k equals kdme_projective_to_real on frame k alone, bit for bit.  KDME_EINVAL: n_frames < 1, a
 * NULL pointer, a non-positive size, a zero fx / fy, or an xyz_dev whose bytes overlap the depth input's. */
int kdme_projective_to_real_batch(const float *depth_dev, float *xyz_dev, int width, int height, int n_frames,
                                  float fx, float fy, int cx, int cy, void *stream);

/* "Next" row f2: Projection_GPU::bilateralfilter (Projection_GPU.cu:213-246, launched :264-265) -- depth-only
 * bilateral on the z of a packed float3 cloud, then x,y = normalized.x,y * z.  Race-free: in != out.
 * Reference constants (Projection_GPU.cpp:3-5): radius 3, sigma_spatial 20, sigma_depth 100.
 * sigma_spatial and sigma_depth must be > 0 (KDME_EINVAL otherwise). */
int kdme_depth_bilateral_xyz(const float *normalized_dev, const float *in_dev, float *out_dev, int width,
                             int height, int window_radius, float sigma_spatial, float sigma_depth, void *stream);

/* "Next" row f4: the evaluation metric of main.cpp:217-308 -- mean Euclidean distance (mm) between a
 * method's cloud and the averaged ground-truth cloud over pixels whose z are both in (50, 15000).
 * Packed float3 device clouds; synchronous (returns the mean and the pixel count on the host). */
int kdme_mean_3d_error(const float *points_dev, const float *truth_dev, long long n_points, double *mean_out,
                       long long *count_out, void *stream);

/* ================= EdgeRefinedSuperpixel::depthmap_enhancement ============ */
/* The guided cross-bilateral stage reached from TOFDepthInterpolation.cpp:65 ->
 * EdgeRefinedSuperpixel::EdgeRefining (EdgeRefinedSuperpixel.cu:208-223) ->
 * depthmap_enhancement (:104-205), with race-free read-input/write-output
 * semantics.  labels_dev may be NULL (one label).  Reference constants
 * (EdgeRefinedSuperpixel.cpp:4-7): radius 3, sigma_s 30, sigma_c 50, sigma_d 70.
 * The guide is the RAW colour image (no pre-smooth). */
int kdme_guided_fill(const float *depth_dev, const int32_t *labels_dev, const uint8_t *bgr_dev,
                     size_t bgr_step, float *out_dev, int width, int height, int window_radius,
                     float sigma_spatial, float sigma_color, float sigma_depth, void *stream);
/* Same with a guide of guide_channels bytes per pixel (KDME_GUIDE_*); kdme_guided_fill is this with
 * KDME_GUIDE_BGR. */
int kdme_guided_fill_ex(const float *depth_dev, const int32_t *labels_dev, const uint8_t *bgr_dev,
                        size_t bgr_step, int guide_channels, float *out_dev, int width, int height,
                        int window_radius, float sigma_spatial, float sigma_color, float sigma_depth,
                        void *stream);

/* Label-guided upsampling (SURVEY.md 8(d) config 3, "a5 label-guided variant when labels are supplied"):
 * the wl x hl low-res depth is scattered onto its high-res sites while tiles are staged (never
 * materialised) and the depthmap_enhancement sweeps (EdgeRefinedSuperpixel.cu:104-205) run at the
 * high-res size with the high-res label map (nullable) and RAW high-res guide. */
int kdme_guided_upsample(const float *depth_lo_dev, int wl, int hl, const int32_t *labels_hi_dev,
                         const uint8_t *bgr_hi_dev, size_t bgr_step, float *out_hi_dev, int width, int height,
                         int window_radius, float sigma_spatial, float sigma_color, float sigma_depth,
                         void *stream);
/* Same with a guide of guide_channels bytes per pixel (KDME_GUIDE_*). */
int kdme_guided_upsample_ex(const float *depth_lo_dev, int wl, int hl, const int32_t *labels_hi_dev,
                            const uint8_t *bgr_hi_dev, size_t bgr_step, int guide_channels, float *out_hi_dev,
                            int width, int height, int window_radius, float sigma_spatial, float sigma_color,
                            float sigma_depth, void *stream);

/* Streams of frames (a recorded ToF or Kinect sequence in one call): n_frames independent fills stored back to
 * back, asynchronous on `stream`.  Frame strides: width*height depth samples, height*bgr_step guide bytes,
 * width*height labels (labels_dev is NULL for one label, or holds n_frames label maps) and width*height output
 * floats.  Frame k of the result equals kdme_guided_fill_ex on frame k alone, bit for bit; kdme_guided_fill(_ex)
 * is the batch of one.  KDME_EINVAL: n_frames < 1, a NULL depth / guide / output pointer, a non-positive size, a
 * radius outside [0, KDME_MAX_RADIUS], a guide format other than KDME_GUIDE_*, a guide step below C*width, or
 * an output whose bytes overlap the depth input's (the fill does not run in place). */
int kdme_guided_fill_batch(const float *depth_dev, const int32_t *labels_dev, const uint8_t *bgr_dev,
                           size_t bgr_step, int guide_channels, float *out_dev, int width, int height, int n_frames,
                           int window_radius, float sigma_spatial, float sigma_color, float sigma_depth,
                           void *stream);
/* The same with sensor depth: uint16 millimetres, read directly by the kernels (no conversion pass); a sample s
 * filters exactly as the float (float)s, so values <= 50 are holes as before. */
int kdme_guided_fill_batch_u16(const uint16_t *depth_dev, const int32_t *labels_dev, const uint8_t *bgr_dev,
                               size_t bgr_step, int guide_channels, float *out_dev, int width, int height,
                               int n_frames, int window_radius, float sigma_spatial, float sigma_color,
                               float sigma_depth, void *stream);
/* n_frames independent label-guided upsamplings, as kdme_guided_fill_batch: frame strides wl*hl low-res depth
 * samples, height*bgr_step guide bytes, width*height labels (or NULL) and width*height output floats.  Frame k
 * equals kdme_guided_upsample_ex on frame k alone, bit for bit; kdme_guided_upsample(_ex) is the batch of one.
 * KDME_EINVAL as for the fill, with wl / hl outside [1, width] / [1, height] in place of the overlap check. */
int kdme_guided_upsample_batch(const float *depth_lo_dev, int wl, int hl, const int32_t *labels_hi_dev,
                               const uint8_t *bgr_hi_dev, size_t bgr_step, int guide_channels, float *out_hi_dev,
                               int width, int height, int n_frames, int window_radius, float sigma_spatial,
                               float sigma_color, float sigma_depth, void *stream);
/* The same with uint16 low-res depth (Kinect v2 512x424, Azure Kinect 640x576 millimetres). */
int kdme_guided_upsample_batch_u16(const uint16_t *depth_lo_dev, int wl, int hl, const int32_t *labels_hi_dev,
                                   const uint8_t *bgr_hi_dev, size_t bgr_step, int guide_channels,
                                   float *out_hi_dev, int width, int height, int n_frames, int window_radius,
                                   float sigma_spatial, float sigma_color, float sigma_depth, void *stream);

/* ========================= ArrayBuffer / Buffer2D ========================= */
typedef struct buf2d_handle buf2d_handle;

/* Buffer2D::Buffer2D(int width,int height) -- Buffer2D.cpp:4-10, ArrayBuffer.cpp:3-17:
 * allocates width*height weighted_d {float d; float w;} (ArrayBuffer.h:12-15) and zeroes it
 * (initDeviceMemoryElementsKernel, ArrayBuffer.cu:9-22). */
int buf2d_create(buf2d_handle **out, int width, int height, int device, void *stream);
void buf2d_destroy(buf2d_handle *b);
/* ArrayBuffer::initDeviceMemoryElements -- ArrayBuffer.cu:27-30 */
int buf2d_init(buf2d_handle *b);
/* Buffer2D::insertData(float*) -- Buffer2D.cu:33-56: d = data, w = 1 */
int buf2d_insert_f32(buf2d_handle *b, const float *data_dev);
/* Buffer2D::insertData(weighted_d*) -- Buffer2D.cpp:13-15: D2D copy of the AoS */
int buf2d_insert_dw(buf2d_handle *b, const float *dw_dev);
/* Buffer2D::insertData(float2*) -- Buffer2D.cu:123-147: d = data.x, w = ROW INDEX
 * (reference behaviour, Buffer2D.cu:137, reproduced and documented). */
int buf2d_insert_f32x2(buf2d_handle *b, const float *xy_dev);
/* Buffer2D::updateData(float*) -- Buffer2D.cu:97-120 -> updateWaitedDepth :13-30 */
int buf2d_update_f32(buf2d_handle *b, const float *data_dev);
/* n_frames successive updateData calls fused into one pass over the buffer
 * (the 1000-frame averaging loop, main.cpp:86-101); frames are back to back. */
int buf2d_update_batch_f32(buf2d_handle *b, const float *data_dev, int n_frames);
/* Buffer2D::insertData(xn::DepthMetaData*) -- Buffer2D.cpp:18-32, without OpenNI:
 * a HOST uint16 depth map (XnDepthPixel) is converted to float, uploaded and passed
 * to updateData.  Synchronous. */
int buf2d_update_u16_host(buf2d_handle *b, const uint16_t *depth_host);
/* Buffer2D::getDepthMap / getWeightMap -- Buffer2D.cu:59-77, 79-94 */
int buf2d_get_depth(buf2d_handle *b, float *out_dev);
int buf2d_get_weight(buf2d_handle *b, float *out_dev);
/* ArrayBuffer::getRawPointer -- ArrayBuffer.cpp:19-21 (borrowed; {d,w} interleaved) */
float *buf2d_raw(buf2d_handle *b);

#ifdef __cplusplus
}
#endif
#endif /* KDME_B200_H */
