/*
 * cofusion_b200.h -- C ABI of the B200-native Co-Fusion hot path (libcofusion_b200.so).
 *
 * The reference (martinruenz/co-fusion @ 11b9fef) has no plugin/FFI layer; its seam is C++ source
 * level.  This header exports both usable cut lines (SURVEY.md section 8b):
 *
 *   1. the free-function seam of Core/Cuda/cudafuncs.cuh:64-193 -- one entry point per reference
 *      function, raw device pointers + pitch in bytes (the layout contract of DeviceArray2D,
 *      Core/Cuda/containers/kernel_containers.hpp:60-93), host scalars/matrices by value;
 *   2. the class seam -- cfb_odom_* mirrors RGBDOdometry (Core/Utils/RGBDOdometry.h:31-139);
 *      cfb_ctx_* / cfb_model_* mirror CoFusion::processFrame's per-frame calls into Model /
 *      ModelProjection (Core/Model/Model.h:117-157, Core/CoFusion.cpp:171-545) without OpenGL.
 *
 * Conventions
 *   - every function returns 0 on success or a non-zero code; cfb_last_error() gives the text
 *     (thread-local).  Nothing calls exit() (the reference's cudaSafeCall does, convenience.cuh:74-83).
 *   - `stream` is a cudaStream_t passed as void*; NULL = the default stream.
 *   - "planar map" = 3 planes of H rows each ([k*H + y][x] f32), the reference vertex/normal layout
 *     (Core/Cuda/reduce.cu:287-289).  Pitches must be multiples of 8 bytes.
 *   - matrices are row-major; poses are 4x4 row-major camera->world.
 *   - handles own all device memory; callers own host buffers; no allocation after *_create.
 */
#ifndef COFUSION_B200_H_
#define COFUSION_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* cfb_last_error(void);
int cfb_version(void);
/* number of CUDA devices visible (0 if none / driver missing) */
int cfb_device_count(void);

/* DeviceArray::upload / download (Core/Cuda/containers/device_memory.cpp:218-233): synchronous
 * copies between a host buffer and device memory owned by this module or by the caller. */
int cfb_upload(void* dst_dev, const void* src_host, size_t bytes, void* stream);
int cfb_download(void* dst_host, const void* src_dev, size_t bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Seam 1: free functions (device pointers).  Each cites the reference function it replaces.
 * ---------------------------------------------------------------------------------------------- */

/* CoFusion::filterDepth + depth_bilateral_metric.frag (Core/CoFusion.cpp:567-574) */
int cfb_bilateral_filter(const float* depth, size_t depth_pitch, int W, int H, float maxD, float* out,
                         size_t out_pitch, void* stream);
/* pyrDownGaussF (Core/Cuda/cudafuncs.cu:510-532); dst is (sh/2) x (sw/2) */
int cfb_pyr_down_gauss_f(const float* src, size_t src_pitch, int sw, int sh, float* dst, size_t dst_pitch,
                         void* stream);
/* pyrDownUcharGauss (cudafuncs.cu:566-588) */
int cfb_pyr_down_uchar_gauss(const uint8_t* src, size_t src_pitch, int sw, int sh, uint8_t* dst,
                             size_t dst_pitch, void* stream);
/* createVMap (cudafuncs.cu:136-150); mask/maskID are accepted by the reference but unused (:119) */
int cfb_create_vmap(float fx, float fy, float cx, float cy, const float* depth, size_t depth_pitch, int W, int H,
                    float* vmap, size_t vmap_pitch, float depthCutoff, void* stream);
/* createNMap (cudafuncs.cu:191-205) */
int cfb_create_nmap(const float* vmap, size_t vmap_pitch, int W, int H, float* nmap, size_t nmap_pitch,
                    void* stream);
/* tranformMaps [sic] (cudafuncs.cu:251-269); src may alias dst */
int cfb_tranform_maps(const float* vmap_src, size_t vs_pitch, const float* nmap_src, size_t ns_pitch, int W, int H,
                      const float Rmat[9], const float tvec[3], float* vmap_dst, size_t vd_pitch,
                      float* nmap_dst, size_t nd_pitch, void* stream);
/* copyMaps (cudafuncs.cu:313-331): AoS float4 W*H -> planar */
int cfb_copy_maps(const float* vmap_src4, const float* nmap_src4, int W, int H, float* vmap_dst, size_t vd_pitch,
                  float* nmap_dst, size_t nd_pitch, void* stream);
/* resizeVMap / resizeNMap (cudafuncs.cu:437-445); output is (sh/2) rows per plane, sw/2 cols */
int cfb_resize_vmap(const float* in, size_t in_pitch, int sw, int sh, float* out, size_t out_pitch, void* stream);
int cfb_resize_nmap(const float* in, size_t in_pitch, int sw, int sh, float* out, size_t out_pitch, void* stream);
/* verticesToDepth (cudafuncs.cu:615-622) */
int cfb_vertices_to_depth(const float* vmap_src4, int W, int H, float* dst, size_t dst_pitch, float cutOff,
                          void* stream);
/* imageBGRToIntensity (cudafuncs.cu:641-653): source is an interleaved u8 image with `channels`
 * bytes per pixel (3 or 4) instead of a GL-mapped cudaArray */
int cfb_image_bgr_to_intensity(const uint8_t* img, size_t img_pitch, int channels, int W, int H, uint8_t* dst,
                               size_t dst_pitch, void* stream);
/* computeDerivativeImages (cudafuncs.cu:685-715) */
int cfb_compute_derivative_images(const uint8_t* src, size_t src_pitch, int W, int H, int16_t* dx, int16_t* dy,
                                  size_t grad_pitch, void* stream);
/* projectToPointCloud (cudafuncs.cu:738-751): intrinsics are those of `level` already applied by
 * the caller (fx/2^level ...); cloud is AoS float3 */
int cfb_project_to_point_cloud(const float* depth, size_t depth_pitch, int W, int H, float fx, float fy, float cx,
                               float cy, float* cloud3, size_t cloud_pitch, void* stream);

/* Scratch for the reduction steps (the `sum`/`out` DeviceArrays of the reference signatures).
 * Allocate cfb_step_scratch_bytes() of device memory, zero it once, reuse. */
size_t cfb_step_scratch_bytes(void);

/* icpStep (Core/Cuda/reduce.cu:425-499).  Outputs on the host: A 6x6, b 6, residual {sum r^2, inliers}.
 * error_map (device, optional) replaces the cudaSurfaceObject (reduce.cu:301,:325). */
int cfb_icp_step(const float Rcurr[9], const float tcurr[3], const float* vmap_curr, size_t vc_pitch,
                 const float* nmap_curr, size_t nc_pitch, const float Rprev_inv[9], const float tprev[3],
                 float fx, float fy, float cx, float cy, const float* vmap_g_prev, size_t vp_pitch,
                 const float* nmap_g_prev, size_t np_pitch, float distThres, float angleThres, int W, int H,
                 void* scratch, float* matrixA_host, float* vectorB_host, float* residual_host,
                 float* error_map, size_t error_pitch, void* stream);
/* computeRgbResidual (reduce.cu:893-971). corresImg: device, W*H 16-byte DataTerm, unpitched. */
int cfb_compute_rgb_residual(float minScale, const int16_t* dIdx, const int16_t* dIdy, size_t grad_pitch,
                             const float* lastDepth, const float* nextDepth, size_t depth_pitch,
                             const uint8_t* lastImage, const uint8_t* nextImage, size_t img_pitch,
                             void* corresImg, void* scratch, float maxDepthDelta, const float kt[3],
                             const float krkinv[9], int W, int H, int* sigmaSum, int* count, void* stream);
/* rgbStep (reduce.cu:635-687) */
int cfb_rgb_step(const void* corresImg, float sigma, const float* cloud3, size_t cloud_pitch, float fx, float fy,
                 const int16_t* dIdx, const int16_t* dIdy, size_t grad_pitch, float sobelScale, int W, int H,
                 void* scratch, float* matrixA_host, float* vectorB_host, void* stream);
/* so3Step (reduce.cu:1118-1176): A 3x3, b 3 */
int cfb_so3_step(const uint8_t* lastImage, const uint8_t* nextImage, size_t img_pitch, const float imageBasis[9],
                 const float kinv[9], const float krlr[9], int W, int H, void* scratch, float* matrixA_host,
                 float* vectorB_host, float* residual_host, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Seam 2a: RGBDOdometry (Core/Utils/RGBDOdometry.h)
 * ---------------------------------------------------------------------------------------------- */
typedef struct cfb_odom cfb_odom;

typedef struct cfb_track_stats { /* RGBDOdometry.h:62-70 */
  float lastICPError, lastICPCount, lastRGBError, lastRGBCount, lastSO3Error, lastSO3Count;
  double lastA[36];
  double lastb[6];
  int so3_iterations;
  int pad_;
} cfb_track_stats;

int cfb_odom_create(int width, int height, float cx, float cy, float fx, float fy, float distThresh,
                    float angleThresh, cfb_odom** out);
void cfb_odom_destroy(cfb_odom* o);
/* initICP(depthPyramid, maskPyramid, depthCutoff) (RGBDOdometry.cpp:110-118): 3 device depth levels */
int cfb_odom_init_icp(cfb_odom* o, const float* const depth_pyr[3], const size_t pitch[3], float depthCutoff,
                      void* stream);
/* initICPModel (RGBDOdometry.cpp:143-175): device AoS float4 vertex/normal predictions, host pose */
int cfb_odom_init_icp_model(cfb_odom* o, const float* vertices4, const float* normals4, float depthCutoff,
                            const float modelPose[16], void* stream);
/* initRGBModel / initRGB / initFirstRGB (RGBDOdometry.cpp:196-215): device interleaved u8 image */
int cfb_odom_init_rgb_model(cfb_odom* o, const uint8_t* img, size_t pitch, int channels, void* stream);
int cfb_odom_init_rgb(cfb_odom* o, const uint8_t* img, size_t pitch, int channels, void* stream);
int cfb_odom_init_first_rgb(cfb_odom* o, const uint8_t* img, size_t pitch, int channels, void* stream);
/* getIncrementalTransformation (RGBDOdometry.cpp:217-477). trans/rot host in/out.
 * force_host_loop != 0 selects the generic per-step host loop even for default flags. */
int cfb_odom_get_incremental_transformation(cfb_odom* o, float trans[3], float rot[9], int rgbOnly,
                                            float icpWeight, int pyramid, int fastOdom, int so3,
                                            float* icp_error_map, size_t error_pitch, int force_host_loop,
                                            cfb_track_stats* stats_out, void* stream);
/* Measurement aid: CUDA events around the dominant tracker kernel on the stream it is launched on;
 * cfb_odom_kernel_timing returns the accumulated milliseconds and launch count (optionally resets). */
int cfb_odom_enable_kernel_timing(cfb_odom* o, int on);
int cfb_odom_kernel_timing(cfb_odom* o, double* sum_ms, int* launches, int reset);
/* Profiling aid: device buffer of >= 2048 uint64 that receives a %globaltimer trace of the
 * persistent kernel's phases (NULL disables). */
int cfb_odom_set_debug_trace(cfb_odom* o, void* dev_u64);
/* device views of the internal pyramids. which: 0 vmap_curr 1 nmap_curr 2 vmap_g_prev 3 nmap_g_prev
 * 4 lastDepth 5 nextDepth 6 lastImage 7 nextImage 8 dIdx 9 dIdy 10 lastNextImage 11 cloud 12 corres */
int cfb_odom_view(cfb_odom* o, int which, int level, const void** dev_ptr, size_t* pitch);

/* ------------------------------------------------------------------------------------------------
 * Seam 2b: CoFusion::processFrame's calls into Model / ModelProjection, without OpenGL
 * ---------------------------------------------------------------------------------------------- */
typedef struct cfb_ctx cfb_ctx;     /* per-device frame state shared by all models (CoFusion textures) */
typedef struct cfb_model cfb_model; /* Core/Model/Model.h */

/* replaces the Resolution / Intrinsics singletons (Core/Utils/Resolution.h, Intrinsics.h) */
int cfb_ctx_create(int device, int W, int H, float fx, float fy, float cx, float cy, cfb_ctx** out);
void cfb_ctx_destroy(cfb_ctx* c);
/* the CUDA stream every ctx/model call is enqueued on (cudaStream_t) */
void* cfb_ctx_stream(cfb_ctx* c);
/* CoFusion::processFrame :179-197: host RGB8 (HxWx3), metric f32 depth, optional u8 label mask
 * (NULL = everything background).  Asynchronous H2D; pinned host buffers are used in place. */
int cfb_ctx_upload_frame(cfb_ctx* c, const uint8_t* rgb_hwc, const float* depth, const uint8_t* mask);
/* same with inputs already in device memory */
int cfb_ctx_set_frame_device(cfb_ctx* c, const uint8_t* rgb_hwc, const float* depth, const uint8_t* mask);
/* CoFusion::filterDepth (:567-574) + Model::generateCUDATextures (Model.cpp:319-348) */
int cfb_ctx_preprocess(cfb_ctx* c, float depthCutoff);
int cfb_ctx_sync(cfb_ctx* c);
/* which: 0 rgb(u8x3) 1 depthRaw 2 depthFiltered 3 depthPyr[1] 4 depthPyr[2] 5 mask */
int cfb_ctx_view(cfb_ctx* c, int which, const void** dev_ptr, size_t* pitch);
/* kernels launched by ctx/model calls since the last call (bench accounting); resets the counter */
int cfb_ctx_take_launch_count(cfb_ctx* c);

typedef struct cfb_track_params { /* arguments of Model::performTracking (Model.h:128-129) */
  int frameToFrameRGB, rgbOnly;
  float icpWeight;
  int pyramid, fastOdom, so3;
  float maxDepthProcessed;
  int force_host_loop;
} cfb_track_params;

/* Model::Model (Model.h:100-103).  max_surfels replaces COFUSION_NUM_SURFELS / TEXTURE_DIMENSION^2
 * (Model.cpp:92-98); enable_fill_in as the reference's enableFillIn (true only for the background). */
int cfb_model_create(cfb_ctx* c, unsigned id, float confidenceThreshold, unsigned max_surfels, int enable_fill_in,
                     cfb_model** out);
void cfb_model_destroy(cfb_model* m);
int cfb_model_get_pose(cfb_model* m, float pose[16]);
int cfb_model_override_pose(cfb_model* m, const float pose[16]); /* Model::overridePose (Model.h:218-221) */
/* pose <- `pose` while lastPose keeps its value: the state Model::performTracking leaves behind
 * (lastPose = pose; pose = tracked), for callers that track elsewhere (ground-truth / tests) */
int cfb_model_set_pose_keep_last(cfb_model* m, const float pose[16]);
/* install prediction images rendered elsewhere (AoS float4 vertex+conf, normal+radius, RGB8/RGBA8) */
int cfb_model_set_prediction(cfb_model* m, const float* vertices4, const float* normals4, const uint8_t* img,
                             int channels, int device_ptrs);
/* RGBDOdometry::initFirstRGB on the current frame (CoFusion.cpp:205) */
int cfb_model_init_first_rgb(cfb_model* m);
/* Model::performTracking (Model.cpp:369-389): pose is updated in the model and returned */
int cfb_model_perform_tracking(cfb_model* m, const cfb_track_params* p, float pose_out[16],
                               cfb_track_stats* stats_out);
/* Model::setConfidenceThreshold / setMaxDepth (Model.h:161-165) */
int cfb_model_set_confidence_threshold(cfb_model* m, float confThresh);
int cfb_model_set_max_depth(cfb_model* m, float d);
/* Model::getID / getConfidenceThreshold / getMaxDepth (Model.h:160-166) */
int cfb_model_get_info(cfb_model* m, unsigned* id, float* confThresh, float* maxDepth);
/* Model::initialise (Model.cpp:227-272) + CoFusion::computeFeedbackBuffers (CoFusion.cpp:161-169):
 * surfels from the current frame's raw + filtered depth */
int cfb_model_initialise(cfb_model* m, int time, float maxDepthProcessed);
/* Model::predictIndices -> ModelProjection::predictIndices (ModelProjection.cpp:105-157) */
int cfb_model_predict_indices(cfb_model* m, int time, float depthCutoff, int timeDelta);
/* Model::fuse (Model.cpp:408-563) against the current frame of the context */
int cfb_model_fuse(cfb_model* m, int time, float depthCutoff, float weightMultiplier);
/* Model::clean (Model.cpp:565-697); outlierCoefficient = GPUSetup::outlierCoefficient (GUI default 3) */
int cfb_model_clean(cfb_model* m, int time, int timeDelta, float depthCutoff, float outlierCoefficient);
/* Model::combinedPredict(ACTIVE) (ModelProjection.cpp:192-273) */
int cfb_model_combined_predict(cfb_model* m, float depthCutoff, int time, int maxTime, int timeDelta);
/* Model::performFillIn (Model.cpp:901-909) (+ CoFusion::requiresFillIn evaluated on the device) */
int cfb_model_perform_fill_in(cfb_model* m, int frameToFrameRGB, int lost);
/* Model::computeFusionWeight (Model.cpp:391-406) */
float cfb_model_compute_fusion_weight(cfb_model* m, float weightMultiplier);
/* Model::downloadMap (Model.cpp:868-899): 12 floats per surfel (pos+conf | colour,0,init,last | normal+radius) */
int cfb_model_download_map(cfb_model* m, float* dst, size_t capacity_surfels, unsigned* count_out);
/* test / restore helper: replace the map with `count` host surfels */
int cfb_model_upload_map(cfb_model* m, const float* src, unsigned count);
/* Model::lastCount (Model.h:107) */
int cfb_model_last_count(cfb_model* m, unsigned* count_out);
/* the model's tracker (frameToModel), e.g. for cfb_odom_view */
cfb_odom* cfb_model_odometry(cfb_model* m);
/* which: 0 tracker-input vertex+conf (float4) 1 tracker-input normal+radius (float4) 2 tracker-input
 * image (RGBA8) 3 ICP error (f32) | index maps: 4 index (u32) 5 vertConf 6 colorTime 7 normRad (float4)
 * | splat prediction: 8 image (RGBA8) 9 vertexConf 10 normalRad (float4) 11 time (u16)
 * | fill-in: 12 image 13 vertex 14 normal | 15 new-unstable buffer (48-B surfels) */
int cfb_model_view(cfb_model* m, int which, const void** dev_ptr, size_t* pitch);

/* ------------------------------------------------------------------------------------------------
 * Seam 2b': motion segmentation (Core/Segmentation/Segmentation.h:104-106 performSegmentationCRF,
 * Core/Segmentation/Slic.h:30-147).  CPU code in the reference (gSLICr + densecrf); here SLIC, the
 * super-pixel reductions, the CRF mean field, the component post-processing and the label upsampling
 * all run on the device; only ModelData comes back to the host.
 * ---------------------------------------------------------------------------------------------- */
typedef struct cfb_segmentation cfb_segmentation;
typedef struct cfb_seg_params { /* Segmentation.h:135-149; defaults = GUI/Tools/GUI.h:212-227 */
  int crfIterations;
  float scaleFeaturesRGB, scaleFeaturesDepth, scaleFeaturesPos;
  float weightAppearance, weightSmoothness;
  float unaryThresholdNew, unaryKError, unaryWeightError;
  float maxRelSizeNew, minRelSizeNew;
} cfb_seg_params;
typedef struct cfb_model_data { /* SegmentationResult::ModelData (Segmentation.h:41-67) */
  unsigned id;
  unsigned superPixelCount;
  float avgConfidence, depthMean, depthStd;
  unsigned short top, right, bottom, left;
} cfb_model_data;
#define CFB_SEG_MAX_MODELS 15
void cfb_seg_default_params(cfb_seg_params* p);
/* W and H must be multiples of 16 (the super-pixel size, Segmentation.cpp:55) */
int cfb_segmentation_create(int device, int W, int H, cfb_segmentation** out);
void cfb_segmentation_destroy(cfb_segmentation* s);
/* Slic::setInputImage + processFrame (Slic.cpp:48-80): rgb HxWx3 u8 (device) -> labels (view 0) */
int cfb_segmentation_slic(cfb_segmentation* s, const uint8_t* rgb, void* stream);
/* Segmentation::performSegmentationCRF(models, frame, nextModelID, allowNew).  rgb (HxWx3 u8), depth
 * (HxW f32, raw metres), icpError[m] (HxW f32, Model::downloadICPErrorTexture), vertConf4[m] (HxW
 * float4, Model::downloadVertexConfTexture; .w read) and fullSeg (HxW u8 out:
 * SegmentationResult::fullSegmentation, model ids / 255) are DEVICE pointers; the pointer arrays, ids
 * and md_out (numModels + 1 entries) live on the host.  Synchronises the stream. */
int cfb_segmentation_perform_crf(cfb_segmentation* s, const uint8_t* rgb, const float* depth, int numModels,
                                 const unsigned char* modelIds, const float* const* icpError,
                                 const float* const* vertConf4, unsigned char nextModelID, int allowNew,
                                 const cfb_seg_params* prm, uint8_t* fullSeg, cfb_model_data* md_out, int* md_count,
                                 int* hasNewLabel, void* stream);
/* device scratch of the last call: 0 SLIC labels (i32 HxW) 1 super-pixel pixel counts (u32 N)
 * 2 unaries (f32 N x numLabels, node major) 3 low-res label map after post-processing (u8 N)
 * 4 low-res maps (f32 [1+2*numModels][N]: depth, then icp/conf per model) 5 CRF marginals Q (f32 N x L) */
int cfb_segmentation_view(cfb_segmentation* s, int which, const void** dev_ptr, size_t* bytes);

/* ------------------------------------------------------------------------------------------------
 * Seam 2c: CoFusion::processFrame (Core/CoFusion.h:67-68, Core/CoFusion.cpp:171-524)
 * ---------------------------------------------------------------------------------------------- */
typedef struct cfb_cofusion cfb_cofusion;
typedef struct cfb_cofusion_params { /* CoFusion ctor args / setters (CoFusion.h:47-66, :130-246) */
  int timeDelta;            /* 200 */
  float depthCutoff;        /* 5   (bilateral maxD) */
  float maxDepthProcessed;  /* 20  (CoFusion.cpp:51) */
  float icpWeight;          /* 10 */
  int pyramid, fastOdom, so3, frameToFrameRGB, rgbOnly; /* 1,0,1,0,0 */
  float confGlobalInit;     /* 10 */
  float confObjectInit;     /* 0.01 */
  float outlierCoefficient; /* 3 */
  unsigned maxSurfels;      /* per model (reference: 3072^2) */
  int predictBeforeFuse;    /* 0: skip the predict() of CoFusion.cpp:347 (its images are overwritten by
                               the final predict() before anything reads them without loop closure) */
  int enableMultipleModels; /* 1: run the motion segmentation after tracking and spawn / deactivate
                               object models from its result (CoFusion.cpp:227-299) */
  unsigned modelSpawnOffset;/* 20 (CoFusion.h:50) */
  cfb_seg_params seg;       /* cfb_seg_default_params */
} cfb_cofusion_params;
void cfb_cofusion_default_params(cfb_cofusion_params* p);
int cfb_cofusion_create(int device, int W, int H, float fx, float fy, float cx, float cy,
                        const cfb_cofusion_params* p, cfb_cofusion** out);
void cfb_cofusion_destroy(cfb_cofusion* f);
/* processFrame(frame, inPose = NULL, weightMultiplier, bootstrap = false).  rgb: HxWx3 u8, depth: HxW
 * f32 metres, mask: HxW u8 labels or NULL (static scene).  Host buffers unless device_ptrs != 0. */
int cfb_cofusion_process_frame(cfb_cofusion* f, const uint8_t* rgb, const float* depth, const uint8_t* mask,
                               int device_ptrs, float weightMultiplier);
/* FrameData (Core/FrameData.h:25-50) as the log readers hand it to processFrame, plus the two conversions
 * they perform on the CPU (GUI/Tools/KlgLogReader.cpp:53-84: raw u16 depth x 0.001 -> f32 metres;
 * FrameData::flipColors :38-41: BGR -> RGB), which this module runs on the device instead. */
typedef struct cfb_frame {
  const uint8_t* rgb;         /* H x W x 3, 8 bit */
  const float* depth;         /* metric f32, or NULL when depth_u16 is given */
  const uint16_t* depth_u16;  /* raw sensor units, or NULL */
  float depth_scale;          /* metres per raw unit (0.001) */
  int flip_colors;            /* != 0: the image is BGR */
  const uint8_t* mask;        /* external label image or NULL */
  int device_ptrs;            /* != 0: the pointers above are device pointers */
  int64_t timestamp;          /* FrameData::timestamp, logged with the poses (CoFusion.cpp:516) */
} cfb_frame;
/* bool CoFusion::processFrame(const FrameData& frame, const Eigen::Matrix4f* inPose, const float
 * weightMultiplier, const bool bootstrap) (Core/CoFusion.h:67-68, Core/CoFusion.cpp:170).  inPose16 (row-major
 * 4x4) NULL: regular tracking.  inPose16 && !bootstrap: the camera pose is overridden, nothing is tracked or
 * segmented (CoFusion.cpp:343-345).  bootstrap (needs inPose16): track, then pose <- pose * inPose (:219-222). */
int cfb_cofusion_process_frame_ex(cfb_cofusion* f, const cfb_frame* frame, const float* inPose16, float weightMultiplier,
                                  int bootstrap);
/* Model pose logging (Model.h:230-242, enablePoseLogging) and the exports of CoFusion.cpp:646-783.
 * pose_log: entries of model `index` -- ts[k], pose7[7k..7k+6] = t.xyz, q.xyzw: camera -> world for model 0,
 * object -> world = cameraPose * modelPose^-1 otherwise (CoFusion.cpp:503-518).  *n = entries available. */
int cfb_cofusion_enable_pose_logging(cfb_cofusion* f, int on);
int cfb_cofusion_pose_log(cfb_cofusion* f, int index, int64_t* ts, float* pose7, int capacity, int* n);
int cfb_cofusion_export_poses(cfb_cofusion* f, const char* directory); /* poses-<id>.txt (exportPoses) */
int cfb_cofusion_save_ply(cfb_cofusion* f, const char* directory);     /* cloud-<id>.ply (savePly) */
/* Object sharding over the GPUs of one node (one process per GPU): rank r owns the models spawned in ITS cfb_cofusion
 * (convention: model k of the scene on rank k % world).  cfb_nccl_unique_id on rank 0, distributed by the application;
 * cfb_cofusion_shard_init is collective.  Afterwards EVERY rank calls cfb_cofusion_process_frame(_ex) for every frame:
 * only rank 0's rgb / f32 depth / mask pointers are read (the others may pass NULL), the packed frame reaches the other
 * ranks by one ncclBroadcast, every rank filters the depth and builds the pyramids locally.  External label masks only
 * (enableMultipleModels = 0).  Replaces the implicit `for (auto model : models)` loops of Core/CoFusion.cpp:214-217,
 * :465-488, :536-542 by one loop per rank. */
int cfb_nccl_unique_id(unsigned char id[128]);
int cfb_cofusion_shard_init(cfb_cofusion* f, int rank, int world, const unsigned char id[128]);
/* CoFusion::spawnObjectModel + the first fuse of the new model (CoFusion.cpp:252-276) */
int cfb_cofusion_spawn_object_model(cfb_cofusion* f, unsigned id, const float* initialPose16);
int cfb_cofusion_num_models(cfb_cofusion* f);
int cfb_cofusion_tick(cfb_cofusion* f);
/* borrowed handles (owned by the cofusion object) */
cfb_model* cfb_cofusion_model(cfb_cofusion* f, int index);
cfb_ctx* cfb_cofusion_ctx(cfb_cofusion* f);
int cfb_cofusion_last_stats(cfb_cofusion* f, int index, cfb_track_stats* out);
/* SegmentationResult of the last frame (enableMultipleModels): up to CFB_SEG_MAX_MODELS+1 entries.
 * spawned_id: id of the model spawned by the last frame or -1; deactivated: models lost by it. */
int cfb_cofusion_last_segmentation(cfb_cofusion* f, cfb_model_data* md_out, int* md_count, int* hasNewLabel,
                                   int* spawned_id, int* deactivated);
int cfb_cofusion_num_inactive_models(cfb_cofusion* f);
/* 1 (default): all models of a frame are tracked by ONE persistent kernel launch (<= 5 per launch);
 * 0: one launch per model, as the reference's `for (auto model : models) performTracking` loop.
 * Results are bit-identical either way. */
int cfb_cofusion_set_batched_tracking(cfb_cofusion* f, int on);
/* tools only: >= 2048 u64 of device memory receiving a %globaltimer phase trace of the frame's tracker launch */
int cfb_cofusion_set_debug_trace(cfb_cofusion* f, void* dev_u64);
cfb_segmentation* cfb_cofusion_segmentation(cfb_cofusion* f); /* borrowed; NULL when segmentation is off */

#ifdef __cplusplus
}
#endif
#endif /* COFUSION_B200_H_ */
