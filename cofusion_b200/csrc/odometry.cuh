// odometry.cuh -- cfb::RGBDOdometry, the host-side mirror of the reference tracker class
// (Core/Utils/RGBDOdometry.h:31-139): same method names, argument meaning and call order, but
//   * no GL textures: model predictions arrive as device pointers (AoS float4 maps, u8 image);
//   * every device buffer is allocated once in the constructor (the reference allocates inside the
//     hot loop, reduce.cu:958, cudafuncs.cu:525/:581);
//   * no cudaDeviceSynchronize inside: everything is enqueued on one stream.
// Two execution paths for getIncrementalTransformation:
//   HostLoop   - generic (all flag combinations); taken when ICP or RGB is off (rgbOnly, icpWeight <= 0
//                or >= 100) or force_host_loop is set: one fused launch per step, one stream sync + tiny
//                D2H per step, FP64 GN step on the host (gn_math.h).  Mirrors the reference loop 1:1.
//   Persistent - ICP and RGB both on (the default flags): the whole SO3 + GN sequence is ONE persistent
//                cooperative kernel over shared-memory tiles (gn_tiled.cu, trackTiled) that runs the FP64
//                GN step on the device; the host reads back pose + stats once per frame.
#pragma once
#include <utility>
#include <vector>

#include "cfb_common.cuh"
#include "image_kernels.cuh"
#include "tracker_kernels.cuh"

namespace cfb {

struct PoseDev;  // per-model device pose block (surfel_kernels.cuh)

struct TrackStats {  // RGBDOdometry.h:62-70
  float lastICPError, lastICPCount, lastRGBError, lastRGBCount, lastSO3Error, lastSO3Count;
  double lastA[36];
  double lastb[6];
  int so3_iterations;
  int pad;
};

// Device-resident Gauss-Newton state (persistent kernel).
struct GNState {
  double resultRt[16];
  double resultR[9], lastResultR[9];
  float R_lr[9];
  IcpPose pose;
  float Rprev[9];
  RgbWarp warp;
  Mat33 so3_imageBasis, so3_krlr, so3_kinv;
  float so3_lastError, so3_lastCount;
  int so3_done;
  float icp_result[32];
  float out_trans[3];
  float out_rot[9];
  TrackStats stats;
};

class RGBDOdometry {
 public:
  static const int NUM_PYRS = 3;
  RGBDOdometry(int width, int height, float cx, float cy, float fx, float fy, float distThresh = 0.10f,
               float angleThresh = 0.34202014332f /* sin(20 deg) */);
  ~RGBDOdometry();
  bool ok() const { return ok_; }

  // frame side: Model::generateCUDATextures + initICP(depth pyramid) (RGBDOdometry.cpp:110-118)
  cudaError_t initICP(const float* const depthPyr[NUM_PYRS], const size_t pitch[NUM_PYRS], float depthCutoff,
                      cudaStream_t s);
  // model side (RGBDOdometry.cpp:143-175). v4/n4: device AoS float4 W*H; pose row-major 4x4 (host)
  cudaError_t initICPModel(const float* v4, const float* n4, float depthCutoff, const float pose[16],
                           cudaStream_t s);
  // RGBDOdometry.cpp:196-204 -- both read vmaps_tmp (the model prediction), quirk kept
  cudaError_t initRGBModel(const unsigned char* img, size_t pitch, int channels, cudaStream_t s);
  cudaError_t initRGB(const unsigned char* img, size_t pitch, int channels, cudaStream_t s);
  cudaError_t initFirstRGB(const unsigned char* img, size_t pitch, int channels, cudaStream_t s);
  // initICPModel + initRGBModel + initICP + initRGB in 7 launches instead of 26 (identical results;
  // exploits that both RGB inits read the same model depth, RGBDOdometry.cpp:179,:196-204).
  // modelImg: RGBA8/RGB8 prediction image, frameImg: RGB8 frame; depthPyr: unpitched levels.
  cudaError_t initAll(const float* v4, const float* n4, const unsigned char* modelImg, int modelCh,
                      const float* const depthPyr[NUM_PYRS], const unsigned char* frameImg, int frameCh,
                      float depthCutoff, const float pose[16], cudaStream_t s,
                      const float* pose34_dev = nullptr /* device 3x4 pose: overrides `pose` without a host copy */,
                      const PredAlt* alt = nullptr /* fill-in alternative of the model prediction, chosen on the device */);

  // RGBDOdometry.cpp:217-477. trans[3], rot[9] (row-major) in/out on the host.
  // icp_error_map: optional device f32 W*H (pitch bytes) written on the last level-0 iteration.
  cudaError_t getIncrementalTransformation(float trans[3], float rot[9], bool rgbOnly, float icpWeight,
                                           bool pyramid, bool fastOdom, bool so3, float* icp_error_map,
                                           size_t error_pitch, bool force_host_loop, cudaStream_t s);
  const TrackStats& stats() const { return stats_; }

  // ---- all models of one frame in ONE persistent launch (gn_tiled.cu).  Every object had initAll() called
  // for the same frame on stream s; od[0] is the camera model (its tiles live in shared memory).
  // trans / rot: n x 3 / n x 9 host arrays (in/out), err: n device error maps (or null),
  // scratch: tiledScratchBytes() of zero-initialised device memory.
  static const int kMaxBatch = 5;
  static size_t tiledScratchBytes();
  bool canBatch(int n) const;
  static cudaError_t trackTiled(RGBDOdometry* const* od, int n, float (*trans)[3], float (*rot)[9], float icpWeight,
                                bool pyramid, bool fastOdom, bool so3, float* const* err, size_t err_pitch, void* scratch,
                                cudaStream_t s, PoseDev* const* pd = nullptr, bool async = false, bool prepared = false);
  // pd: optional per-model device pose blocks (surfel_kernels.cuh): the incoming pose is read from pd[m]->tr
  // and the kernel's epilogue refreshes the block.  async: return right after the launch -- no host
  // synchronisation, trans / rot / stats() are not updated (read statsDevice() / the pose block later).
  const TrackStats* statsDevice() const { return &gn->stats; }
  void setStats(const TrackStats& s) { stats_ = s; }
  struct TiledState;  // tile plan + tensor maps (gn_tiled.cu)

  // device views (tests / map_view): which as in oracle orc_odom_view
  const void* view(int which, int level, size_t* pitch) const;

 cudaError_t recycle(cudaStream_t s);  // see odometry.cu
 // Sobel images + photometric candidate gates, 3 levels, 1 launch (+ clears the barrier words `acnt`)
  // extents: also record the extents of the model's candidates / valid vertices per level (object models)
  cudaError_t enqueuePrepare(cudaStream_t s, void* sync_words = nullptr, int nmodels = 1, bool extents = false);

 private:
  cudaError_t populateRGBDData(const unsigned char* img, size_t pitch, int channels, float* const* destDepths,
                               unsigned char* const* destImages, cudaStream_t s);
  cudaError_t hostLoop(float trans[3], float rot[9], bool rgbOnly, float icpWeight, bool pyramid, bool fastOdom,
                       bool so3, float* err, size_t err_pitch, cudaStream_t s);
  cudaError_t prepareTiled(int nmodels);
  void destroyTiled();
  std::vector<std::pair<void*, size_t>> zeroed_;  // device buffers the constructor zero-initialised
  TiledState* tiled_ = nullptr;
  void* tiled_scratch_ = nullptr;  // single-model launches
  int* d_box_ = nullptr;           // model extents, 3 levels x 8 ints (enqueuePrepare)
  void* d_corr_ = nullptr;         // object model: per-iteration correspondences (trackTiled)
  size_t corr_words_ = 0;

  bool ok_ = false;
  int width, height;
  Intr intr;
  float distThres_, angleThres_;
  float sobelScale, maxDepthDeltaRGB, maxDepthRGB;
  float minimumGradientMagnitudes[NUM_PYRS];

  // unpitched device buffers (pitch = cols * sizeof(T))
  float *vmaps_g_prev_[NUM_PYRS], *nmaps_g_prev_[NUM_PYRS], *vmaps_curr_[NUM_PYRS], *nmaps_curr_[NUM_PYRS];
  float *lastDepth[NUM_PYRS], *nextDepth[NUM_PYRS], *pointClouds[NUM_PYRS];
  unsigned char *lastImage[NUM_PYRS], *nextImage[NUM_PYRS], *lastNextImage[NUM_PYRS];
  short *nextdIdx[NUM_PYRS], *nextdIdy[NUM_PYRS];
  DataTerm* corresImg[NUM_PYRS];
  float* vmaps_tmp;  // AoS float4 copy of the model prediction
  StepScratch* scratch;
  GNState* gn;       // device
  IcpPose* d_pose;
  RgbWarp* d_warp;
  void* h_pinned;    // pinned staging for small H2D/D2H
  unsigned char* rgbCand[NUM_PYRS];  // iteration-invariant photometric gates, one byte per pixel
  float* d_pose_in;                  // t[3], R[9] of the incoming pose
  void* grid_sync_ = nullptr;  // software grid barrier state of the persistent kernel
  void* dbg_trace_ = nullptr;
  bool time_kernel_ = false;
  cudaEvent_t ev_k0_ = nullptr, ev_k1_ = nullptr;
  bool ev_pending_ = false;
  double kernel_ms_sum_ = 0;
  int kernel_launches_ = 0;
  bool next_is_last_ = false;  // initAll(): nextDepth pyramid aliases lastDepth (reference quirk)

 public:
  // tools only: device buffer of >= 256 u64 receiving a %globaltimer trace of the persistent kernel
  void setDebugTrace(void* dev_u64) { dbg_trace_ = dev_u64; }
  // bench: CUDA-event timing of the dominant kernel (the persistent GN kernel) on its own stream
  void enableKernelTiming(bool on);
  void kernelTiming(double* sum_ms, int* launches, bool reset);

 private:
  TrackStats stats_;
};

}  // namespace cfb
