// odometry.cu -- cfb::RGBDOdometry (see odometry.cuh).  Host orchestration of the tracker.
#include "odometry.cuh"

#include <float.h>
#include <math.h>
#include <string.h>

#include "gn_math.h"
#include "image_kernels.cuh"

namespace cfb {

#define RET_IF(e)                         \
  do {                                    \
    cudaError_t e__ = (e);                \
    if (e__ != cudaSuccess) return e__;   \
  } while (0)

namespace {
template <class T>
bool dalloc(T** p, size_t n, std::vector<std::pair<void*, size_t>>* reg) {
  if (cudaMalloc((void**)p, n * sizeof(T)) != cudaSuccess || cudaMemset(*p, 0, n * sizeof(T)) != cudaSuccess) return false;
  reg->push_back({(void*)*p, n * sizeof(T)});
  return true;
}
}  // namespace

RGBDOdometry::RGBDOdometry(int w, int h, float cx, float cy, float fx, float fy, float distThresh,
                           float angleThresh)
    : width(w), height(h), intr{fx, fy, cx, cy}, distThres_(distThresh), angleThres_(angleThresh) {
  // RGBDOdometry.cpp:31-34, :103-105
  sobelScale = (float)(1.0 / pow(2.0, 3));
  maxDepthDeltaRGB = 0.07f;
  maxDepthRGB = 6.0f;
  minimumGradientMagnitudes[0] = 5;
  minimumGradientMagnitudes[1] = 3;
  minimumGradientMagnitudes[2] = 1;
  memset(&stats_, 0, sizeof(stats_));
  bool good = true;
  for (int i = 0; i < NUM_PYRS; ++i) {
    size_t n = (size_t)(w >> i) * (h >> i);
    good = good && dalloc(&vmaps_g_prev_[i], n * 3, &zeroed_) && dalloc(&nmaps_g_prev_[i], n * 3, &zeroed_) &&
           dalloc(&vmaps_curr_[i], n * 3, &zeroed_) && dalloc(&nmaps_curr_[i], n * 3, &zeroed_) && dalloc(&lastDepth[i], n, &zeroed_) &&
           dalloc(&nextDepth[i], n, &zeroed_) && dalloc(&pointClouds[i], n * 3, &zeroed_) && dalloc(&lastImage[i], n, &zeroed_) &&
           dalloc(&nextImage[i], n, &zeroed_) && dalloc(&lastNextImage[i], n, &zeroed_) && dalloc(&nextdIdx[i], n, &zeroed_) &&
           dalloc(&nextdIdy[i], n, &zeroed_) && dalloc(&corresImg[i], n, &zeroed_) && dalloc(&rgbCand[i], n, &zeroed_);
  }
  good = good && dalloc(&vmaps_tmp, (size_t)w * h * 4, &zeroed_) && dalloc(&scratch, 1, &zeroed_) && dalloc(&gn, 1, &zeroed_) &&
         dalloc(&d_pose, 1, &zeroed_) && dalloc(&d_warp, 1, &zeroed_) && dalloc(&d_pose_in, 16, &zeroed_) &&
         dalloc((unsigned**)&grid_sync_, 256, &zeroed_);
  good = good && cudaMallocHost(&h_pinned, 4096) == cudaSuccess;
  // what the tracker needs of an OBJECT model (extents, correspondences of an iteration): here rather than inside
  // the first multi-model frame.  Sized for the largest grid the tile planner makes (one CTA per SM, <= 160).
  corr_words_ = (size_t)4 * 160 * 576;
  good = good && dalloc((int**)&d_box_, 24, &zeroed_) && cudaMalloc(&d_corr_, corr_words_ * 8) == cudaSuccess &&
         cudaMemset(d_corr_, 0, corr_words_ * 8) == cudaSuccess;
  ok_ = good;
}

// Back to the state of a freshly constructed object (a pooled Model is handed to a new object id): every device
// buffer the constructor zeroed is zeroed again on `s`; plans and tensor maps (tied to the buffers) stay.
cudaError_t RGBDOdometry::recycle(cudaStream_t s) {
  for (auto& z : zeroed_) RET_IF(cudaMemsetAsync(z.first, 0, z.second, s));
  memset(&stats_, 0, sizeof(stats_));
  next_is_last_ = false;
  return cudaSuccess;
}

RGBDOdometry::~RGBDOdometry() {
  for (int i = 0; i < NUM_PYRS; ++i) {
    cudaFree(vmaps_g_prev_[i]);
    cudaFree(nmaps_g_prev_[i]);
    cudaFree(vmaps_curr_[i]);
    cudaFree(nmaps_curr_[i]);
    cudaFree(lastDepth[i]);
    cudaFree(nextDepth[i]);
    cudaFree(pointClouds[i]);
    cudaFree(lastImage[i]);
    cudaFree(nextImage[i]);
    cudaFree(lastNextImage[i]);
    cudaFree(nextdIdx[i]);
    cudaFree(nextdIdy[i]);
    cudaFree(corresImg[i]);
    cudaFree(rgbCand[i]);
  }
  cudaFree(d_pose_in);
  cudaFree(grid_sync_);
  cudaFree(tiled_scratch_);
  cudaFree(d_box_);
  cudaFree(d_corr_);
  destroyTiled();
  if (ev_k0_) cudaEventDestroy(ev_k0_);
  if (ev_k1_) cudaEventDestroy(ev_k1_);
  cudaFree(vmaps_tmp);
  cudaFree(scratch);
  cudaFree(gn);
  cudaFree(d_pose);
  cudaFree(d_warp);
  cudaFreeHost(h_pinned);
}

const void* RGBDOdometry::view(int which, int level, size_t* pitch) const {
  size_t w = (size_t)(width >> level);
  switch (which) {
    case 0: *pitch = w * 4; return vmaps_curr_[level];
    case 1: *pitch = w * 4; return nmaps_curr_[level];
    case 2: *pitch = w * 4; return vmaps_g_prev_[level];
    case 3: *pitch = w * 4; return nmaps_g_prev_[level];
    case 4: *pitch = w * 4; return lastDepth[level];
    case 5: *pitch = w * 4; return next_is_last_ ? lastDepth[level] : nextDepth[level];
    case 6: *pitch = w; return lastImage[level];
    case 7: *pitch = w; return nextImage[level];
    case 8: *pitch = w * 2; return nextdIdx[level];
    case 9: *pitch = w * 2; return nextdIdy[level];
    case 10: *pitch = w; return lastNextImage[level];
    case 11: *pitch = w * 12; return pointClouds[level];
    case 12: *pitch = w * 16; return corresImg[level];
  }
  *pitch = 0;
  return nullptr;
}

cudaError_t RGBDOdometry::initICP(const float* const depthPyr[NUM_PYRS], const size_t pitch[NUM_PYRS],
                                  float depthCutoff, cudaStream_t s) {
  for (int i = 0; i < NUM_PYRS; ++i) {
    int w = width >> i, h = height >> i;
    RET_IF(launch_create_vmap(depthPyr[i], pitch[i], w, h, intr.level(i), depthCutoff, vmaps_curr_[i],
                              (size_t)w * 4, s));
    RET_IF(launch_create_nmap(vmaps_curr_[i], (size_t)w * 4, w, h, nmaps_curr_[i], (size_t)w * 4, s));
  }
  return cudaSuccess;
}

cudaError_t RGBDOdometry::initICPModel(const float* v4, const float* n4, float /*depthCutoff*/,
                                       const float pose[16], cudaStream_t s) {
  RET_IF(cudaMemcpyAsync(vmaps_tmp, v4, (size_t)width * height * 16, cudaMemcpyDeviceToDevice, s));
  RET_IF(launch_copy_maps(v4, n4, width, height, vmaps_g_prev_[0], (size_t)width * 4, nmaps_g_prev_[0],
                          (size_t)width * 4, s));
  for (int i = 1; i < NUM_PYRS; ++i) {
    int sw = width >> (i - 1), sh = height >> (i - 1);
    RET_IF(launch_resize_map(vmaps_g_prev_[i - 1], (size_t)sw * 4, sw, sh, false, vmaps_g_prev_[i],
                             (size_t)(sw / 2) * 4, s));
    RET_IF(launch_resize_map(nmaps_g_prev_[i - 1], (size_t)sw * 4, sw, sh, true, nmaps_g_prev_[i],
                             (size_t)(sw / 2) * 4, s));
  }
  Mat33 R;
  float t[3];
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) R.m[r * 3 + c] = pose[r * 4 + c];
    t[r] = pose[r * 4 + 3];
  }
  for (int i = 0; i < NUM_PYRS; ++i) {
    int w = width >> i, h = height >> i;
    size_t p = (size_t)w * 4;
    RET_IF(launch_transform_maps(vmaps_g_prev_[i], p, nmaps_g_prev_[i], p, w, h, R, t, vmaps_g_prev_[i], p,
                                 nmaps_g_prev_[i], p, s));
  }
  return cudaSuccess;
}

cudaError_t RGBDOdometry::populateRGBDData(const unsigned char* img, size_t pitch, int channels,
                                           float* const* destDepths, unsigned char* const* destImages,
                                           cudaStream_t s) {
  RET_IF(launch_vertices_to_depth(vmaps_tmp, width, height, maxDepthRGB, destDepths[0], (size_t)width * 4, s));
  for (int i = 0; i + 1 < NUM_PYRS; i++) {
    int sw = width >> i, sh = height >> i;
    RET_IF(launch_pyr_down_gauss_f(destDepths[i], (size_t)sw * 4, sw, sh, destDepths[i + 1], (size_t)(sw / 2) * 4, s));
  }
  RET_IF(launch_rgb_to_intensity(img, pitch, channels, width, height, destImages[0], (size_t)width, s));
  for (int i = 0; i + 1 < NUM_PYRS; i++) {
    int sw = width >> i, sh = height >> i;
    RET_IF(launch_pyr_down_uchar(destImages[i], (size_t)sw, sw, sh, destImages[i + 1], (size_t)(sw / 2), s));
  }
  return cudaSuccess;
}

cudaError_t RGBDOdometry::initRGBModel(const unsigned char* img, size_t pitch, int channels, cudaStream_t s) {
  return populateRGBDData(img, pitch, channels, lastDepth, lastImage, s);
}
cudaError_t RGBDOdometry::initRGB(const unsigned char* img, size_t pitch, int channels, cudaStream_t s) {
  next_is_last_ = false;
  return populateRGBDData(img, pitch, channels, nextDepth, nextImage, s);
}
cudaError_t RGBDOdometry::initFirstRGB(const unsigned char* img, size_t pitch, int channels, cudaStream_t s) {
  RET_IF(launch_rgb_to_intensity(img, pitch, channels, width, height, lastNextImage[0], (size_t)width, s));
  for (int i = 0; i + 1 < NUM_PYRS; i++) {
    int sw = width >> i, sh = height >> i;
    RET_IF(launch_pyr_down_uchar(lastNextImage[i], (size_t)sw, sw, sh, lastNextImage[i + 1], (size_t)(sw / 2), s));
  }
  return cudaSuccess;
}

cudaError_t RGBDOdometry::initAll(const float* v4, const float* n4, const unsigned char* modelImg, int modelCh,
                                  const float* const depthPyr[NUM_PYRS], const unsigned char* frameImg, int frameCh,
                                  float depthCutoff, const float pose[16], cudaStream_t s, const float* pose34_dev,
                                  const PredAlt* alt) {
  if ((width % 4) || (height % 4)) return cudaErrorInvalidValue;
  Mat33 R;
  float t[3];
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) R.m[r * 3 + c] = pose[r * 4 + c];
    t[r] = pose[r * 4 + 3];
  }
  // model side: global-frame vertex/normal pyramid + lastDepth level 0
  RET_IF(launch_model_pyramid(v4, n4, width, height, R, t, maxDepthRGB, vmaps_g_prev_, nmaps_g_prev_, lastDepth[0], s,
                              pose34_dev, alt));
  // quirk kept: initRGB derives nextDepth from the same model prediction (vmaps_tmp) -> it IS
  // lastDepth; the device loop reads lastDepth for both instead of building a second copy
  next_is_last_ = true;
  // frame side
  // + both grey images (model prediction, frame) in the same launch
  RET_IF(launch_frame_maps(depthPyr, width, height, intr, depthCutoff, vmaps_curr_, nmaps_curr_, s, modelImg, modelCh, lastImage[0],
                           frameImg, frameCh, nextImage[0], alt));
  {  // lastDepth + both grey images, both levels each, in ONE launch
    const void* src[3] = {lastDepth[0], lastImage[0], nextImage[0]};
    void* l1[3] = {lastDepth[1], lastImage[1], nextImage[1]};
    void* l2[3] = {lastDepth[2], lastImage[2], nextImage[2]};
    const int u8[3] = {0, 1, 1};
    RET_IF(launch_pyramid2(3, src, l1, l2, u8, width, height, s));
  }
  return cudaSuccess;
}

cudaError_t RGBDOdometry::getIncrementalTransformation(float trans[3], float rot[9], bool rgbOnly,
                                                       float icpWeight, bool pyramid, bool fastOdom, bool so3,
                                                       float* err, size_t err_pitch, bool force_host_loop,
                                                       cudaStream_t s) {
  bool icp = !rgbOnly && icpWeight > 0;
  bool rgb = rgbOnly || icpWeight < 100;
  if (!force_host_loop && icp && rgb) {
    if (!tiled_scratch_) {
      RET_IF(cudaMalloc(&tiled_scratch_, tiledScratchBytes()));
      RET_IF(cudaMemsetAsync(tiled_scratch_, 0, tiledScratchBytes(), s));
    }
    RGBDOdometry* od[1] = {this};
    float* errs[1] = {err};
    return trackTiled(od, 1, (float(*)[3])trans, (float(*)[9])rot, icpWeight, pyramid, fastOdom, so3, errs, err_pitch,
                      tiled_scratch_, s);
  }
  return hostLoop(trans, rot, rgbOnly, icpWeight, pyramid, fastOdom, so3, err, err_pitch, s);
}

// ------------------------------------------------------------------------------------------------
// Generic host loop: RGBDOdometry.cpp:217-477 step for step.
cudaError_t RGBDOdometry::hostLoop(float trans[3], float rot[9], bool rgbOnly, float icpWeight, bool pyramid,
                                   bool fastOdom, bool so3, float* err, size_t err_pitch, cudaStream_t s) {
  bool icp = !rgbOnly && icpWeight > 0;
  bool rgb = rgbOnly || icpWeight < 100;
  float Rprev[9], tprev[3], Rcurr[9], tcurr[3];
  memcpy(Rprev, rot, sizeof(Rprev));
  memcpy(tprev, trans, sizeof(tprev));
  memcpy(Rcurr, rot, sizeof(Rcurr));
  memcpy(tcurr, trans, sizeof(tcurr));
  TrackStats st;
  memset(&st, 0, sizeof(st));
  float* hres = (float*)h_pinned;         // 32 floats
  int* hcnt = (int*)((char*)h_pinned + 256);  // 2 ints

  if (rgb)
    for (int i = 0; i < NUM_PYRS; i++) {
      int w = width >> i, h = height >> i;
      RET_IF(launch_derivative_images(nextImage[i], (size_t)w, w, h, nextdIdx[i], nextdIdy[i], (size_t)w * 2, s));
    }

  double resultR[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  if (so3) {
    const int L = 2;
    Intr k = intr.level(L);
    double K[9], Kinv[9];
    gn::make_K(k.fx, k.fy, k.cx, k.cy, K, Kinv);
    float R_lr[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    float lastError = FLT_MAX / 2, lastCount = FLT_MAX / 2;
    double lastResultR[9];
    memcpy(lastResultR, resultR, sizeof(resultR));
    for (int it = 0; it < 10; it++) {
      double tmp[9], H[9], KR[9];
      gn::mul3(K, resultR, KR);
      gn::mul3(KR, Kinv, H);
      (void)tmp;
      So3Args a;
      a.lastImage = lastNextImage[L];
      a.nextImage = nextImage[L];
      a.img_pitch = (size_t)(width >> L);
      a.cols = width >> L;
      a.rows = height >> L;
      for (int q = 0; q < 9; ++q) {
        a.imageBasis.m[q] = (float)H[q];
        a.kinv.m[q] = (float)Kinv[q];
        a.krlr.m[q] = (float)KR[q];
      }
      RET_IF(launch_so3_step(a, scratch, s));
      RET_IF(cudaMemcpyAsync(hres, scratch->result, 32 * sizeof(float), cudaMemcpyDeviceToHost, s));
      RET_IF(cudaStreamSynchronize(s));
      st.so3_iterations++;
      float jtj[9], jtr[3];
      gn::unpack_so3(hres, jtj, jtr);
      st.lastSO3Error = sqrtf(hres[9]) / hres[10];
      st.lastSO3Count = hres[10];
      if (st.lastSO3Error < lastError && fabsf(lastError - st.lastSO3Count) < 0.001f) {
        break;
      } else if (st.lastSO3Error > lastError + 0.001f) {
        st.lastSO3Error = lastError;
        st.lastSO3Count = lastCount;
        memcpy(resultR, lastResultR, sizeof(resultR));
        break;
      }
      lastError = st.lastSO3Error;
      lastCount = st.lastSO3Count;
      memcpy(lastResultR, resultR, sizeof(resultR));
      double Ad[9], bd[3], xd[3];
      for (int q = 0; q < 9; ++q) Ad[q] = jtj[q];
      for (int q = 0; q < 3; ++q) bd[q] = jtr[q];
      gn::ldlt_solve<3>(Ad, bd, xd);
      double delta[3] = {(double)(float)xd[0], (double)(float)xd[1], (double)(float)xd[2]};
      double rotUpdate[9];
      gn::rodrigues(delta, rotUpdate);
      float ru[9], nr[9];
      for (int q = 0; q < 9; ++q) ru[q] = (float)rotUpdate[q];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c)
          nr[r * 3 + c] = ru[r * 3] * R_lr[c] + ru[r * 3 + 1] * R_lr[3 + c] + ru[r * 3 + 2] * R_lr[6 + c];
      memcpy(R_lr, nr, sizeof(nr));
      for (int q = 0; q < 9; ++q) resultR[q] = R_lr[q];
    }
  }

  int iterations[NUM_PYRS];
  iterations[0] = fastOdom ? 3 : 10;
  iterations[1] = pyramid ? 5 : 0;
  iterations[2] = pyramid ? 4 : 0;

  float Rprev_inv[9];
  gn::inverse3f(Rprev, Rprev_inv);
  double resultRt[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  if (so3)
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) resultRt[r * 4 + c] = resultR[r * 3 + c];

  IcpPose* hpose = (IcpPose*)((char*)h_pinned + 512);
  RgbWarp* hwarp = (RgbWarp*)((char*)h_pinned + 1024);

  for (int i = NUM_PYRS - 1; i >= 0; i--) {
    const int w = width >> i, h = height >> i;
    const Intr k = intr.level(i);
    if (rgb)
      RET_IF(launch_project_to_point_cloud(lastDepth[i], (size_t)w * 4, w, h, k, pointClouds[i], (size_t)w * 12, s));
    double K[9], Kinv[9];
    gn::make_K(k.fx, k.fy, k.cx, k.cy, K, Kinv);
    float lastRGBError = FLT_MAX;
    for (int j = 0; j < iterations[i]; j++) {
      int sigma = 0, rgbSize = 0;
      if (rgb) {
        gn::pose_to_warp(resultRt, K, Kinv, hwarp->krkinv.m, hwarp->kt);
        RET_IF(cudaMemcpyAsync(d_warp, hwarp, sizeof(RgbWarp), cudaMemcpyHostToDevice, s));
        RgbResidualArgs a;
        a.minScale = (float)(pow(minimumGradientMagnitudes[i], 2.0) / pow(sobelScale, 2.0));
        a.maxDepthDelta = maxDepthDeltaRGB;
        a.dIdx = nextdIdx[i];
        a.dIdy = nextdIdy[i];
        a.grad_pitch = (size_t)w * 2;
        a.lastDepth = lastDepth[i];
        a.nextDepth = next_is_last_ ? lastDepth[i] : nextDepth[i];
        a.depth_pitch = (size_t)w * 4;
        a.lastImage = lastImage[i];
        a.nextImage = nextImage[i];
        a.img_pitch = (size_t)w;
        a.corres = corresImg[i];
        a.cols = w;
        a.rows = h;
        RET_IF(launch_rgb_residual(a, d_warp, scratch, s));
        RET_IF(cudaMemcpyAsync(hcnt, &scratch->rgb_count, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
        RET_IF(cudaStreamSynchronize(s));
        rgbSize = hcnt[0];
        sigma = hcnt[1];
      }
      float tmpError = (float)(sqrt((double)sigma) / (double)rgbSize);
      float sigmaVal = (tmpError == 0) ? 1 : (float)rgbSize;
      if (rgbOnly && tmpError > lastRGBError) break;
      lastRGBError = tmpError;
      st.lastRGBError = tmpError;
      st.lastRGBCount = (float)rgbSize;
      if (rgbOnly) sigmaVal = -1;

      float A_icp[36], b_icp[6], residual[2] = {0, 0};
      memset(A_icp, 0, sizeof(A_icp));
      memset(b_icp, 0, sizeof(b_icp));
      if (icp) {
        memcpy(hpose->Rcurr.m, Rcurr, sizeof(Rcurr));
        memcpy(hpose->tcurr, tcurr, sizeof(tcurr));
        memcpy(hpose->Rprev_inv.m, Rprev_inv, sizeof(Rprev_inv));
        memcpy(hpose->tprev, tprev, sizeof(tprev));
        RET_IF(cudaMemcpyAsync(d_pose, hpose, sizeof(IcpPose), cudaMemcpyHostToDevice, s));
        IcpArgs a;
        size_t p = (size_t)w * 4;
        a.vmap_curr = {vmaps_curr_[i], p};
        a.nmap_curr = {nmaps_curr_[i], p};
        a.vmap_g_prev = {vmaps_g_prev_[i], p};
        a.nmap_g_prev = {nmaps_g_prev_[i], p};
        a.intr = k;
        a.distThres = distThres_;
        a.angleThres = angleThres_;
        a.cols = w;
        a.rows = h;
        bool last = (i == 0 && j == iterations[i] - 1);
        a.error_map = last ? err : nullptr;
        a.error_pitch = err_pitch;
        RET_IF(launch_icp_step(a, d_pose, scratch, s));
        RET_IF(cudaMemcpyAsync(hres, scratch->result, 32 * sizeof(float), cudaMemcpyDeviceToHost, s));
        RET_IF(cudaStreamSynchronize(s));
        gn::unpack_se3(hres, A_icp, b_icp);
        residual[0] = hres[27];
        residual[1] = hres[28];
      }
      st.lastICPError = sqrtf(residual[0]) / residual[1];
      st.lastICPCount = residual[1];

      float A_rgbd[36], b_rgbd[6];
      memset(A_rgbd, 0, sizeof(A_rgbd));
      memset(b_rgbd, 0, sizeof(b_rgbd));
      if (rgb) {
        RgbStepArgs a;
        a.corres = corresImg[i];
        a.cloud = pointClouds[i];
        a.cloud_pitch = (size_t)w * 12;
        a.dIdx = nextdIdx[i];
        a.dIdy = nextdIdy[i];
        a.grad_pitch = (size_t)w * 2;
        a.fx = k.fx;
        a.fy = k.fy;
        a.sobelScale = sobelScale;
        a.cols = w;
        a.rows = h;
        RET_IF(launch_rgb_step(a, sigmaVal, scratch, s));
        RET_IF(cudaMemcpyAsync(hres, scratch->result, 32 * sizeof(float), cudaMemcpyDeviceToHost, s));
        RET_IF(cudaStreamSynchronize(s));
        gn::unpack_se3(hres, A_rgbd, b_rgbd);
      }

      if (icp && rgb) {
        double wgt = icpWeight;
        for (int q = 0; q < 36; ++q) st.lastA[q] = (double)A_rgbd[q] + wgt * wgt * (double)A_icp[q];
        for (int q = 0; q < 6; ++q) st.lastb[q] = (double)b_rgbd[q] + wgt * (double)b_icp[q];
      } else if (icp) {
        for (int q = 0; q < 36; ++q) st.lastA[q] = A_icp[q];
        for (int q = 0; q < 6; ++q) st.lastb[q] = b_icp[q];
      } else {
        for (int q = 0; q < 36; ++q) st.lastA[q] = A_rgbd[q];
        for (int q = 0; q < 6; ++q) st.lastb[q] = b_rgbd[q];
      }
      double result[6];
      gn::ldlt_solve<6>(st.lastA, st.lastb, result);
      gn::update_se3(resultRt, result);
      gn::compose_pose(Rprev, tprev, resultRt, Rcurr, tcurr);
    }
  }

  if (rgb) {
    float d[3] = {tcurr[0] - tprev[0], tcurr[1] - tprev[1], tcurr[2] - tprev[2]};
    if (sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]) > 0.3f) {
      memcpy(Rcurr, Rprev, sizeof(Rcurr));
      memcpy(tcurr, tprev, sizeof(tcurr));
    }
  }
  if (so3)
    for (int i = 0; i < NUM_PYRS; i++) {
      unsigned char* t = lastNextImage[i];
      lastNextImage[i] = nextImage[i];
      nextImage[i] = t;
    }
  memcpy(trans, tcurr, sizeof(tcurr));
  memcpy(rot, Rcurr, sizeof(Rcurr));
  stats_ = st;
  return cudaSuccess;
}

}  // namespace cfb
