// cabi.cu -- extern "C" boundary of libcofusion_b200.so (declarations: include/cofusion_b200.h).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "../../include/cofusion_b200.h"
#include "gn_math.h"
#include "image_kernels.cuh"
#include "odometry.cuh"
#include "pipeline.cuh"
#include "cofusion.cuh"
#include "tracker_kernels.cuh"

namespace cfb {
static thread_local bool g_pdl_frame = true;
bool pdl_enabled() {  // cfb_common.cuh
  static const bool on = getenv("CFB_NO_PDL") == nullptr;
  return on && g_pdl_frame;
}
void pdl_set(bool on) { g_pdl_frame = on; }
static thread_local char g_err[512] = "";
int set_error(cudaError_t e, const char* what, const char* file, int line) {
  snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) in %s at %s:%d", (int)e, cudaGetErrorString(e), what, file,
           line);
  return 1000 + (int)e;
}
int set_error_msg(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}
}  // namespace cfb

using namespace cfb;

#define CK(expr) CFB_CUDA_OK(expr)
#define REQUIRE(cond, msg) \
  do {                     \
    if (!(cond)) return set_error_msg(2, "invalid argument: " msg); \
  } while (0)
#define ST(s) ((cudaStream_t)(s))

static_assert(sizeof(cfb_track_stats) == sizeof(cfb::TrackStats), "stats layout");

#pragma GCC visibility push(default)
extern "C" {

const char* cfb_last_error(void) { return g_err; }
int cfb_version(void) { return 100; }
int cfb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int cfb_upload(void* dst_dev, const void* src_host, size_t bytes, void* stream) {
  REQUIRE(dst_dev && src_host, "upload");
  CK(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, ST(stream)));
  CK(cudaStreamSynchronize(ST(stream)));
  return 0;
}
int cfb_download(void* dst_host, const void* src_dev, size_t bytes, void* stream) {
  REQUIRE(dst_host && src_dev, "download");
  CK(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, ST(stream)));
  CK(cudaStreamSynchronize(ST(stream)));
  return 0;
}

int cfb_bilateral_filter(const float* depth, size_t dp, int W, int H, float maxD, float* out, size_t op,
                         void* stream) {
  REQUIRE(depth && out && W > 0 && H > 0, "bilateral");
  CK(launch_bilateral(depth, dp, W, H, maxD, out, op, ST(stream)));
  return 0;
}
int cfb_pyr_down_gauss_f(const float* src, size_t sp, int sw, int sh, float* dst, size_t dp, void* stream) {
  REQUIRE(src && dst && sw > 1 && sh > 1, "pyr_down_gauss_f");
  CK(launch_pyr_down_gauss_f(src, sp, sw, sh, dst, dp, ST(stream)));
  return 0;
}
int cfb_pyr_down_uchar_gauss(const uint8_t* src, size_t sp, int sw, int sh, uint8_t* dst, size_t dp,
                             void* stream) {
  REQUIRE(src && dst && sw > 1 && sh > 1, "pyr_down_uchar_gauss");
  CK(launch_pyr_down_uchar(src, sp, sw, sh, dst, dp, ST(stream)));
  return 0;
}
int cfb_create_vmap(float fx, float fy, float cx, float cy, const float* depth, size_t dp, int W, int H,
                    float* vmap, size_t vp, float cutoff, void* stream) {
  REQUIRE(depth && vmap && W > 0 && H > 0, "create_vmap");
  CK(launch_create_vmap(depth, dp, W, H, Intr{fx, fy, cx, cy}, cutoff, vmap, vp, ST(stream)));
  return 0;
}
int cfb_create_nmap(const float* vmap, size_t vp, int W, int H, float* nmap, size_t np, void* stream) {
  REQUIRE(vmap && nmap && W > 0 && H > 0, "create_nmap");
  CK(launch_create_nmap(vmap, vp, W, H, nmap, np, ST(stream)));
  return 0;
}
int cfb_tranform_maps(const float* vs, size_t vsp, const float* ns, size_t nsp, int W, int H, const float R[9],
                      const float t[3], float* vd, size_t vdp, float* nd, size_t ndp, void* stream) {
  REQUIRE(vs && ns && vd && nd && R && t, "tranform_maps");
  Mat33 Rm;
  memcpy(Rm.m, R, sizeof(Rm.m));
  CK(launch_transform_maps(vs, vsp, ns, nsp, W, H, Rm, t, vd, vdp, nd, ndp, ST(stream)));
  return 0;
}
int cfb_copy_maps(const float* v4, const float* n4, int W, int H, float* vd, size_t vdp, float* nd, size_t ndp,
                  void* stream) {
  REQUIRE(v4 && n4 && vd && nd, "copy_maps");
  CK(launch_copy_maps(v4, n4, W, H, vd, vdp, nd, ndp, ST(stream)));
  return 0;
}
int cfb_resize_vmap(const float* in, size_t ip, int sw, int sh, float* out, size_t op, void* stream) {
  REQUIRE(in && out && (ip % 8) == 0, "resize_vmap (pitch must be a multiple of 8)");
  CK(launch_resize_map(in, ip, sw, sh, false, out, op, ST(stream)));
  return 0;
}
int cfb_resize_nmap(const float* in, size_t ip, int sw, int sh, float* out, size_t op, void* stream) {
  REQUIRE(in && out && (ip % 8) == 0, "resize_nmap (pitch must be a multiple of 8)");
  CK(launch_resize_map(in, ip, sw, sh, true, out, op, ST(stream)));
  return 0;
}
int cfb_vertices_to_depth(const float* v4, int W, int H, float* dst, size_t dp, float cutOff, void* stream) {
  REQUIRE(v4 && dst, "vertices_to_depth");
  CK(launch_vertices_to_depth(v4, W, H, cutOff, dst, dp, ST(stream)));
  return 0;
}
int cfb_image_bgr_to_intensity(const uint8_t* img, size_t ip, int channels, int W, int H, uint8_t* dst, size_t dp,
                               void* stream) {
  REQUIRE(img && dst && (channels == 3 || channels == 4), "image_bgr_to_intensity");
  CK(launch_rgb_to_intensity(img, ip, channels, W, H, dst, dp, ST(stream)));
  return 0;
}
int cfb_compute_derivative_images(const uint8_t* src, size_t sp, int W, int H, int16_t* dx, int16_t* dy, size_t gp,
                                  void* stream) {
  REQUIRE(src && dx && dy, "compute_derivative_images");
  CK(launch_derivative_images(src, sp, W, H, dx, dy, gp, ST(stream)));
  return 0;
}
int cfb_project_to_point_cloud(const float* depth, size_t dp, int W, int H, float fx, float fy, float cx, float cy,
                               float* cloud3, size_t cp, void* stream) {
  REQUIRE(depth && cloud3, "project_to_point_cloud");
  CK(launch_project_to_point_cloud(depth, dp, W, H, Intr{fx, fy, cx, cy}, cloud3, cp, ST(stream)));
  return 0;
}

size_t cfb_step_scratch_bytes(void) { return sizeof(StepScratch) + 256; }

// Per-call small device parameter blocks live behind the scratch (after StepScratch).
static IcpPose* scratch_pose(void* scratch) { return (IcpPose*)((char*)scratch + sizeof(StepScratch)); }
static RgbWarp* scratch_warp(void* scratch) { return (RgbWarp*)((char*)scratch + sizeof(StepScratch) + 128); }
static_assert(sizeof(IcpPose) <= 128 && sizeof(RgbWarp) <= 128, "param blocks");

int cfb_icp_step(const float Rcurr[9], const float tcurr[3], const float* vc, size_t vcp, const float* nc,
                 size_t ncp, const float Rprev_inv[9], const float tprev[3], float fx, float fy, float cx,
                 float cy, const float* vp, size_t vpp, const float* np, size_t npp, float distThres,
                 float angleThres, int W, int H, void* scratch, float* A, float* b, float* residual,
                 float* error_map, size_t error_pitch, void* stream) {
  REQUIRE(vc && nc && vp && np && scratch && A && b && residual, "icp_step");
  IcpPose hp;
  memcpy(hp.Rcurr.m, Rcurr, 36);
  memcpy(hp.tcurr, tcurr, 12);
  memcpy(hp.Rprev_inv.m, Rprev_inv, 36);
  memcpy(hp.tprev, tprev, 12);
  CK(cudaMemcpyAsync(scratch_pose(scratch), &hp, sizeof(hp), cudaMemcpyHostToDevice, ST(stream)));
  IcpArgs a;
  a.vmap_curr = {vc, vcp};
  a.nmap_curr = {nc, ncp};
  a.vmap_g_prev = {vp, vpp};
  a.nmap_g_prev = {np, npp};
  a.intr = Intr{fx, fy, cx, cy};
  a.distThres = distThres;
  a.angleThres = angleThres;
  a.cols = W;
  a.rows = H;
  a.error_map = error_map;
  a.error_pitch = error_pitch;
  StepScratch* sc = (StepScratch*)scratch;
  CK(launch_icp_step(a, scratch_pose(scratch), sc, ST(stream)));
  float host[32];
  CK(cudaMemcpyAsync(host, sc->result, sizeof(host), cudaMemcpyDeviceToHost, ST(stream)));
  CK(cudaStreamSynchronize(ST(stream)));
  gn::unpack_se3(host, A, b);
  residual[0] = host[27];
  residual[1] = host[28];
  return 0;
}

int cfb_compute_rgb_residual(float minScale, const int16_t* dIdx, const int16_t* dIdy, size_t gp,
                             const float* lastDepth, const float* nextDepth, size_t dp, const uint8_t* lastImage,
                             const uint8_t* nextImage, size_t ip, void* corresImg, void* scratch,
                             float maxDepthDelta, const float kt[3], const float krkinv[9], int W, int H,
                             int* sigmaSum, int* count, void* stream) {
  REQUIRE(dIdx && dIdy && lastDepth && nextDepth && lastImage && nextImage && corresImg && scratch, "rgb_residual");
  RgbWarp hw;
  memcpy(hw.krkinv.m, krkinv, 36);
  memcpy(hw.kt, kt, 12);
  CK(cudaMemcpyAsync(scratch_warp(scratch), &hw, sizeof(hw), cudaMemcpyHostToDevice, ST(stream)));
  RgbResidualArgs a;
  a.minScale = minScale;
  a.maxDepthDelta = maxDepthDelta;
  a.dIdx = dIdx;
  a.dIdy = dIdy;
  a.grad_pitch = gp;
  a.lastDepth = lastDepth;
  a.nextDepth = nextDepth;
  a.depth_pitch = dp;
  a.lastImage = lastImage;
  a.nextImage = nextImage;
  a.img_pitch = ip;
  a.corres = (DataTerm*)corresImg;
  a.cols = W;
  a.rows = H;
  StepScratch* sc = (StepScratch*)scratch;
  CK(launch_rgb_residual(a, scratch_warp(scratch), sc, ST(stream)));
  int host[2];
  CK(cudaMemcpyAsync(host, &sc->rgb_count, sizeof(host), cudaMemcpyDeviceToHost, ST(stream)));
  CK(cudaStreamSynchronize(ST(stream)));
  *count = host[0];
  *sigmaSum = host[1];
  return 0;
}

int cfb_rgb_step(const void* corresImg, float sigma, const float* cloud3, size_t cp, float fx, float fy,
                 const int16_t* dIdx, const int16_t* dIdy, size_t gp, float sobelScale, int W, int H,
                 void* scratch, float* A, float* b, void* stream) {
  REQUIRE(corresImg && cloud3 && dIdx && dIdy && scratch && A && b, "rgb_step");
  RgbStepArgs a;
  a.corres = (const DataTerm*)corresImg;
  a.cloud = cloud3;
  a.cloud_pitch = cp;
  a.dIdx = dIdx;
  a.dIdy = dIdy;
  a.grad_pitch = gp;
  a.fx = fx;
  a.fy = fy;
  a.sobelScale = sobelScale;
  a.cols = W;
  a.rows = H;
  StepScratch* sc = (StepScratch*)scratch;
  CK(launch_rgb_step(a, sigma, sc, ST(stream)));
  float host[32];
  CK(cudaMemcpyAsync(host, sc->result, sizeof(host), cudaMemcpyDeviceToHost, ST(stream)));
  CK(cudaStreamSynchronize(ST(stream)));
  gn::unpack_se3(host, A, b);
  return 0;
}

int cfb_so3_step(const uint8_t* lastImage, const uint8_t* nextImage, size_t ip, const float imageBasis[9],
                 const float kinv[9], const float krlr[9], int W, int H, void* scratch, float* A, float* b,
                 float* residual, void* stream) {
  REQUIRE(lastImage && nextImage && scratch && A && b && residual, "so3_step");
  So3Args a;
  a.lastImage = lastImage;
  a.nextImage = nextImage;
  a.img_pitch = ip;
  memcpy(a.imageBasis.m, imageBasis, 36);
  memcpy(a.kinv.m, kinv, 36);
  memcpy(a.krlr.m, krlr, 36);
  a.cols = W;
  a.rows = H;
  StepScratch* sc = (StepScratch*)scratch;
  CK(launch_so3_step(a, sc, ST(stream)));
  float host[32];
  CK(cudaMemcpyAsync(host, sc->result, sizeof(host), cudaMemcpyDeviceToHost, ST(stream)));
  CK(cudaStreamSynchronize(ST(stream)));
  gn::unpack_so3(host, A, b);
  residual[0] = host[9];
  residual[1] = host[10];
  return 0;
}

/* ------------------------------------------------------------------------------ RGBDOdometry */
// Every entry that enqueues work runs under the device of its handle (two instances on different GPUs in one
// process, or a caller that changed the current device, must not launch on the wrong one); the caller's current
// device is restored on return.
struct DevScope {
  int prev = -1, dev;
  explicit DevScope(int d) : dev(d) {
    if (d >= 0 && cudaGetDevice(&prev) == cudaSuccess && prev != d) cudaSetDevice(d); else prev = -1;
  }
  ~DevScope() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};
static int current_device() {
  int d = -1;
  return cudaGetDevice(&d) == cudaSuccess ? d : -1;
}

struct cfb_odom {
  RGBDOdometry* p;  // owned unless `borrowed`
  bool borrowed;
  int device;
  RGBDOdometry& impl_ref() { return *p; }
};
#define impl impl_ref()
extern "C++" inline int device_of(const cfb_odom* h) { return h ? h->device : -1; }

int cfb_odom_create(int width, int height, float cx, float cy, float fx, float fy, float distThresh,
                    float angleThresh, cfb_odom** out) {
  REQUIRE(out && width >= 32 && height >= 32 && (width % 8) == 0 && (height % 4) == 0,
          "odom_create (width must be a multiple of 8, height of 4)");
  *out = nullptr;
  if (cfb_device_count() <= 0) return set_error_msg(3, "no CUDA device: libcofusion_b200 has no CPU fallback");
  RGBDOdometry* r = new (std::nothrow) RGBDOdometry(width, height, cx, cy, fx, fy, distThresh, angleThresh);
  if (!r || !r->ok()) {
    delete r;
    return set_error_msg(4, "odom_create: device allocation failed");
  }
  *out = new cfb_odom{r, false, current_device()};
  return 0;
}
void cfb_odom_destroy(cfb_odom* o) {
  if (!o) return;
  if (!o->borrowed) delete o->p;
  delete o;
}

int cfb_odom_init_icp(cfb_odom* o, const float* const depth_pyr[3], const size_t pitch[3], float cutoff,
                      void* stream) {
  REQUIRE(o && depth_pyr && pitch, "odom_init_icp");
  DevScope dev_scope__(device_of(o));
  CK(o->impl.initICP(depth_pyr, pitch, cutoff, ST(stream)));
  return 0;
}
int cfb_odom_init_icp_model(cfb_odom* o, const float* v4, const float* n4, float cutoff, const float pose[16],
                            void* stream) {
  REQUIRE(o && v4 && n4 && pose, "odom_init_icp_model");
  DevScope dev_scope__(device_of(o));
  CK(o->impl.initICPModel(v4, n4, cutoff, pose, ST(stream)));
  return 0;
}
int cfb_odom_init_rgb_model(cfb_odom* o, const uint8_t* img, size_t pitch, int channels, void* stream) {
  REQUIRE(o && img && (channels == 3 || channels == 4), "odom_init_rgb_model");
  DevScope dev_scope__(device_of(o));
  CK(o->impl.initRGBModel(img, pitch, channels, ST(stream)));
  return 0;
}
int cfb_odom_init_rgb(cfb_odom* o, const uint8_t* img, size_t pitch, int channels, void* stream) {
  REQUIRE(o && img && (channels == 3 || channels == 4), "odom_init_rgb");
  DevScope dev_scope__(device_of(o));
  CK(o->impl.initRGB(img, pitch, channels, ST(stream)));
  return 0;
}
int cfb_odom_init_first_rgb(cfb_odom* o, const uint8_t* img, size_t pitch, int channels, void* stream) {
  REQUIRE(o && img && (channels == 3 || channels == 4), "odom_init_first_rgb");
  DevScope dev_scope__(device_of(o));
  CK(o->impl.initFirstRGB(img, pitch, channels, ST(stream)));
  return 0;
}
int cfb_odom_get_incremental_transformation(cfb_odom* o, float trans[3], float rot[9], int rgbOnly,
                                            float icpWeight, int pyramid, int fastOdom, int so3, float* err,
                                            size_t err_pitch, int force_host_loop, cfb_track_stats* stats_out,
                                            void* stream) {
  REQUIRE(o && trans && rot, "odom_get_incremental_transformation");
  DevScope dev_scope__(device_of(o));
  CK(o->impl.getIncrementalTransformation(trans, rot, rgbOnly != 0, icpWeight, pyramid != 0, fastOdom != 0,
                                          so3 != 0, err, err_pitch, force_host_loop != 0, ST(stream)));
  if (stats_out) memcpy(stats_out, &o->impl.stats(), sizeof(cfb_track_stats));
  return 0;
}
int cfb_odom_enable_kernel_timing(cfb_odom* o, int on) {
  REQUIRE(o, "odom_enable_kernel_timing");
  DevScope dev_scope__(device_of(o));
  o->impl.enableKernelTiming(on != 0);
  return 0;
}
int cfb_odom_kernel_timing(cfb_odom* o, double* sum_ms, int* launches, int reset) {
  REQUIRE(o, "odom_kernel_timing");
  DevScope dev_scope__(device_of(o));
  o->impl.kernelTiming(sum_ms, launches, reset != 0);
  return 0;
}
int cfb_odom_set_debug_trace(cfb_odom* o, void* dev_u64) {
  REQUIRE(o, "odom_set_debug_trace");
  DevScope dev_scope__(device_of(o));
  o->impl.setDebugTrace(dev_u64);
  return 0;
}
int cfb_odom_view(cfb_odom* o, int which, int level, const void** dev_ptr, size_t* pitch) {
  REQUIRE(o && dev_ptr && pitch && level >= 0 && level < 3, "odom_view");
  DevScope dev_scope__(device_of(o));
  *dev_ptr = o->impl.view(which, level, pitch);
  return *dev_ptr ? 0 : set_error_msg(2, "odom_view: unknown view");
}

#undef impl

/* ------------------------------------------------------------------------------ Context / Model */
struct cfb_ctx {
  Context* owned;
  Context& c;
  cfb_ctx(int d, int w, int h, float fx, float fy, float cx, float cy)
      : owned(new Context(d, w, h, fx, fy, cx, cy)), c(*owned) {}
  explicit cfb_ctx(Context* b) : owned(nullptr), c(*b) {}
  ~cfb_ctx() { delete owned; }
};
struct cfb_model {
  Model* owned;
  Model& m;
  cfb_odom odom_handle;
  cfb_model(Context* c, unsigned id, float conf, unsigned maxSurfels, bool fillIn)
      : owned(new Model(c, id, conf, maxSurfels, fillIn)), m(*owned), odom_handle{&owned->odom, true, c->device} {}
  explicit cfb_model(Model* b) : owned(nullptr), m(*b), odom_handle{&b->odom, true, b->ctx->device} {}
  ~cfb_model() { delete owned; }
};
extern "C++" inline int device_of(const cfb_ctx* h) { return h ? h->c.device : -1; }
extern "C++" inline int device_of(const cfb_model* h) { return h ? h->m.ctx->device : -1; }


int cfb_ctx_create(int device, int W, int H, float fx, float fy, float cx, float cy, cfb_ctx** out) {
  REQUIRE(out && W >= 32 && H >= 32 && (W % 8) == 0 && (H % 4) == 0,
          "ctx_create (W must be a multiple of 8, H of 4)");
  *out = nullptr;
  if (cfb_device_count() <= device || device < 0)
    return set_error_msg(3, "no such CUDA device: libcofusion_b200 has no CPU fallback");
  cfb_ctx* c = new (std::nothrow) cfb_ctx(device, W, H, fx, fy, cx, cy);
  if (!c || !c->c.ok()) {
    delete c;
    return set_error_msg(4, "ctx_create: device allocation failed");
  }
  *out = c;
  return 0;
}
void cfb_ctx_destroy(cfb_ctx* c) { delete c; }
void* cfb_ctx_stream(cfb_ctx* c) { return c ? (void*)c->c.stream : nullptr; }
int cfb_ctx_upload_frame(cfb_ctx* c, const uint8_t* rgb, const float* depth, const uint8_t* mask) {
  REQUIRE(c && rgb && depth, "ctx_upload_frame");
  DevScope dev_scope__(device_of(c));
  CK(c->c.uploadFrame(rgb, depth, mask));
  return 0;
}
int cfb_ctx_set_frame_device(cfb_ctx* c, const uint8_t* rgb, const float* depth, const uint8_t* mask) {
  REQUIRE(c && rgb && depth, "ctx_set_frame_device");
  DevScope dev_scope__(device_of(c));
  CK(c->c.setFrameDevice(rgb, depth, mask, true));
  return 0;
}
int cfb_ctx_preprocess(cfb_ctx* c, float depthCutoff) {
  REQUIRE(c, "ctx_preprocess");
  DevScope dev_scope__(device_of(c));
  CK(c->c.preprocess(depthCutoff));
  return 0;
}
int cfb_ctx_sync(cfb_ctx* c) {
  REQUIRE(c, "ctx_sync");
  DevScope dev_scope__(device_of(c));
  CK(c->c.sync());
  return 0;
}
int cfb_ctx_view(cfb_ctx* c, int which, const void** dev_ptr, size_t* pitch) {
  REQUIRE(c && dev_ptr && pitch, "ctx_view");
  DevScope dev_scope__(device_of(c));
  Context& x = c->c;
  switch (which) {
    case 0: *dev_ptr = x.rgb; *pitch = (size_t)x.W * 3; break;
    case 1: *dev_ptr = x.depthRaw; *pitch = (size_t)x.W * 4; break;
    case 2: *dev_ptr = x.depthFiltered; *pitch = (size_t)x.W * 4; break;
    case 3: *dev_ptr = x.depthPyr[1]; *pitch = (size_t)(x.W / 2) * 4; break;
    case 4: *dev_ptr = x.depthPyr[2]; *pitch = (size_t)(x.W / 4) * 4; break;
    case 5: *dev_ptr = x.mask; *pitch = (size_t)x.W; x.maskIsZero = false; break;  // (the caller may write through it)
    default: return set_error_msg(2, "ctx_view: unknown view");
  }
  return 0;
}
int cfb_ctx_take_launch_count(cfb_ctx* c) {
  if (!c) return 0;
  int n = c->c.launches;
  c->c.launches = 0;
  return n;
}

int cfb_model_create(cfb_ctx* c, unsigned id, float conf, unsigned max_surfels, int enable_fill_in,
                     cfb_model** out) {
  REQUIRE(c && out && max_surfels > 0 && id < 256, "model_create");
  DevScope dev_scope__(device_of(c));
  *out = nullptr;
  cfb_model* m = new (std::nothrow) cfb_model(&c->c, id, conf, max_surfels, enable_fill_in != 0);

  if (!m || !m->m.ok()) {
    delete m;
    return set_error_msg(4, "model_create: device allocation failed");
  }
  *out = m;
  return 0;
}
void cfb_model_destroy(cfb_model* m) { delete m; }
int cfb_model_get_pose(cfb_model* m, float pose[16]) {
  REQUIRE(m && pose, "model_get_pose");
  DevScope dev_scope__(device_of(m));
  CK(m->m.syncPose());
  memcpy(pose, m->m.pose, sizeof(float) * 16);
  return 0;
}
int cfb_model_override_pose(cfb_model* m, const float pose[16]) {
  REQUIRE(m && pose, "model_override_pose");
  DevScope dev_scope__(device_of(m));
  CK(m->m.syncPose());
  memcpy(m->m.pose, pose, sizeof(float) * 16);
  memcpy(m->m.lastPose, pose, sizeof(float) * 16);
  CK(m->m.uploadPose());
  return 0;
}
int cfb_model_set_pose_keep_last(cfb_model* m, const float pose[16]) {
  REQUIRE(m && pose, "model_set_pose_keep_last");
  DevScope dev_scope__(device_of(m));
  CK(m->m.syncPose());
  memcpy(m->m.pose, pose, sizeof(float) * 16);
  CK(m->m.uploadPose());
  return 0;
}
int cfb_model_set_prediction(cfb_model* m, const float* v4, const float* n4, const uint8_t* img, int channels,
                             int device_ptrs) {
  REQUIRE(m && v4 && n4 && img && (channels == 3 || channels == 4), "model_set_prediction");
  DevScope dev_scope__(device_of(m));
  CK(m->m.setPrediction(v4, n4, img, channels, device_ptrs != 0));
  return 0;
}
int cfb_model_init_first_rgb(cfb_model* m) {
  REQUIRE(m, "model_init_first_rgb");
  DevScope dev_scope__(device_of(m));
  CK(m->m.initFirstRGB());
  return 0;
}
int cfb_model_perform_tracking(cfb_model* m, const cfb_track_params* p, float pose_out[16],
                               cfb_track_stats* stats_out) {
  REQUIRE(m && p, "model_perform_tracking");
  DevScope dev_scope__(device_of(m));
  TrackParams tp;
  static_assert(sizeof(TrackParams) == sizeof(cfb_track_params), "track params layout");
  memcpy(&tp, p, sizeof(tp));
  CK(m->m.performTracking(tp));
  if (pose_out) memcpy(pose_out, m->m.pose, sizeof(float) * 16);
  if (stats_out) memcpy(stats_out, &m->m.odom.stats(), sizeof(cfb_track_stats));
  return 0;
}
int cfb_model_set_confidence_threshold(cfb_model* m, float v) {
  REQUIRE(m, "model_set_confidence_threshold");
  DevScope dev_scope__(device_of(m));
  m->m.confidenceThreshold = v;
  return 0;
}
int cfb_model_get_info(cfb_model* m, unsigned* id, float* confThresh, float* maxDepth) {
  REQUIRE(m, "model_get_info");
  DevScope dev_scope__(device_of(m));
  if (id) *id = m->m.id;
  if (confThresh) *confThresh = m->m.confidenceThreshold;
  if (maxDepth) *maxDepth = m->m.maxDepth;
  return 0;
}
int cfb_model_set_max_depth(cfb_model* m, float d) {
  REQUIRE(m, "model_set_max_depth");
  DevScope dev_scope__(device_of(m));
  m->m.maxDepth = d;
  return 0;
}
int cfb_model_initialise(cfb_model* m, int time, float maxDepthProcessed) {
  REQUIRE(m, "model_initialise");
  DevScope dev_scope__(device_of(m));
  CK(m->m.initialise(time, maxDepthProcessed));
  return 0;
}
int cfb_model_predict_indices(cfb_model* m, int time, float depthCutoff, int timeDelta) {
  REQUIRE(m, "model_predict_indices");
  DevScope dev_scope__(device_of(m));
  CK(m->m.predictIndices(time, depthCutoff, timeDelta));
  return 0;
}
int cfb_model_fuse(cfb_model* m, int time, float depthCutoff, float weightMultiplier) {
  REQUIRE(m, "model_fuse");
  DevScope dev_scope__(device_of(m));
  CK(m->m.fuse(time, depthCutoff, weightMultiplier));
  return 0;
}
int cfb_model_clean(cfb_model* m, int time, int timeDelta, float depthCutoff, float outlierCoefficient) {
  REQUIRE(m, "model_clean");
  DevScope dev_scope__(device_of(m));
  CK(m->m.clean(time, timeDelta, depthCutoff, outlierCoefficient));
  return 0;
}
int cfb_model_combined_predict(cfb_model* m, float depthCutoff, int time, int maxTime, int timeDelta) {
  REQUIRE(m, "model_combined_predict");
  DevScope dev_scope__(device_of(m));
  CK(m->m.combinedPredict(depthCutoff, time, maxTime, timeDelta));
  return 0;
}
int cfb_model_perform_fill_in(cfb_model* m, int frameToFrameRGB, int lost) {
  REQUIRE(m, "model_perform_fill_in");
  DevScope dev_scope__(device_of(m));
  CK(m->m.performFillIn(frameToFrameRGB != 0, lost != 0));
  return 0;
}
float cfb_model_compute_fusion_weight(cfb_model* m, float weightMultiplier) {
  if (!m || m->m.syncPose() != cudaSuccess) return 0.f;
  return m->m.computeFusionWeight(weightMultiplier);
}
int cfb_model_download_map(cfb_model* m, float* dst, size_t cap, unsigned* count_out) {
  REQUIRE(m, "model_download_map");
  DevScope dev_scope__(device_of(m));
  CK(m->m.downloadMap(dst, cap, count_out));
  return 0;
}
int cfb_model_upload_map(cfb_model* m, const float* src, unsigned count) {
  REQUIRE(m && (src || !count), "model_upload_map");
  DevScope dev_scope__(device_of(m));
  CK(m->m.uploadMap(src, count));
  return 0;
}
int cfb_model_last_count(cfb_model* m, unsigned* count_out) {
  REQUIRE(m && count_out, "model_last_count");
  DevScope dev_scope__(device_of(m));
  CK(m->m.lastCount(count_out));
  return 0;
}
cfb_odom* cfb_model_odometry(cfb_model* m) { return m ? &m->odom_handle : nullptr; }
int cfb_model_view(cfb_model* m, int which, const void** dev_ptr, size_t* pitch) {
  REQUIRE(m && dev_ptr && pitch, "model_view");
  DevScope dev_scope__(device_of(m));
  const size_t W = (size_t)m->m.ctx->W;
  const bool direct = m->m.usePrediction;  // the tracker reads the splat maps themselves (views 0-2: an installed prediction)
  switch (which) {
    case 0: *dev_ptr = direct ? (const void*)m->m.splat.vertexConf : m->m.predVertex; *pitch = W * 16; break;
    case 1: *dev_ptr = direct ? (const void*)m->m.splat.normalRad : m->m.predNormal; *pitch = W * 16; break;
    case 2: *dev_ptr = direct ? (const void*)m->m.splat.image : m->m.predImage; *pitch = W * 4; break;
    case 3: *dev_ptr = m->m.icpError; *pitch = W * 4; break;
    case 4: *dev_ptr = m->m.indexMaps.index; *pitch = W * 4; break;
    case 5: *dev_ptr = m->m.indexMaps.vertConf; *pitch = W * 16; break;
    case 6: *dev_ptr = m->m.indexMaps.colorTime; *pitch = W * 16; break;
    case 7: *dev_ptr = m->m.indexMaps.normRad; *pitch = W * 16; break;
    case 8: *dev_ptr = m->m.splat.image; *pitch = W * 4; break;
    case 9: *dev_ptr = m->m.splat.vertexConf; *pitch = W * 16; break;
    case 10: *dev_ptr = m->m.splat.normalRad; *pitch = W * 16; break;
    case 11: *dev_ptr = m->m.splat.time; *pitch = W * 2; break;
    case 12: *dev_ptr = m->m.fill.image; *pitch = W * 4; break;
    case 13: *dev_ptr = m->m.fill.vertex; *pitch = W * 16; break;
    case 14: *dev_ptr = m->m.fill.normal; *pitch = W * 16; break;
    case 15: *dev_ptr = m->m.unstable; *pitch = 48; break;
    default: return set_error_msg(2, "model_view: unknown view");
  }
  return 0;
}


/* ------------------------------------------------------------------------------ segmentation */
struct cfb_segmentation {
  Segmentation* owned;
  Segmentation& s;
  int lastLabels = 0, lastModels = 0;
  int device = current_device();
  cfb_segmentation(int W, int H) : owned(new Segmentation(W, H)), s(*owned) {}
  explicit cfb_segmentation(Segmentation* b) : owned(nullptr), s(*b) {}
  ~cfb_segmentation() { delete owned; }
};
extern "C++" inline int device_of(const cfb_segmentation* h) { return h ? h->device : -1; }
void cfb_seg_default_params(cfb_seg_params* p) {
  static_assert(sizeof(cfb_seg_params) == sizeof(SegParams), "seg params layout");
  static_assert(sizeof(cfb_model_data) == sizeof(SegModelData), "model data layout");
  static_assert(CFB_SEG_MAX_MODELS == SegLimits::kMaxModels, "label budget");
  if (p) seg_default_params((SegParams*)p);
}
int cfb_segmentation_create(int device, int W, int H, cfb_segmentation** out) {
  REQUIRE(out && W >= 32 && H >= 32 && (W % 16) == 0 && (H % 16) == 0, "segmentation_create (W, H multiples of 16)");
  *out = nullptr;
  if (cfb_device_count() <= device || device < 0)
    return set_error_msg(3, "no such CUDA device: libcofusion_b200 has no CPU fallback");
  CK(cudaSetDevice(device));
  cfb_segmentation* s = new (std::nothrow) cfb_segmentation(W, H);
  if (!s || !s->s.ok()) {
    delete s;
    return set_error_msg(4, "segmentation_create: device allocation failed");
  }
  *out = s;
  return 0;
}
void cfb_segmentation_destroy(cfb_segmentation* s) { delete s; }
int cfb_segmentation_slic(cfb_segmentation* s, const uint8_t* rgb, void* stream) {
  REQUIRE(s && rgb, "segmentation_slic");
  DevScope dev_scope__(device_of(s));
  CK(s->s.slic(rgb, ST(stream)));
  return 0;
}
int cfb_segmentation_perform_crf(cfb_segmentation* s, const uint8_t* rgb, const float* depth, int numModels,
                                 const unsigned char* modelIds, const float* const* icpError,
                                 const float* const* vertConf4, unsigned char nextModelID, int allowNew,
                                 const cfb_seg_params* prm, uint8_t* fullSeg, cfb_model_data* md_out, int* md_count,
                                 int* hasNewLabel, void* stream) {
  REQUIRE(s && rgb && depth && modelIds && icpError && vertConf4 && prm && fullSeg && md_out && md_count &&
              hasNewLabel && numModels >= 1 && numModels <= CFB_SEG_MAX_MODELS,
          "segmentation_perform_crf");
  DevScope dev_scope__(device_of(s));
  SegParams p;
  memcpy(&p, prm, sizeof(p));
  bool hn = false;
  CK(s->s.performSegmentationCRF(rgb, depth, numModels, modelIds, icpError, vertConf4, nextModelID, allowNew != 0, p,
                                 fullSeg, (SegModelData*)md_out, md_count, &hn, ST(stream)));
  *hasNewLabel = hn ? 1 : 0;
  s->lastModels = numModels;
  s->lastLabels = numModels + (allowNew ? 1 : 0);
  return 0;
}
int cfb_segmentation_view(cfb_segmentation* s, int which, const void** dev_ptr, size_t* bytes) {
  REQUIRE(s && dev_ptr && bytes, "segmentation_view");
  DevScope dev_scope__(device_of(s));
  const Segmentation& g = s->s;
  const size_t N = g.N;
  switch (which) {
    case 0: *dev_ptr = g.labels; *bytes = (size_t)g.W * g.H * 4; break;
    case 1: *dev_ptr = g.counts; *bytes = N * 4; break;
    case 2: *dev_ptr = g.unary; *bytes = N * s->lastLabels * 4; break;
    case 3: *dev_ptr = g.lowMap; *bytes = N; break;
    case 4: *dev_ptr = g.low; *bytes = N * (1 + 2 * s->lastModels) * 4; break;
    case 5: *dev_ptr = g.Q; *bytes = N * s->lastLabels * 4; break;
    default: return set_error_msg(2, "segmentation_view: unknown view");
  }
  return 0;
}

/* ------------------------------------------------------------------------------ CoFusion */
struct cfb_cofusion {
  CoFusion f;
  cfb_ctx ctx_handle;
  std::vector<cfb_model*> model_handles;
  std::vector<cfb_model*> retired_handles;  // of models that left the active list: kept (callers may still hold them)
  cfb_cofusion(int d, int w, int h, float fx, float fy, float cx, float cy, const CoFusionParams& p)
      : f(d, w, h, fx, fy, cx, cy, p), ctx_handle(&f.ctx) {}
  ~cfb_cofusion() {
    for (auto* h : model_handles) delete h;
    for (auto* h : retired_handles) delete h;
    delete seg_handle;
  }
  cfb_segmentation* seg_handle = nullptr;
  // handle[i] wraps model(i).  The handle of a model that left the active list stays valid memory until the
  // cfb_cofusion is destroyed (its Model object lives on in the pool); it then refers to whatever that object holds.
  void sync_handles() {
    std::vector<cfb_model*> next;
    for (size_t i = 0; i < f.numModels(); ++i) {
      cfb_model* h = nullptr;
      for (auto*& old : model_handles)
        if (old && &old->m == f.model(i)) {
          h = old;
          old = nullptr;
        }
      next.push_back(h ? h : new cfb_model(f.model(i)));
    }
    for (auto* old : model_handles)
      if (old) retired_handles.push_back(old);
    model_handles.swap(next);
  }
};

extern "C++" inline int device_of(const cfb_cofusion* h) { return h ? h->f.ctx.device : -1; }

void cfb_cofusion_default_params(cfb_cofusion_params* p) {
  if (!p) return;
  cfb_cofusion_params d = {200, 5.0f, 20.0f, 10.0f, 1, 0, 1, 0, 0, 10.0f, 0.01f, 3.0f, 3072u * 3072u, 0, 0, 20u, {}};
  cfb_seg_default_params(&d.seg);
  *p = d;
}
int cfb_cofusion_create(int device, int W, int H, float fx, float fy, float cx, float cy,
                        const cfb_cofusion_params* p, cfb_cofusion** out) {
  REQUIRE(out && p && W >= 32 && H >= 32 && (W % 8) == 0 && (H % 4) == 0 && p->maxSurfels > 0, "cofusion_create");
  REQUIRE(!p->enableMultipleModels || ((W % 16) == 0 && (H % 16) == 0),
          "cofusion_create: segmentation needs W, H multiples of 16");
  *out = nullptr;
  if (cfb_device_count() <= device || device < 0)
    return set_error_msg(3, "no such CUDA device: libcofusion_b200 has no CPU fallback");
  static_assert(sizeof(CoFusionParams) == sizeof(cfb_cofusion_params), "params layout");
  CoFusionParams cp;
  memcpy(&cp, p, sizeof(cp));
  cfb_cofusion* f = new (std::nothrow) cfb_cofusion(device, W, H, fx, fy, cx, cy, cp);
  if (!f || !f->f.ok()) {
    delete f;
    return set_error_msg(4, "cofusion_create: device allocation failed");
  }
  f->sync_handles();
  *out = f;
  return 0;
}
void cfb_cofusion_destroy(cfb_cofusion* f) { delete f; }
int cfb_cofusion_process_frame(cfb_cofusion* f, const uint8_t* rgb, const float* depth, const uint8_t* mask,
                               int device_ptrs, float weightMultiplier) {
  REQUIRE(f && ((rgb && depth) || (f->f.shard.active() && f->f.shard.rank() != 0)), "cofusion_process_frame");
  DevScope dev_scope__(device_of(f));
  CK(f->f.processFrame(rgb, depth, mask, device_ptrs != 0, weightMultiplier));
  if (f->f.params.enableMultipleModels) f->sync_handles();
  return 0;
}
int cfb_cofusion_process_frame_ex(cfb_cofusion* f, const cfb_frame* fr, const float* inPose16, float weightMultiplier,
                                  int bootstrap) {
  REQUIRE(f && fr && (!bootstrap || inPose16), "cofusion_process_frame_ex");
  DevScope dev_scope__(device_of(f));
  REQUIRE((f->f.shard.active() && f->f.shard.rank() != 0) || (fr->rgb && (fr->depth || fr->depth_u16)), "cofusion_process_frame_ex: frame");
  FrameInput in;
  in.rgb = fr->rgb;
  in.depth = fr->depth;
  in.depth16 = fr->depth ? nullptr : fr->depth_u16;
  in.depthScale = fr->depth_scale;
  in.flipColors = fr->flip_colors != 0;
  in.mask = fr->mask;
  in.device_ptrs = fr->device_ptrs != 0;
  in.timestamp = fr->timestamp;
  CK(f->f.processFrameEx(in, inPose16, bootstrap != 0, weightMultiplier));
  if (f->f.params.enableMultipleModels) f->sync_handles();
  return 0;
}
int cfb_nccl_unique_id(unsigned char id[128]) {
  REQUIRE(id, "nccl_unique_id");
  const char* err = "";
  if (FrameShard::uniqueId(id, &err) != 0) return set_error_msg(5, err);
  return 0;
}
int cfb_cofusion_shard_init(cfb_cofusion* f, int rank, int world, const unsigned char id[128]) {
  REQUIRE(f && id, "cofusion_shard_init");
  DevScope dev_scope__(device_of(f));
  const char* err = "";
  if (f->f.shardInit(rank, world, id, &err) != cudaSuccess) return set_error_msg(5, err);
  return 0;
}
int cfb_cofusion_enable_pose_logging(cfb_cofusion* f, int on) {
  REQUIRE(f, "cofusion_enable_pose_logging");
  DevScope dev_scope__(device_of(f));
  f->f.enablePoseLogging(on != 0);
  return 0;
}
int cfb_cofusion_pose_log(cfb_cofusion* f, int index, int64_t* ts, float* pose7, int capacity, int* n) {
  REQUIRE(f && n && index >= 0 && (size_t)index < f->f.numModels(), "cofusion_pose_log");
  DevScope dev_scope__(device_of(f));
  std::vector<int64_t> t;
  std::vector<float> p;
  CK(f->f.poseLog((size_t)index, &t, &p));
  *n = (int)t.size();
  const int m = *n < capacity ? *n : capacity;
  if (ts && m > 0) memcpy(ts, t.data(), sizeof(int64_t) * m);
  if (pose7 && m > 0) memcpy(pose7, p.data(), sizeof(float) * 7 * m);
  return 0;
}
int cfb_cofusion_export_poses(cfb_cofusion* f, const char* dir) {
  REQUIRE(f && dir, "cofusion_export_poses");
  DevScope dev_scope__(device_of(f));
  CK(f->f.exportPoses(dir));
  return 0;
}
int cfb_cofusion_save_ply(cfb_cofusion* f, const char* dir) {
  REQUIRE(f && dir, "cofusion_save_ply");
  DevScope dev_scope__(device_of(f));
  CK(f->f.savePly(dir));
  return 0;
}
int cfb_cofusion_last_segmentation(cfb_cofusion* f, cfb_model_data* md_out, int* md_count, int* hasNewLabel,
                                   int* spawned_id, int* deactivated) {
  REQUIRE(f && md_count, "cofusion_last_segmentation");
  DevScope dev_scope__(device_of(f));
  *md_count = (int)f->f.lastModelData.size();
  if (md_out && *md_count) memcpy(md_out, f->f.lastModelData.data(), sizeof(cfb_model_data) * *md_count);
  if (hasNewLabel) *hasNewLabel = f->f.lastHasNewLabel ? 1 : 0;
  if (spawned_id) *spawned_id = f->f.lastSpawnedId;
  if (deactivated) *deactivated = f->f.lastDeactivated;
  return 0;
}
int cfb_cofusion_num_inactive_models(cfb_cofusion* f) { return f ? (int)f->f.inactiveModels.size() : 0; }
int cfb_cofusion_set_batched_tracking(cfb_cofusion* f, int on) {
  REQUIRE(f, "cofusion_set_batched_tracking");
  DevScope dev_scope__(device_of(f));
  f->f.batchedTracking = on != 0;
  return 0;
}
int cfb_cofusion_set_debug_trace(cfb_cofusion* f, void* dev_u64) {
  REQUIRE(f && !f->f.models.empty(), "cofusion_set_debug_trace");
  DevScope dev_scope__(device_of(f));
  f->f.models[0]->odom.setDebugTrace(dev_u64);
  return 0;
}
cfb_segmentation* cfb_cofusion_segmentation(cfb_cofusion* f) {
  if (!f || !f->f.segmentation) return nullptr;
  if (!f->seg_handle) f->seg_handle = new cfb_segmentation(f->f.segmentation.get());
  return f->seg_handle;
}
int cfb_cofusion_spawn_object_model(cfb_cofusion* f, unsigned id, const float* initialPose16) {
  REQUIRE(f && id > 0 && id < 256, "cofusion_spawn_object_model");
  DevScope dev_scope__(device_of(f));
  CK(f->f.spawnObjectModel(id, initialPose16));
  f->sync_handles();
  return 0;
}
int cfb_cofusion_num_models(cfb_cofusion* f) { return f ? (int)f->f.numModels() : 0; }
int cfb_cofusion_tick(cfb_cofusion* f) { return f ? f->f.tick() : 0; }
cfb_model* cfb_cofusion_model(cfb_cofusion* f, int index) {
  if (!f || index < 0 || (size_t)index >= f->model_handles.size()) return nullptr;
  return f->model_handles[index];
}
cfb_ctx* cfb_cofusion_ctx(cfb_cofusion* f) { return f ? &f->ctx_handle : nullptr; }
int cfb_cofusion_last_stats(cfb_cofusion* f, int index, cfb_track_stats* out) {
  REQUIRE(f && out && index >= 0 && (size_t)index < f->f.numModels(), "cofusion_last_stats");
  DevScope dev_scope__(device_of(f));
  TrackStats st;
  CK(f->f.stats((size_t)index, &st));
  memcpy(out, &st, sizeof(cfb_track_stats));
  return 0;
}

}  // extern "C"
#pragma GCC visibility pop
