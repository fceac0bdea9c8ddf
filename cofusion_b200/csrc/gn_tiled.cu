// gn_tiled.cu -- the tracker optimisation (SO(3) pre-alignment + 3-level ICP/RGB Gauss-Newton,
// Core/Utils/RGBDOdometry.cpp:217-477 over Core/Cuda/reduce.cu) of ALL models of a frame
// (`for (auto model : models) model->performTracking(...)`, Core/CoFusion.cpp:213-218) as ONE persistent
// cooperative kernel, organised around 2-D image tiles that live in shared memory.
//
// Layout of the work
//   * The image of every pyramid level is cut into the same gx x gy grid of tiles, one tile per CTA
//     (one CTA per SM, 576 threads).  A CTA owns its tile for the whole launch.
//   * Frame side (current vertex / normal map, Sobel images, grey image, and for the camera model the
//     warped-depth plane and the photometric candidate gate): the tile of EVERY level is fetched once,
//     at kernel start, by TMA (cp.async.bulk.tensor + mbarrier; 3-D tensor maps over the planar
//     pyramids) -- the copies of the finer levels land while the coarser levels iterate.
//   * Model side (global-frame vertex / normal prediction, lastDepth, lastImage): projective data
//     association maps pixel (x, y) to a pixel a few columns away, coherently over a tile.  At the
//     start of a level the CTA measures the mean displacement of its tile under the current pose
//     estimate and fetches ONE window (tile + halo, shifted by that displacement) by TMA.  A Gauss-
//     Newton iteration then touches shared memory only; an association that leaves the window falls
//     back to the same values in global memory (identical results, only slower).
//   * Object models (m >= 1) cover a few percent of the image: they share the frame tiles and read their
//     own prediction from global memory (x plane first, the other five only where the object is).
//   * Levels whose tiles do not fit (1280x960 level 0) run the same code on global memory.
//
// One Gauss-Newton iteration
//     photometric correspondences -> red.add.u64 {arrived, count, sum floor(diff^2)} (barrier A, no fence:
//     the payload IS the atomic) -> ICP rows (hides A) -> RGB rows weighted with the global count ->
//     every CTA adds its 58 partial sums to 58 global accumulators with integer atomics: each f32 partial is
//     split exactly into two fixed-point words (value = hi * 2^8 + lo * 2^-39) whose low byte counts the
//     contributions, so the sum is order independent (integers commute: bit-reproducible run to run), needs
//     no fence (a word that does not show all G contributions yet is simply read again) and no per-CTA rows
//     have to be re-read by everybody -> every CTA reads the 116 words once -> FP64 Gauss-Newton step on the
//     CTA's own copy of the state, spread over the lanes of a warp (warp m solves model m).
// Within a CTA sums are folded in a fixed order (thread -> warp -> CTA); across CTAs they are exact.
// Per-pixel arithmetic: SURVEY.md Appendix A1-A5 (tracker_device.cuh holds the stand-alone form).
#include <cuda.h>  // CUtensorMap + enums only; the encoder is fetched through cudaGetDriverEntryPoint

#include <float.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "gn_math.h"
#include "image_kernels.cuh"
#include "odometry.cuh"
#include "pose_math.cuh"
#include "tracker_device.cuh"

namespace cfb {
namespace dev {

struct LevelK {  // f32 level intrinsics (CameraModel::operator())
  float fx, fy, cx, cy;
};

// RGBDOdometry.cpp:373-374
__device__ __forceinline__ float rgb_sigma_from_counts(int cnt, int sg, float* tmpErrorOut) {
  const float tmpError = (float)(sqrt((double)sg) / (double)cnt);
  if (tmpErrorOut) *tmpErrorOut = tmpError;
  return (tmpError == 0.f) ? 1.f : (float)cnt;
}

// ---- frame-side photometric preparation, once per level per frame: gradient images
// (cudafuncs.cu:658-683) + every iteration-invariant gate of RGBResidual::getProducts folded into one
// byte per pixel: j0 < W-5, i < H-1 (reduce.cu:799), 4x4 window of nextImage > 0 (:803-814),
// gradient magnitude gate (:823-825), nextDepth not NaN (:832).
__constant__ float c_sx[9] = {0.52201f, 0.00000f, -0.52201f, 0.79451f, -0.00000f, -0.79451f, 0.52201f, 0.00000f, -0.52201f};
__constant__ float c_sy[9] = {0.52201f, 0.79451f, 0.52201f, 0.00000f, 0.00000f, 0.00000f, -0.52201f, -0.79451f, -0.52201f};
__device__ __forceinline__ void rgb_prepare_pixel(const unsigned char* __restrict__ img, int W, int H,
                                                  const float* __restrict__ nextDepth, float minScale,
                                                  short* __restrict__ dx, short* __restrict__ dy,
                                                  unsigned char* __restrict__ cand, int x, int y) {
  float dxVal = 0.f, dyVal = 0.f;
  int k = 8;
  for (int j = max(y - 1, 0); j <= min(y + 1, H - 1); j++)
    for (int i = max(x - 1, 0); i <= min(x + 1, W - 1); i++) {
      float p = (float)__ldg(img + j * W + i);
      dxVal = __fadd_rn(dxVal, __fmul_rn(p, c_sx[k]));  // no FMA contraction: bit-identical to
      dyVal = __fadd_rn(dyVal, __fmul_rn(p, c_sy[k]));  // computeDerivativeImages in image_kernels.cu
      --k;
    }
  const short sx = (short)dxVal, sy = (short)dyVal;
  dx[y * W + x] = sx;
  dy[y * W + x] = sy;
  unsigned ok = (x < W - 5 && y < H - 1) ? 1u : 0u;
  for (int u = max(y - 2, 0); u < min(y + 2, H); u++)
    for (int v = max(x - 2, 0); v < min(x + 2, W); v++) ok &= (unsigned)(__ldg(img + u * W + v) > 0);
  const float mTwo = (float)((sx * sx) + (sy * sy));
  ok &= (unsigned)(mTwo >= minScale);
  ok &= (unsigned)(!isnan(__ldg(nextDepth + y * W + x)));
  cand[y * W + x] = (unsigned char)ok;
}

}  // namespace dev

namespace {
using namespace dev;

constexpr int kT = 576;               // threads per CTA, one CTA per SM
constexpr int kNW = kT / 32;          // 18 warps
constexpr int kPP = 4;                // pixels per thread of a shared-memory tile
constexpr int kMaxM = RGBDOdometry::kMaxBatch;
constexpr int kSums = 58;             // 29 ICP + 29 RGB sums of a Gauss-Newton iteration (11 for an SO(3) iteration)
constexpr int kXWords = 2 * kSums;    // two fixed-point words per sum
constexpr int kXStride = 32;          // u64 per accumulator slot: every word sits in its own 256-byte block, so the
                                      // 16,000 atomics of a round spread over the L2 slices instead of queueing on 8 lines
constexpr unsigned kNoCorr = 0xffffffffu;
constexpr int kMaxRounds = 32;        // 10 SO(3) + 19 GN reduction rounds
constexpr int kMaxHalo = 4;           // model window = tile + halo pixels on every side (less when shared memory is short)

struct MLevel {  // per model, per level
  const float *vmap_g_prev, *nmap_g_prev, *lastDepth, *nextDepth;
  const unsigned char *lastImage, *cand;
  // extents of the model in this level's image, or null (= everywhere): [minx, miny, -maxx, -maxy] of the photometric
  // candidates, then the same of the valid model vertices (written by rgb_prepare_tiled_kernel with atomicMin)
  const int* box;
  const CUtensorMap *tm_d1, *tm_cand, *tm_pv, *tm_pn, *tm_ld, *tm_li;  // camera model (m == 0) only
};
struct MParams {
  MLevel L[3];
  const unsigned char *so3_last, *so3_next;
  GNState* g;
  const float* pose_in;
  float* err;
  unsigned* corrZ;  // object models: photometric correspondences of the iteration, [kPP][grid][kT] (see phase1_obj)
  float* corrD;
  PoseDev* pd;  // optional device pose block: refreshed by the epilogue, so the frame needs no host round trip
};
struct FLevel {  // frame side + tile plan of one level
  const float *vmap_curr, *nmap_curr;
  const unsigned char* nextImage;
  const short *dIdx, *dIdy;
  const CUtensorMap *tm_v, *tm_n, *tm_dx, *tm_dy, *tm_img;
  int w, h;
  LevelK k;
  int tw, th, npx;  // tile size in pixels, tw * th
  int staged;       // 0: global memory, 1: shared-memory tiles filled by TMA, 2: filled by the threads
  // Shared-memory tiles.  A TMA box must start on a 16-byte boundary of the image row, so every element
  // type has its own box: origin = tile origin rounded down to 16 bytes, pitch wide enough for any shift.
  int pf, ps, pb;   // row pitch (elements) of the f32 / s16 / u8 frame tiles
  int wwl, wh, halo;  // logical model window (pixels): tile + halo on every side
  int wpf, wpb;     // row pitch of the f32 / u8 window planes
  unsigned o_v, o_n, o_dx, o_dy, o_img, o_d1, o_cand;  // byte offsets into dynamic shared memory
  unsigned o_pv, o_pn, o_ld, o_li;
  unsigned frame_bytes, win_bytes;  // TMA transaction sizes
};
struct TParams {
  MParams M[kMaxM];
  FLevel F[3];
  int nmodels, gx, gy;
  unsigned long long* acnt;  // [kMaxRounds][kMaxM] barrier-A words, zero before the launch
  unsigned long long* xacc;  // [kMaxRounds][nmodels][kXWords] fixed-point accumulators, zero before the launch
  size_t err_pitch;
  float distThres, angleThres, maxDepthDelta, sobelScale, icpWeight;
  int use_so3;
  int iters[3];
  unsigned o_wrow, o_blk, o_out, o_corr;
  unsigned long long* dbg;
};
static_assert(sizeof(TParams) <= 4000, "kernel parameter block");

// per level, per CTA: everything the pixel phases address, derived once per level (kept in shared memory:
// the phase functions are separate register-allocation units and read it with uniform LDS).  Tiles are
// named by byte offsets into the dynamic shared memory, never by generic pointers: the compiler then
// emits LDS with immediate offsets.
struct LvCtx {
  int W, H, x0, y0, tw, th, npx;
  int step_lx, step_ly;  // kT % tw, kT / tw: the pixel enumeration advances without a division
  float fx, fy, cx, cy;
  unsigned oV, oN, oD1, oDX, oDY, oIMG, oCAND;  // frame tiles
  int pf, ps, pb, shf, shs, shb, fplane;       // pitches, x shifts (tile origin - box origin), f32 plane stride
  unsigned oPV, oPN, oLD, oLI;                  // model window of the camera model
  int wpf, wpb, wshf, wshb, wplane;
  int wwl, wh, wx0, wy0;                        // logical window: columns [wx0, wx0 + wwl), rows [wy0, wy0 + wh)
  unsigned oCorrZ, oCorrD;                      // [kPP][kT] packed correspondence / depth of the matched point
};

struct TFixed {  // fixed head of the dynamic shared memory
  TParams prm;
  LvCtx lv;
  GNState S[kMaxM];  // every CTA keeps (and identically updates) its own copy of every model's state
  double K[3][9], Kinv[3][9];
  double solveA[kMaxM][42];
  unsigned long long bar_frame[3], bar_win;
  int cntw[kMaxM][kNW], sigw[kMaxM][kNW];
  int tot[kMaxM][2];
  int box[kMaxM][8];  // this level: candidates [minx, miny, maxx, maxy], valid model vertices [minx, miny, maxx, maxy]
  float tmpErr[kMaxM];
  int winacc[3];
  int win_x0, win_y0;
  int sched[20];
  int nsched;
};

#define TSMEM()                                                   \
  extern __shared__ __align__(128) unsigned char dyn_smem_raw[]; \
  TFixed& sm = *reinterpret_cast<TFixed*>(dyn_smem_raw);          \
  const TParams& p = sm.prm
#define SM_F32(off) (reinterpret_cast<float*>(dyn_smem_raw + (off)))
#define SM_S16(off) (reinterpret_cast<short*>(dyn_smem_raw + (off)))
#define SM_U8(off) (dyn_smem_raw + (off))
#define SM_U32(off) (reinterpret_cast<unsigned*>(dyn_smem_raw + (off)))

__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// The trace is compiled into its own instantiations of the kernel (DBGT): in the production ones it costs nothing.
// per-CTA stamps of iteration 12 (a level-0 iteration): slots 256 + 8 * cta + e, e = 0..4
#define DBG_CTA(q, e)                                                                                      \
  do {                                                                                                     \
    if (DBGT && p.dbg && (q) == 12 && threadIdx.x == 0) p.dbg[256 + 8 * blockIdx.x + (e)] = gtime();       \
  } while (0)
#define DBG_MARK(slot)                                                       \
  do {                                                                       \
    if (DBGT && p.dbg && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[(slot)] = gtime(); \
  } while (0)

// ------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ unsigned smem_u32(const void* q) { return (unsigned)__cvta_generic_to_shared(q); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  unsigned ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
// A tensor map that lives in global memory (written by the host with cudaMemcpy) is read through the
// tensormap proxy: the issuing thread acquires it first (CUDA programming guide, "tensor map in global memory").
__device__ __forceinline__ void tmap_acquire(const CUtensorMap* tm) {
  asm volatile("fence.proxy.tensormap::generic.acquire.sys [%0], 128;" ::"l"(tm) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tm, int c0, int c1, unsigned long long* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(tm), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2,
                                            unsigned long long* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(dst)),
      "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ unsigned long long ld_u64_relaxed(const unsigned long long* q) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(q) : "memory");
  return v;
}
__device__ __forceinline__ void red_add_u64(unsigned long long* q, unsigned long long v) {
  asm volatile("red.relaxed.gpu.global.add.u64 [%0], %1;" ::"l"(q), "l"(v) : "memory");
}
__device__ __forceinline__ int floor_to(int x, int a) {  // largest multiple of a (power of two) <= x
  return x & ~(a - 1);
}

// correspondence of one pixel packed into 32 bits: u0 (11) | v0 (11) | diff + 256 (10).  diff is the
// difference of two 8-bit intensities, an integer in [-255, 255]: lossless for images below 2048 x 2048.
__device__ __forceinline__ unsigned pack_corr(int u0, int v0, float diff) {
  return (unsigned)u0 | ((unsigned)v0 << 11) | ((unsigned)((int)diff + 256) << 22);
}

__device__ __forceinline__ void make_lvctx(int lvl) {  // one thread
  TSMEM();
  LvCtx& c = sm.lv;
  const FLevel& F = p.F[lvl];
  const int bx = blockIdx.x % p.gx, by = blockIdx.x / p.gx;
  c.W = F.w;
  c.H = F.h;
  c.tw = F.tw;
  c.th = F.th;
  c.npx = F.npx;
  c.x0 = bx * F.tw;
  c.y0 = by * F.th;
  c.step_lx = kT % F.tw;
  c.step_ly = kT / F.tw;
  c.fx = F.k.fx;
  c.fy = F.k.fy;
  c.cx = F.k.cx;
  c.cy = F.k.cy;
  c.oV = F.o_v;
  c.oN = F.o_n;
  c.oD1 = F.o_d1;
  c.oDX = F.o_dx;
  c.oDY = F.o_dy;
  c.oIMG = F.o_img;
  c.oCAND = F.o_cand;
  c.pf = F.pf;
  c.ps = F.ps;
  c.pb = F.pb;
  c.shf = c.x0 - floor_to(c.x0, 4);
  c.shs = c.x0 - floor_to(c.x0, 8);
  c.shb = c.x0 - floor_to(c.x0, 16);
  c.fplane = F.pf * F.th;
  c.oPV = F.o_pv;
  c.oPN = F.o_pn;
  c.oLD = F.o_ld;
  c.oLI = F.o_li;
  c.wpf = F.wpf;
  c.wpb = F.wpb;
  c.wwl = F.wwl;
  c.wh = F.wh;
  c.wx0 = sm.win_x0;
  c.wy0 = sm.win_y0;
  c.wshf = c.wx0 - floor_to(c.wx0, 4);
  c.wshb = c.wx0 - floor_to(c.wx0, 16);
  c.wplane = F.wpf * F.wh;
  c.oCorrZ = p.o_corr;
  c.oCorrD = p.o_corr + kPP * kT * 4;
}

// the pixel enumeration of a thread: i = tid, tid + kT, ... < npx over the tw x th tile, row-major
struct PixIt {
  int i, lx, ly;
};
__device__ __forceinline__ PixIt pix_begin(const LvCtx& c) {
  PixIt it;
  it.i = threadIdx.x;
  it.ly = (int)threadIdx.x / c.tw;
  it.lx = (int)threadIdx.x - it.ly * c.tw;
  return it;
}
__device__ __forceinline__ void pix_next(const LvCtx& c, PixIt& it) {
  it.i += kT;
  it.lx += c.step_lx;
  it.ly += c.step_ly;
  if (it.lx >= c.tw) {
    it.lx -= c.tw;
    it.ly += 1;
  }
}

// ------------------------------------------------------------------------------------------ arithmetic
// Every operation that feeds a decision or a sum is written with an explicit rounding (no implicit FMA
// contraction): the three instantiations of each phase (shared-memory tiles / global memory, camera model /
// object model) then perform the same operation sequence, so a model tracked alone and the same model
// tracked inside a batch produce the same bits.
__device__ __forceinline__ float3 xsub(float3 a, float3 b) { return make_float3(__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y), __fsub_rn(a.z, b.z)); }
__device__ __forceinline__ float3 xadd(float3 a, float3 b) { return make_float3(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z)); }
__device__ __forceinline__ float xdot(float3 a, float3 b) { return __fmaf_rn(a.z, b.z, __fmaf_rn(a.y, b.y, __fmul_rn(a.x, b.x))); }
__device__ __forceinline__ float xnorm(float3 a) { return __fsqrt_rn(xdot(a, a)); }
__device__ __forceinline__ float3 xcross(float3 a, float3 b) {
  return make_float3(__fmaf_rn(a.y, b.z, -__fmul_rn(a.z, b.y)), __fmaf_rn(a.z, b.x, -__fmul_rn(a.x, b.z)),
                     __fmaf_rn(a.x, b.y, -__fmul_rn(a.y, b.x)));
}
__device__ __forceinline__ float3 xmul(const Mat33& m, float3 a) {
  return make_float3(__fmaf_rn(m.m[2], a.z, __fmaf_rn(m.m[1], a.y, __fmul_rn(m.m[0], a.x))),
                     __fmaf_rn(m.m[5], a.z, __fmaf_rn(m.m[4], a.y, __fmul_rn(m.m[3], a.x))),
                     __fmaf_rn(m.m[8], a.z, __fmaf_rn(m.m[7], a.y, __fmul_rn(m.m[6], a.x))));
}
// 27 upper-triangular products + row6^2 + inlier (JtJJtrSE3 order, types.cuh:101-112)
__device__ __forceinline__ void xaccumulate_se3(float (&acc)[32], const float (&row)[7]) {
  int k = 0;
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = i; j < 7; ++j, ++k) acc[k] = __fmaf_rn(row[i], row[j], acc[k]);
  acc[27] = __fmaf_rn(row[6], row[6], acc[27]);
  acc[28] = __fadd_rn(acc[28], 1.f);
}

// ------------------------------------------------------------------------------------------ phase 1
// RGBResidual::getProducts for a candidate pixel (reduce.cu:827-853).  FS: frame tiles in shared
// memory, MS: this model's window in shared memory.  Returns validity, fills u0 / v0 / diff / d0.
template <bool FS, bool MS>
__device__ __forceinline__ bool residual_pixel(const LvCtx& c, const MLevel& L, const RgbWarp& Wp, float maxDepthDelta,
                                               int lx, int ly, int x, int y, const unsigned char* nextImage, int& u0,
                                               int& v0, float& diff, float& d0, const int* box) {
  extern __shared__ __align__(128) unsigned char dyn_smem_raw[];
  bool cand;
  float d1;
  // an object model fills a few percent of the image: outside the extent of its candidates the gate is 0, known
  // without the (long-latency, per-pixel serial) global load
  if (!MS && (x < box[0] || y < box[1] || x > box[2] || y > box[3])) return false;
  if (MS) {
    cand = SM_U8(c.oCAND)[ly * c.pb + lx + c.shb] != 0;
    d1 = SM_F32(c.oD1)[ly * c.pf + lx + c.shf];
  } else {
    cand = __ldg(L.cand + y * c.W + x) != 0;
    d1 = cand ? __ldg(L.nextDepth + y * c.W + x) : 0.f;
  }
  if (!cand) return false;
  const float* kk = Wp.krkinv.m;
  const float fx_ = (float)x, fy_ = (float)y;
  const float td1 = __fmaf_rn(d1, __fadd_rn(__fmaf_rn(kk[7], fy_, __fmul_rn(kk[6], fx_)), kk[8]), Wp.kt[2]);
  u0 = __float2int_rn(__fdiv_rn(__fmaf_rn(d1, __fadd_rn(__fmaf_rn(kk[1], fy_, __fmul_rn(kk[0], fx_)), kk[2]), Wp.kt[0]), td1));
  v0 = __float2int_rn(__fdiv_rn(__fmaf_rn(d1, __fadd_rn(__fmaf_rn(kk[4], fy_, __fmul_rn(kk[3], fx_)), kk[5]), Wp.kt[1]), td1));
  if (!(u0 >= 0 && v0 >= 0 && u0 < c.W && v0 < c.H)) return false;
  unsigned char li;
  const int wu = u0 - c.wx0, wv = v0 - c.wy0;
  if (MS && (unsigned)wu < (unsigned)c.wwl && (unsigned)wv < (unsigned)c.wh) {
    d0 = SM_F32(c.oLD)[wv * c.wpf + wu + c.wshf];
    li = SM_U8(c.oLI)[wv * c.wpb + wu + c.wshb];
  } else {
    d0 = __ldg(L.lastDepth + v0 * c.W + u0);
    li = __ldg(L.lastImage + v0 * c.W + u0);
  }
  if (!(d0 > 0 && fabsf(__fsub_rn(td1, d0)) <= maxDepthDelta && li != 0)) return false;
  const unsigned char ni = FS ? SM_U8(c.oIMG)[ly * c.pb + lx + c.shb] : __ldg(nextImage + y * c.W + x);
  diff = __fsub_rn((float)ni, (float)li);
  return true;
}

template <bool FS, bool MS>
__device__ __noinline__ void phase1(int lvl, int m) {
  TSMEM();
  const LvCtx& c = sm.lv;
  const MLevel& L = p.M[m].L[lvl];
  const RgbWarp& Wp = sm.S[m].warp;
  const unsigned char* nextImage = p.F[lvl].nextImage;
  int cnt = 0, sig = 0;
  int k = 0;
  // a tile the model's candidates do not reach has nothing to enumerate
  const int* bc = sm.box[m];
  const bool none = !MS && (c.x0 > bc[2] || c.x0 + c.tw <= bc[0] || c.y0 > bc[3] || c.y0 + c.th <= bc[1]);
  for (PixIt it = pix_begin(c); !none && it.i < c.npx; pix_next(c, it), ++k) {
    const int x = c.x0 + it.lx, y = c.y0 + it.ly;
    int u0, v0;
    float diff, d0;
    unsigned zero = kNoCorr;
    if (x < c.W && y < c.H &&
        residual_pixel<FS, MS>(c, L, Wp, p.maxDepthDelta, it.lx, it.ly, x, y, nextImage, u0, v0, diff, d0, sm.box[m])) {
      cnt += 1;
      sig += (int)__fmul_rn(diff, diff);  // float -> int truncation, reduce.cu:851
      if (MS) {
        zero = pack_corr(u0, v0, diff);
        SM_F32(c.oCorrD)[k * kT + threadIdx.x] = d0;
      }
    }
    if (MS) SM_U32(c.oCorrZ)[k * kT + threadIdx.x] = zero;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    sig += __shfl_xor_sync(0xffffffffu, sig, o);
  }
  if ((threadIdx.x & 31) == 0) {
    sm.cntw[m][threadIdx.x >> 5] = cnt;
    sm.sigw[m][threadIdx.x >> 5] = sig;
  }
}

// ------------------------------------------------------------------------------------------ phase 2
// Per-CTA reduction of a phase: every warp leaves its 32 sums (warp transpose) in one of two alternating
// row buffers; after the block barrier that follows the phase, fold_warp_rows() adds the 18 rows in warp order
// into blk[m][set * 29 + j].  The buffers alternate from phase to phase, so the fold of one phase overlaps the
// next phase and one barrier per phase suffices (the buffer written two phases ago has been folded by then).
__device__ __forceinline__ void store_warp_row(int buf, bool any, float (&acc)[32]) {
  TSMEM();
  float* wrow = SM_F32(p.o_wrow) + ((size_t)buf * kNW + (threadIdx.x >> 5)) * 32;
  // a warp without any contribution adds exact zeros: skip its 31-shuffle transpose
  wrow[threadIdx.x & 31] = __any_sync(0xffffffffu, any) ? warp_transpose_reduce32(acc) : 0.f;
}
__device__ __forceinline__ void fold_warp_rows(int buf, int m, int set, int nsums) {
  TSMEM();
  if ((int)threadIdx.x < nsums) {
    const float* r = SM_F32(p.o_wrow) + (size_t)buf * kNW * 32 + threadIdx.x;
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kNW; ++w) s += r[w * 32];  // warp order
    SM_F32(p.o_blk)[m * 64 + set * 29 + threadIdx.x] = s;
  }
}

__device__ __forceinline__ void icp_found_row(const IcpPose& P, float3 tprev, float3 vcurr_cp, float3 vp, float3 np,
                                              float (&acc)[32]) {
  const float3 d_cp = xmul(P.Rprev_inv, xsub(vp, tprev));
  const float3 n_cp = xmul(P.Rprev_inv, np);
  const float3 cr = xcross(vcurr_cp, n_cp);
  const float row[7] = {n_cp.x, n_cp.y, n_cp.z, cr.x, cr.y, cr.z, xdot(n_cp, xsub(vcurr_cp, d_cp))};
  xaccumulate_se3(acc, row);
}

template <bool FS, bool MS>
__device__ __noinline__ void phase2(int lvl, int m, float* error_map, int buf) {
  TSMEM();
  const LvCtx& c = sm.lv;
  const MLevel& L = p.M[m].L[lvl];
  const FLevel& F = p.F[lvl];
  const IcpPose& P = sm.S[m].pose;
  float acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.f;
  const float3 tcurr = make_float3(P.tcurr[0], P.tcurr[1], P.tcurr[2]);
  const float3 tprev = make_float3(P.tprev[0], P.tprev[1], P.tprev[2]);
  const int HW = c.W * c.H;
  bool any = false;
  for (PixIt it = pix_begin(c); it.i < c.npx; pix_next(c, it)) {
    const int x = c.x0 + it.lx, y = c.y0 + it.ly;
    if (x >= c.W || y >= c.H) continue;
    const int fi = it.ly * c.pf + it.lx + c.shf;  // index into the f32 frame tiles
    const int gi = y * c.W + x;
    float3 vcurr;
    vcurr.x = FS ? SM_F32(c.oV)[fi] : __ldg(F.vmap_curr + gi);
    float* const err = error_map ? row_ptr(error_map, p.err_pitch, y) + x : nullptr;
    // an invalid vertex has NaN in x: every coordinate of vcurr_g is NaN, dist is NaN -> no
    // correspondence, error 0 (same outcome as running the arithmetic, without the gathers)
    if (isnan(vcurr.x)) {
      if (err) *err = 0.0f;
      continue;
    }
    vcurr.y = FS ? SM_F32(c.oV)[c.fplane + fi] : __ldg(F.vmap_curr + HW + gi);
    vcurr.z = FS ? SM_F32(c.oV)[2 * c.fplane + fi] : __ldg(F.vmap_curr + 2 * HW + gi);
    const float3 vcurr_g = xadd(xmul(P.Rcurr, vcurr), tcurr);
    const float3 vcurr_cp = xmul(P.Rprev_inv, xsub(vcurr_g, tprev));
    const int ux = __float2int_rn(__fadd_rn(__fdiv_rn(__fmul_rn(vcurr_cp.x, c.fx), vcurr_cp.z), c.cx));
    const int uy = __float2int_rn(__fadd_rn(__fdiv_rn(__fmul_rn(vcurr_cp.y, c.fy), vcurr_cp.z), c.cy));
    if (ux < 0 || uy < 0 || ux >= c.W || uy >= c.H || vcurr_cp.z < 0) {
      if (err) *err = 0.0f;
      continue;
    }
    float3 vp, np;
    const int wu = ux - c.wx0, wv = uy - c.wy0;
    if (MS && (unsigned)wu < (unsigned)c.wwl && (unsigned)wv < (unsigned)c.wh) {
      const int j = wv * c.wpf + wu + c.wshf;
      vp = make_float3(SM_F32(c.oPV)[j], SM_F32(c.oPV)[c.wplane + j], SM_F32(c.oPV)[2 * c.wplane + j]);
      np = make_float3(SM_F32(c.oPN)[j], SM_F32(c.oPN)[c.wplane + j], SM_F32(c.oPN)[2 * c.wplane + j]);
    } else {
      // An object model predicts a few percent of the image; everywhere else its vertex map is NaN.
      // A NaN in the x plane makes dist NaN whatever the other five planes hold -- and outside the extent of
      // the valid vertices it is NaN without looking.
      const int* bv = sm.box[m] + 4;
      if (ux < bv[0] || uy < bv[1] || ux > bv[2] || uy > bv[3]) {
        if (err) *err = 0.0f;
        continue;
      }
      const int j = uy * c.W + ux;
      vp.x = __ldg(L.vmap_g_prev + j);
      if (isnan(vp.x)) {
        if (err) *err = 0.0f;
        continue;
      }
      vp.y = __ldg(L.vmap_g_prev + HW + j);
      vp.z = __ldg(L.vmap_g_prev + 2 * HW + j);
      np = make_float3(__ldg(L.nmap_g_prev + j), __ldg(L.nmap_g_prev + HW + j), __ldg(L.nmap_g_prev + 2 * HW + j));
    }
    float3 ncurr;
    if (FS)
      ncurr = make_float3(SM_F32(c.oN)[fi], SM_F32(c.oN)[c.fplane + fi], SM_F32(c.oN)[2 * c.fplane + fi]);
    else
      ncurr = make_float3(__ldg(F.nmap_curr + gi), __ldg(F.nmap_curr + HW + gi), __ldg(F.nmap_curr + 2 * HW + gi));
    const float3 ncurr_g = xmul(P.Rcurr, ncurr);
    const float dist = xnorm(xsub(vp, vcurr_g));
    const float sine = xnorm(xcross(ncurr_g, np));
    if (err) *err = isfinite(dist) ? dist : 0.0f;
    if (sine < p.angleThres && dist <= p.distThres && !isnan(ncurr.x) && !isnan(np.x)) {
      any = true;
      icp_found_row(P, tprev, vcurr_cp, vp, np, acc);
    }
  }
  store_warp_row(buf, any, acc);
}

// ------------------------------------------------------------------------------------------ phase 3
__device__ __forceinline__ void rgb_row(const LvCtx& c, float sigma, float sobelScale, int zx, int zy, float z, float diff,
                                        short sdx, short sdy, float (&acc)[32]) {
  float w = __fadd_rn(sigma, fabsf(diff));
  w = w > 1.19209290E-07F ? __fdiv_rn(1.0f, w) : 1.0f;
  if (sigma == -1.f) w = 1.f;
  const float invFx = __fdiv_rn(1.0f, c.fx), invFy = __fdiv_rn(1.0f, c.fy);
  const float3 Pt = make_float3(__fmul_rn(__fmul_rn(__fsub_rn((float)zx, c.cx), z), invFx),
                                __fmul_rn(__fmul_rn(__fsub_rn((float)zy, c.cy), z), invFy), z);
  const float invz = (float)(1.0 / (double)Pt.z);
  const float dI_dx_val = __fmul_rn(__fmul_rn(w, sobelScale), (float)sdx);
  const float dI_dy_val = __fmul_rn(__fmul_rn(w, sobelScale), (float)sdy);
  const float v0 = __fmul_rn(__fmul_rn(dI_dx_val, c.fx), invz);
  const float v1 = __fmul_rn(__fmul_rn(dI_dy_val, c.fy), invz);
  const float v2 = __fmul_rn(-__fmaf_rn(v1, Pt.y, __fmul_rn(v0, Pt.x)), invz);
  const float row[7] = {v0,
                        v1,
                        v2,
                        __fmaf_rn(Pt.y, v2, -__fmul_rn(Pt.z, v1)),
                        __fmaf_rn(Pt.z, v0, -__fmul_rn(Pt.x, v2)),
                        __fmaf_rn(Pt.x, v1, -__fmul_rn(Pt.y, v0)),
                        -__fmul_rn(w, diff)};
  xaccumulate_se3(acc, row);
}

template <bool FS, bool MS>
__device__ __noinline__ void phase3(int lvl, int m, float sigma, int buf) {
  TSMEM();
  const LvCtx& c = sm.lv;
  const FLevel& F = p.F[lvl];
  float acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.f;
  bool any = false;
  int k = 0;
  const int* bc = sm.box[m];
  const bool none = !MS && (c.x0 > bc[2] || c.x0 + c.tw <= bc[0] || c.y0 > bc[3] || c.y0 + c.th <= bc[1]);
  for (PixIt it = pix_begin(c); !none && it.i < c.npx; pix_next(c, it), ++k) {
    if (MS) {  // the correspondences of phase 1 never left the SM
      const unsigned zero = SM_U32(c.oCorrZ)[k * kT + threadIdx.x];
      if (zero == kNoCorr) continue;
      any = true;
      const int si = it.ly * c.ps + it.lx + c.shs;
      rgb_row(c, sigma, p.sobelScale, (int)(zero & 0x7ffu), (int)((zero >> 11) & 0x7ffu), SM_F32(c.oCorrD)[k * kT + threadIdx.x],
              (float)((int)(zero >> 22) - 256), SM_S16(c.oDX)[si], SM_S16(c.oDY)[si], acc);
    } else {  // recomputed: the same decisions and values as phase 1
      const int x = c.x0 + it.lx, y = c.y0 + it.ly;
      int u0, v0;
      float diff, d0;
      if (x >= c.W || y >= c.H) continue;
      if (!residual_pixel<FS, false>(c, p.M[m].L[lvl], sm.S[m].warp, p.maxDepthDelta, it.lx, it.ly, x, y, F.nextImage, u0, v0, diff, d0,
                                     sm.box[m]))
        continue;
      any = true;
      const int si = it.ly * c.ps + it.lx + c.shs;
      const short sdx = FS ? SM_S16(c.oDX)[si] : __ldg(F.dIdx + y * c.W + x);
      const short sdy = FS ? SM_S16(c.oDY)[si] : __ldg(F.dIdy + y * c.W + x);
      rgb_row(c, sigma, p.sobelScale, u0, v0, d0, diff, sdx, sdy, acc);
    }
  }
  store_warp_row(buf, any, acc);
}

// ------------------------------------------------------------------------- object models on staged levels
// The shared memory of a CTA holds the frame tiles and the CAMERA model's window; the maps of an object model
// (m >= 1) stay in global memory.  Written pixel by pixel, a thread's gathers form a chain of dependent L2 round
// trips (gate -> depth -> matched depth / intensity; vertex x -> five more planes), times its four pixels: the CTAs
// whose tiles hold the object took twice as long as the rest, and the whole grid waits for them at every sum.
// These variants run every ROUND of loads for all of the thread's pixels before the first use (2 + 1 + 2 round
// trips per iteration instead of 32) and hand the correspondences of phase 1 to phase 3 through a coalesced
// global array.  Per pixel the operations, their order and roundings are those of residual_pixel / phase2 /
// phase3: the sums are bit-identical.
__device__ __noinline__ void phase1_obj(int lvl, int m) {
  TSMEM();
  const LvCtx& c = sm.lv;
  const MLevel& L = p.M[m].L[lvl];
  const RgbWarp& Wp = sm.S[m].warp;
  int cnt = 0, sig = 0;
  const int* bc = sm.box[m];
  const bool none = c.x0 > bc[2] || c.x0 + c.tw <= bc[0] || c.y0 > bc[3] || c.y0 + c.th <= bc[1];
  if (!none) {
    const size_t kstride = (size_t)gridDim.x * kT;
    unsigned* cz = p.M[m].corrZ + (size_t)blockIdx.x * kT + threadIdx.x;
    float* cd = p.M[m].corrD + (size_t)blockIdx.x * kT + threadIdx.x;
    int xs[kPP], ys[kPP];
    unsigned char cand[kPP];
    float d1[kPP];
    PixIt it = pix_begin(c);
#pragma unroll
    for (int k = 0; k < kPP; ++k) {  // round 1: gate and depth of every pixel
      const int x = c.x0 + it.lx, y = c.y0 + it.ly;
      const bool live = it.i < c.npx && x < c.W && y < c.H && !(x < bc[0] || y < bc[1] || x > bc[2] || y > bc[3]);
      xs[k] = x;
      ys[k] = live ? y : -1;
      cand[k] = live ? __ldg(L.cand + y * c.W + x) : (unsigned char)0;
      d1[k] = live ? __ldg(L.nextDepth + y * c.W + x) : 0.f;
      pix_next(c, it);
    }
    int j[kPP], u0[kPP], v0[kPP];
    float td1[kPP];
    const float* kk = Wp.krkinv.m;
#pragma unroll
    for (int k = 0; k < kPP; ++k) {
      j[k] = -1;
      u0[k] = v0[k] = 0;
      td1[k] = 0.f;
      if (cand[k] != 0) {
        const float fx_ = (float)xs[k], fy_ = (float)ys[k];
        td1[k] = __fmaf_rn(d1[k], __fadd_rn(__fmaf_rn(kk[7], fy_, __fmul_rn(kk[6], fx_)), kk[8]), Wp.kt[2]);
        u0[k] = __float2int_rn(__fdiv_rn(__fmaf_rn(d1[k], __fadd_rn(__fmaf_rn(kk[1], fy_, __fmul_rn(kk[0], fx_)), kk[2]), Wp.kt[0]), td1[k]));
        v0[k] = __float2int_rn(__fdiv_rn(__fmaf_rn(d1[k], __fadd_rn(__fmaf_rn(kk[4], fy_, __fmul_rn(kk[3], fx_)), kk[5]), Wp.kt[1]), td1[k]));
        if (u0[k] >= 0 && v0[k] >= 0 && u0[k] < c.W && v0[k] < c.H) j[k] = v0[k] * c.W + u0[k];
      }
    }
    float d0[kPP];
    unsigned char li[kPP];
#pragma unroll
    for (int k = 0; k < kPP; ++k) {  // round 2: the matched points
      d0[k] = j[k] >= 0 ? __ldg(L.lastDepth + j[k]) : 0.f;
      li[k] = j[k] >= 0 ? __ldg(L.lastImage + j[k]) : (unsigned char)0;
    }
#pragma unroll
    for (int k = 0; k < kPP; ++k) {
      unsigned zero = kNoCorr;
      if (j[k] >= 0 && d0[k] > 0 && fabsf(__fsub_rn(td1[k], d0[k])) <= p.maxDepthDelta && li[k] != 0) {
        const unsigned char ni = SM_U8(c.oIMG)[(ys[k] - c.y0) * c.pb + (xs[k] - c.x0) + c.shb];
        const float diff = __fsub_rn((float)ni, (float)li[k]);
        cnt += 1;
        sig += (int)__fmul_rn(diff, diff);  // float -> int truncation, reduce.cu:851
        zero = pack_corr(u0[k], v0[k], diff);
        cd[k * kstride] = d0[k];
      }
      if (k * kT + (int)threadIdx.x < c.npx) cz[k * kstride] = zero;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    sig += __shfl_xor_sync(0xffffffffu, sig, o);
  }
  if ((threadIdx.x & 31) == 0) {
    sm.cntw[m][threadIdx.x >> 5] = cnt;
    sm.sigw[m][threadIdx.x >> 5] = sig;
  }
}

__device__ __noinline__ void phase2_obj(int lvl, int m, float* error_map, int buf) {
  TSMEM();
  const LvCtx& c = sm.lv;
  const MLevel& L = p.M[m].L[lvl];
  const IcpPose& P = sm.S[m].pose;
  float acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.f;
  const float3 tcurr = make_float3(P.tcurr[0], P.tcurr[1], P.tcurr[2]);
  const float3 tprev = make_float3(P.tprev[0], P.tprev[1], P.tprev[2]);
  const int HW = c.W * c.H;
  const int* bv = sm.box[m] + 4;
  int j[kPP];
  {
    PixIt it = pix_begin(c);
#pragma unroll
    for (int k = 0; k < kPP; ++k) {  // where each pixel lands in the model's maps (-1: nowhere)
      j[k] = -1;
      const int x = c.x0 + it.lx, y = c.y0 + it.ly;
      if (it.i < c.npx && x < c.W && y < c.H) {
        const int fi = it.ly * c.pf + it.lx + c.shf;
        float3 vcurr;
        vcurr.x = SM_F32(c.oV)[fi];
        if (!isnan(vcurr.x)) {
          vcurr.y = SM_F32(c.oV)[c.fplane + fi];
          vcurr.z = SM_F32(c.oV)[2 * c.fplane + fi];
          const float3 vcurr_g = xadd(xmul(P.Rcurr, vcurr), tcurr);
          const float3 vcurr_cp = xmul(P.Rprev_inv, xsub(vcurr_g, tprev));
          const int ux = __float2int_rn(__fadd_rn(__fdiv_rn(__fmul_rn(vcurr_cp.x, c.fx), vcurr_cp.z), c.cx));
          const int uy = __float2int_rn(__fadd_rn(__fdiv_rn(__fmul_rn(vcurr_cp.y, c.fy), vcurr_cp.z), c.cy));
          if (!(ux < 0 || uy < 0 || ux >= c.W || uy >= c.H || vcurr_cp.z < 0) &&
              !(ux < bv[0] || uy < bv[1] || ux > bv[2] || uy > bv[3]))
            j[k] = uy * c.W + ux;
        }
      }
      pix_next(c, it);
    }
  }
  float vx[kPP];
#pragma unroll
  for (int k = 0; k < kPP; ++k) vx[k] = j[k] >= 0 ? __ldg(L.vmap_g_prev + j[k]) : qnan();  // round 1
  float q[kPP][5];
#pragma unroll
  for (int k = 0; k < kPP; ++k) {  // round 2: the other five planes, only where the object is
    const bool have = !isnan(vx[k]);
    q[k][0] = have ? __ldg(L.vmap_g_prev + HW + j[k]) : 0.f;
    q[k][1] = have ? __ldg(L.vmap_g_prev + 2 * HW + j[k]) : 0.f;
    q[k][2] = have ? __ldg(L.nmap_g_prev + j[k]) : 0.f;
    q[k][3] = have ? __ldg(L.nmap_g_prev + HW + j[k]) : 0.f;
    q[k][4] = have ? __ldg(L.nmap_g_prev + 2 * HW + j[k]) : 0.f;
  }
  bool any = false;
  PixIt it = pix_begin(c);
#pragma unroll
  for (int k = 0; k < kPP; ++k) {
    const int x = c.x0 + it.lx, y = c.y0 + it.ly;
    if (it.i < c.npx && x < c.W && y < c.H) {
      float* const err = error_map ? row_ptr(error_map, p.err_pitch, y) + x : nullptr;
      if (j[k] < 0 || isnan(vx[k])) {
        if (err) *err = 0.0f;
      } else {
        const int fi = it.ly * c.pf + it.lx + c.shf;
        const float3 vcurr = make_float3(SM_F32(c.oV)[fi], SM_F32(c.oV)[c.fplane + fi], SM_F32(c.oV)[2 * c.fplane + fi]);
        const float3 vcurr_g = xadd(xmul(P.Rcurr, vcurr), tcurr);
        const float3 vcurr_cp = xmul(P.Rprev_inv, xsub(vcurr_g, tprev));
        const float3 vp = make_float3(vx[k], q[k][0], q[k][1]);
        const float3 np = make_float3(q[k][2], q[k][3], q[k][4]);
        const float3 ncurr = make_float3(SM_F32(c.oN)[fi], SM_F32(c.oN)[c.fplane + fi], SM_F32(c.oN)[2 * c.fplane + fi]);
        const float3 ncurr_g = xmul(P.Rcurr, ncurr);
        const float dist = xnorm(xsub(vp, vcurr_g));
        const float sine = xnorm(xcross(ncurr_g, np));
        if (err) *err = isfinite(dist) ? dist : 0.0f;
        if (sine < p.angleThres && dist <= p.distThres && !isnan(ncurr.x) && !isnan(np.x)) {
          any = true;
          icp_found_row(P, tprev, vcurr_cp, vp, np, acc);
        }
      }
    }
    pix_next(c, it);
  }
  store_warp_row(buf, any, acc);
}

__device__ __noinline__ void phase3_obj(int lvl, int m, float sigma, int buf) {
  TSMEM();
  const LvCtx& c = sm.lv;
  float acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.f;
  bool any = false;
  const int* bc = sm.box[m];
  const bool none = c.x0 > bc[2] || c.x0 + c.tw <= bc[0] || c.y0 > bc[3] || c.y0 + c.th <= bc[1];
  if (!none) {
    const size_t kstride = (size_t)gridDim.x * kT;
    const unsigned* cz = p.M[m].corrZ + (size_t)blockIdx.x * kT + threadIdx.x;
    const float* cd = p.M[m].corrD + (size_t)blockIdx.x * kT + threadIdx.x;
    unsigned z[kPP];
    float d0[kPP];
#pragma unroll
    for (int k = 0; k < kPP; ++k) {  // written by this thread in phase 1 (plain loads: the read-only path may be stale)
      const bool live = k * kT + (int)threadIdx.x < c.npx;
      z[k] = live ? cz[k * kstride] : kNoCorr;
      d0[k] = live ? cd[k * kstride] : 0.f;
    }
    PixIt it = pix_begin(c);
#pragma unroll
    for (int k = 0; k < kPP; ++k) {
      if (z[k] != kNoCorr) {
        any = true;
        const int si = it.ly * c.ps + it.lx + c.shs;
        rgb_row(c, sigma, p.sobelScale, (int)(z[k] & 0x7ffu), (int)((z[k] >> 11) & 0x7ffu), d0[k], (float)((int)(z[k] >> 22) - 256),
                SM_S16(c.oDX)[si], SM_S16(c.oDY)[si], acc);
      }
      pix_next(c, it);
    }
  }
  store_warp_row(buf, any, acc);
}

// ------------------------------------------------------------------------- exact grid-wide sums
// Thread t < nm * NS adds sum (m = t / NS, j = t % NS) of this CTA (blk[m][j], see fold_warp_rows) to the global
// accumulators of the round.  The f32 partial is split exactly: d = hi * 2^8 + rem, |rem| < 2^8,
// lo = rint(rem * 2^39) (|error| <= 2^-40); both integers go up by 8 bits and carry a 1 in the low byte, so a
// word also counts its contributions.  Integer addition commutes: the grid total does not depend on the
// order in which the CTAs arrive.
template <int NS>
__device__ __forceinline__ void publish_sums(unsigned round, bool fold_rows) {
  TSMEM();
  const int t = threadIdx.x, m = t / NS, j = t - m * NS;
  float sum;
  if (fold_rows) {  // one model: the ICP rows are in buffer 0, the RGB rows in buffer 1; folded here, in warp order
    const int set = j >= 29 ? 1 : 0;
    const float* r = SM_F32(p.o_wrow) + (size_t)set * kNW * 32 + (j - 29 * set);
    sum = 0.f;
#pragma unroll
    for (int w = 0; w < kNW; ++w) sum += r[w * 32];
  } else {
    sum = SM_F32(p.o_blk)[m * 64 + j];
  }
  double d = (double)sum;
  if (!(fabs(d) < 9.0e15)) d = 0.0;  // non-finite (or absurd) partial: contributes nothing but still counts
  const long long hi = (long long)(d * (1.0 / 256.0));
  const long long lo = __double2ll_rn((d - (double)hi * 256.0) * 549755813888.0 /* 2^39 */);
  unsigned long long* x = p.xacc + (((size_t)round * p.nmodels + m) * kXWords + 2 * j) * kXStride;
  red_add_u64(x, ((unsigned long long)hi << 8) + 1ull);
  red_add_u64(x + kXStride, ((unsigned long long)lo << 8) + 1ull);
}

// thread t < nm * NS reads its two words -- again while one of them does not count G contributions yet -- into
// outd[m][j] (double).  No fence anywhere: a word is complete when its low byte says so.  (A one-thread wait on word 0
// in front of the readers, as a hint, cost one L2 round trip per iteration: 0.286 -> 0.280 ms per launch without it.)
template <int NS>
__device__ __forceinline__ void collect_sums(unsigned round, int nactive_threads) {
  TSMEM();
  const unsigned G = gridDim.x;
  const int t = threadIdx.x;
  if (t < nactive_threads) {
    const int m = t / NS, j = t - m * NS;
    const unsigned long long* x = p.xacc + (((size_t)round * p.nmodels + m) * kXWords + 2 * j) * kXStride;
    unsigned long long a, b;
    do {
      a = ld_u64_relaxed(x);
      b = ld_u64_relaxed(x + kXStride);
    } while ((unsigned)(a & 0xffull) != G || (unsigned)(b & 0xffull) != G);
    double* outd = reinterpret_cast<double*>(dyn_smem_raw + p.o_out) + m * 64;
    outd[j] = (double)((long long)a >> 8) * 256.0 + (double)((long long)b >> 8) * (1.0 / 549755813888.0);
  }
  __syncthreads();
}

// ------------------------------------------------------------------------- FP64 Gauss-Newton step, one warp
// exp of a rotation vector without sqrt / division / sin / cos: R = I + A [r]x + B [r]x^2 with
// A = sin(t)/t, B = (1 - cos t)/t^2 as series in t^2 (|r| <= 0.5: truncation < 1e-17); the library
// Rodrigues formula (gn_math.h) for anything larger
__device__ __forceinline__ void exp_so3(const double r[3], double R[9]) {
  const double x = r[0], y = r[1], z = r[2];
  const double t2 = x * x + y * y + z * z;
  if (t2 > 0.25) {
    gn::rodrigues(r, R);
    return;
  }
  double A = 1.0 - t2 * (1.0 / 210.0);
  A = 1.0 - t2 * (1.0 / 156.0) * A;
  A = 1.0 - t2 * (1.0 / 110.0) * A;
  A = 1.0 - t2 * (1.0 / 72.0) * A;
  A = 1.0 - t2 * (1.0 / 42.0) * A;
  A = 1.0 - t2 * (1.0 / 20.0) * A;
  A = 1.0 - t2 * (1.0 / 6.0) * A;
  double B = 1.0 - t2 * (1.0 / 240.0);
  B = 1.0 - t2 * (1.0 / 182.0) * B;
  B = 1.0 - t2 * (1.0 / 132.0) * B;
  B = 1.0 - t2 * (1.0 / 90.0) * B;
  B = 1.0 - t2 * (1.0 / 56.0) * B;
  B = 1.0 - t2 * (1.0 / 30.0) * B;
  B = 1.0 - t2 * (1.0 / 12.0) * B;
  B *= 0.5;
  R[0] = 1.0 - B * (y * y + z * z);
  R[1] = B * x * y - A * z;
  R[2] = B * x * z + A * y;
  R[3] = B * x * y + A * z;
  R[4] = 1.0 - B * (x * x + z * z);
  R[5] = B * y * z - A * x;
  R[6] = B * x * z - A * y;
  R[7] = B * y * z + A * x;
  R[8] = 1.0 - B * (x * x + y * y);
}

// lower-triangular LDL^T of the 6x6 normal equations in registers (every lane runs it redundantly: no
// exchange, and the pose update that follows is spread over the lanes)
__device__ __forceinline__ void ldlt6_lower(double (&A)[21], double (&b)[6], double (&x)[6]) {
#define LA(i, j) A[(i) * ((i) + 1) / 2 + (j)]
  double inv[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const double d = LA(k, k);
    inv[k] = (d != 0.0) ? 1.0 / d : 0.0;
    double l[6];
#pragma unroll
    for (int i = k + 1; i < 6; ++i) l[i] = LA(i, k) * inv[k];
#pragma unroll
    for (int i = k + 1; i < 6; ++i)
#pragma unroll
      for (int j = k + 1; j <= i; ++j) LA(i, j) -= l[i] * LA(j, k);
#pragma unroll
    for (int i = k + 1; i < 6; ++i) LA(i, k) = l[i];
  }
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = 0; j < i; ++j) b[i] -= LA(i, j) * b[j];
#pragma unroll
  for (int i = 0; i < 6; ++i) b[i] *= inv[i];  // a zero pivot (no inliers) yields a zero component
#pragma unroll
  for (int i = 5; i >= 0; --i)
#pragma unroll
    for (int j = i + 1; j < 6; ++j) b[i] -= LA(j, i) * b[j];
#pragma unroll
  for (int i = 0; i < 6; ++i) x[i] = b[i];
#undef LA
}

// RGBDOdometry.cpp:412-460 (+ :464-467 on the last iteration) by the 32 lanes of one warp
__device__ __noinline__ void gn_solve_warp(int m, int lvl_next, int is_last, float tmpError, int cnt) {
  TSMEM();
  GNState* g = &sm.S[m];
  const double* out = reinterpret_cast<const double*>(dyn_smem_raw + p.o_out) + m * 64;  // [0..28] ICP sums, [29..57] RGB sums
  double* sA = sm.solveA[m];
  const int lane = threadIdx.x & 31;
  const double w = p.icpWeight;
  // 1. normal equations: lane l combines packed sum l (order aa..ag, bb..bg, ..., fg; types.cuh:101-112)
  if (lane < 27) {
    int i = 0, rem = lane;
    while (rem >= 7 - i) {
      rem -= 7 - i;
      ++i;
    }
    const int j = i + rem;
    const double icp = out[lane], rgb = out[29 + lane];
    if (j == 6) {
      sA[36 + i] = rgb + w * icp;
    } else {
      const double v = rgb + w * w * icp;
      sA[i * 6 + j] = v;
      sA[j * 6 + i] = v;
    }
  }
  if (lane == 27) {
    TrackStats& st = g->stats;
    st.lastRGBError = tmpError;
    st.lastRGBCount = (float)cnt;
    st.lastICPError = sqrtf((float)out[27]) / (float)out[28];
    st.lastICPCount = (float)out[28];
  }
  __syncwarp();
  if (is_last) {  // lastA / lastb are reported for the final iteration (RGBDOdometry.h:62-70)
    for (int q = lane; q < 42; q += 32) (q < 36 ? g->stats.lastA[q] : g->stats.lastb[q - 36]) = sA[q];
  }
  // 2. solve (redundantly in every lane)
  double A[21], b[6], x[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
#pragma unroll
    for (int j = 0; j <= i; ++j) A[i * (i + 1) / 2 + j] = sA[i * 6 + j];
    b[i] = sA[36 + i];
  }
  ldlt6_lower(A, b, x);
  // 3. resultRt <- [exp(x[3..5]) | x[0..2]] * resultRt: lane (r, c) owns one element of the top 3 rows
  double Rm[9];
  {
    const double rv[3] = {x[3], x[4], x[5]};
    exp_so3(rv, Rm);
  }
  double nrt = 0.0;
  if (lane < 12) {
    const int r = lane >> 2, c = lane & 3;
    const double* Rt = g->resultRt;
    nrt = Rm[r * 3] * Rt[c] + Rm[r * 3 + 1] * Rt[4 + c] + Rm[r * 3 + 2] * Rt[8 + c] + x[r] * Rt[12 + c];
  }
  __syncwarp();
  if (lane < 12) g->resultRt[lane] = nrt;
  __syncwarp();
  double Rt[12];
#pragma unroll
  for (int q = 0; q < 12; ++q) Rt[q] = g->resultRt[q];
  // 4a. lanes 0..11: [Rcurr|tcurr] = [Rprev|tprev] * (f32 resultRt)^-1 (gn::compose_pose)
  if (lane < 12) {
    float Ro[9], to[3], ti[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
      for (int c = 0; c < 3; ++c) Ro[r * 3 + c] = (float)Rt[r * 4 + c];
      to[r] = (float)Rt[r * 4 + 3];
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) ti[r] = -(Ro[r] * to[0] + Ro[3 + r] * to[1] + Ro[6 + r] * to[2]);
    const float* Rp = g->Rprev;
    const float* tp = g->pose.tprev;
    float val;
    if (lane < 9) {
      const int r = lane / 3, c = lane - 3 * r;
      val = Rp[r * 3] * Ro[c * 3] + Rp[r * 3 + 1] * Ro[c * 3 + 1] + Rp[r * 3 + 2] * Ro[c * 3 + 2];
    } else {
      const int r = lane - 9;
      val = Rp[r * 3] * ti[0] + Rp[r * 3 + 1] * ti[1] + Rp[r * 3 + 2] * ti[2] + tp[r];
    }
    if (lane < 9)
      g->pose.Rcurr.m[lane] = val;
    else
      g->pose.tcurr[lane - 9] = val;
    if (is_last) {  // RGBDOdometry.cpp:464-467: photometric sanity reset, decided on the translation
      const float tc0 = __shfl_sync(0xfffu, val, 9), tc1 = __shfl_sync(0xfffu, val, 10), tc2 = __shfl_sync(0xfffu, val, 11);
      const float d0 = tc0 - tp[0], d1 = tc1 - tp[1], d2 = tc2 - tp[2];
      const bool reset = sqrtf(d0 * d0 + d1 * d1 + d2 * d2) > 0.3f;
      if (lane < 9)
        g->out_rot[lane] = reset ? Rp[lane] : val;
      else
        g->out_trans[lane - 9] = reset ? tp[lane - 9] : val;
    }
  } else if (lane >= 16 && lane < 28 && !is_last) {
    // 4b. lanes 16..27: warp of the next iteration, krkinv = K R' K^-1, kt = K t' with [R'|t'] = resultRt^-1
    const int e = lane - 16;
    const double* K = sm.K[lvl_next];
    const double* Kinv = sm.Kinv[lvl_next];
    double R[9], tt[3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) R[i * 3 + j] = Rt[j * 4 + i];
#pragma unroll
    for (int i = 0; i < 3; ++i) tt[i] = -(R[i * 3] * Rt[3] + R[i * 3 + 1] * Rt[7] + R[i * 3 + 2] * Rt[11]);
    if (e < 9) {
      const int i = e / 3, j = e - 3 * i;
      double tmp[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) tmp[k] = K[i * 3] * R[k] + K[i * 3 + 1] * R[3 + k] + K[i * 3 + 2] * R[6 + k];
      g->warp.krkinv.m[e] = (float)(tmp[0] * Kinv[j] + tmp[1] * Kinv[3 + j] + tmp[2] * Kinv[6 + j]);
    } else {
      const int i = e - 9;
      g->warp.kt[i] = (float)(K[i * 3] * tt[0] + K[i * 3 + 1] * tt[1] + K[i * 3 + 2] * tt[2]);
    }
  }
  __syncwarp();
}

// H = K R K^-1 etc. of the SO(3) step (as the host loop in odometry.cu), lane e < 9 owns element e
__device__ __forceinline__ void so3_matrices_warp(GNState* g) {
  TSMEM();
  const int lane = threadIdx.x & 31;
  if (lane < 9) {
    const double* K = sm.K[2];
    const double* Kinv = sm.Kinv[2];
    const double* R = g->resultR;
    const int i = lane / 3, j = lane - 3 * i;
    double kr[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) kr[k] = K[i * 3] * R[k] + K[i * 3 + 1] * R[3 + k] + K[i * 3 + 2] * R[6 + k];
    g->so3_imageBasis.m[lane] = (float)(kr[0] * Kinv[j] + kr[1] * Kinv[3 + j] + kr[2] * Kinv[6 + j]);
    g->so3_kinv.m[lane] = (float)Kinv[lane];
    g->so3_krlr.m[lane] = (float)kr[j];
  }
  __syncwarp();
}

// RGBDOdometry.cpp:320-328: seed resultRt with the SO(3) rotation, first photometric warp
__device__ __forceinline__ void gn_begin_warp(GNState* g, int use_so3, int lvl_first) {
  TSMEM();
  const int lane = threadIdx.x & 31;
  if (lane < 16) {
    const int r = lane >> 2, c = lane & 3;
    double v = (r == c) ? 1.0 : 0.0;
    if (use_so3 && r < 3 && c < 3) v = g->resultR[r * 3 + c];
    g->resultRt[lane] = v;
  }
  __syncwarp();
  if (lane < 12) {  // translation of resultRt is zero: krkinv = K R^T K^-1, kt = 0
    const double* K = sm.K[lvl_first];
    const double* Kinv = sm.Kinv[lvl_first];
    const double* Rt = g->resultRt;
    if (lane < 9) {
      const int i = lane / 3, j = lane - 3 * i;
      double tmp[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) tmp[k] = K[i * 3] * Rt[k * 4] + K[i * 3 + 1] * Rt[k * 4 + 1] + K[i * 3 + 2] * Rt[k * 4 + 2];
      g->warp.krkinv.m[lane] = (float)(tmp[0] * Kinv[j] + tmp[1] * Kinv[3 + j] + tmp[2] * Kinv[6 + j]);
    } else {
      g->warp.kt[lane - 9] = 0.f;
    }
  }
  __syncwarp();
}

// host logic of one SO(3) iteration after the reduction (RGBDOdometry.cpp:281-308) by one warp
__device__ __noinline__ void so3_update_warp(int m, int it) {
  TSMEM();
  GNState* g = &sm.S[m];
  const double* outd = reinterpret_cast<const double*>(dyn_smem_raw + p.o_out) + m * 64;
  float out[11];
#pragma unroll
  for (int q = 0; q < 11; ++q) out[q] = (float)outd[q];
  const int lane = threadIdx.x & 31;
  TrackStats& st = g->stats;
  const float err = sqrtf(out[9]) / out[10], count = out[10];
  const float lastError = g->so3_lastError, lastCount = g->so3_lastCount;
  __syncwarp();
  int done = 0;
  if (err < lastError && fabsf(lastError - count) < 0.001f) {
    done = 1;
    if (lane == 0) {
      st.lastSO3Error = err;
      st.lastSO3Count = count;
    }
  } else if (err > lastError + 0.001f) {
    done = 1;
    if (lane == 0) {
      st.lastSO3Error = lastError;
      st.lastSO3Count = lastCount;
    }
    if (lane < 9) g->resultR[lane] = g->lastResultR[lane];
  }
  if (lane == 0) st.so3_iterations++;
  if (!done) {
    float jtj[9], jtr[3];
    gn::unpack_so3(out, jtj, jtr);
    double Ad[9], bd[3], xd[3];
#pragma unroll
    for (int q = 0; q < 9; ++q) Ad[q] = jtj[q];
#pragma unroll
    for (int q = 0; q < 3; ++q) bd[q] = jtr[q];
    gn::ldlt_solve_unrolled<3>(Ad, bd, xd);
    const double delta[3] = {(double)(float)xd[0], (double)(float)xd[1], (double)(float)xd[2]};
    double rotUpdate[9];
    exp_so3(delta, rotUpdate);
    float nr = 0.f;
    if (lane < 9) {
      const int r = lane / 3, c = lane - 3 * r;
      nr = (float)rotUpdate[r * 3] * g->R_lr[c] + (float)rotUpdate[r * 3 + 1] * g->R_lr[3 + c] +
           (float)rotUpdate[r * 3 + 2] * g->R_lr[6 + c];
    }
    __syncwarp();
    if (lane < 9) {
      g->lastResultR[lane] = g->resultR[lane];
      g->R_lr[lane] = nr;
      g->resultR[lane] = nr;
    }
    if (lane == 0) {
      st.lastSO3Error = err;
      st.lastSO3Count = count;
      g->so3_lastError = err;
      g->so3_lastCount = count;
    }
    __syncwarp();
    so3_matrices_warp(g);
  }
  __syncwarp();
  if (done || it == 9) {
    if (lane == 0) g->so3_done = 1;
    gn_begin_warp(g, 1, sm.nsched ? sm.sched[0] : 0);
  }
  __syncwarp();
}

// reset the state of model m for a new frame (RGBDOdometry.cpp:224-255, :316-318) by one warp
__device__ __forceinline__ void gn_init_warp(int m) {
  TSMEM();
  GNState* g = &sm.S[m];
  const float* pose_in = p.M[m].pose_in;
  const int lane = threadIdx.x & 31;
  if (lane < 9) {
    const float r = __ldcg(pose_in + 3 + lane);
    g->Rprev[lane] = r;
    g->pose.Rcurr.m[lane] = r;
    g->out_rot[lane] = r;
    const double id = (lane % 4 == 0) ? 1.0 : 0.0;
    g->resultR[lane] = id;
    g->lastResultR[lane] = id;
    g->R_lr[lane] = (float)id;
  } else if (lane < 12) {
    const float t = __ldcg(pose_in + lane - 9);
    g->pose.tprev[lane - 9] = t;
    g->pose.tcurr[lane - 9] = t;
    g->out_trans[lane - 9] = t;
  } else if (lane == 12) {
    g->so3_lastError = FLT_MAX / 2;
    g->so3_lastCount = FLT_MAX / 2;
    g->so3_done = 0;
    TrackStats z = {};
    g->stats = z;
  } else if (lane >= 16) {  // resultRt = identity; the top rows are set again by gn_begin_warp
    const int q = lane - 16;
    g->resultRt[q] = (q % 5 == 0) ? 1.0 : 0.0;
  }
  __syncwarp();
  if (lane == 0) gn::inverse3f(g->Rprev, g->pose.Rprev_inv.m);
  so3_matrices_warp(g);
}

// --------------------------------------------------------------------------------- level set-up
// cooperative fill of a shared-memory box from a planar image (zero outside): staged == 2
template <class T>
__device__ __forceinline__ void fill_box(T* dst, const T* src, int W, int H, int x0, int y0, int bw, int bh) {
  for (int i = threadIdx.x; i < bw * bh; i += kT) {
    const int ly = i / bw, lx = i - ly * bw, x = x0 + lx, y = y0 + ly;
    dst[i] = (x >= 0 && y >= 0 && x < W && y < H) ? __ldg(src + (size_t)y * W + x) : (T)0;
  }
}

__device__ __forceinline__ void issue_frame_tma(int lvl) {  // one thread
  TSMEM();
  const FLevel& F = p.F[lvl];
  const MLevel& L = p.M[0].L[lvl];
  const int x0 = (blockIdx.x % p.gx) * F.tw, y0 = (blockIdx.x / p.gx) * F.th;
  const int xf = floor_to(x0, 4), xs = floor_to(x0, 8), xb = floor_to(x0, 16);  // 16-byte aligned box origins
  unsigned long long* bar = &sm.bar_frame[lvl];
  tmap_acquire(F.tm_v);
  tmap_acquire(F.tm_n);
  tmap_acquire(F.tm_dx);
  tmap_acquire(F.tm_dy);
  tmap_acquire(F.tm_img);
  tmap_acquire(L.tm_d1);
  tmap_acquire(L.tm_cand);
  tmap_acquire(L.tm_pv);
  tmap_acquire(L.tm_pn);
  tmap_acquire(L.tm_ld);
  tmap_acquire(L.tm_li);
  mbar_expect_tx(bar, F.frame_bytes);
  tma_load_3d(dyn_smem_raw + F.o_v, F.tm_v, xf, y0, 0, bar);
  tma_load_3d(dyn_smem_raw + F.o_n, F.tm_n, xf, y0, 0, bar);
  tma_load_2d(dyn_smem_raw + F.o_dx, F.tm_dx, xs, y0, bar);
  tma_load_2d(dyn_smem_raw + F.o_dy, F.tm_dy, xs, y0, bar);
  tma_load_2d(dyn_smem_raw + F.o_img, F.tm_img, xb, y0, bar);
  tma_load_2d(dyn_smem_raw + F.o_d1, L.tm_d1, xf, y0, bar);
  tma_load_2d(dyn_smem_raw + F.o_cand, L.tm_cand, xb, y0, bar);
}

__device__ __noinline__ void level_begin(int lvl, unsigned& win_phase) {
  TSMEM();
  const FLevel& F = p.F[lvl];
  if ((int)threadIdx.x < p.nmodels * 8) {  // model extents of this level (visible after the barriers below)
    const int m = threadIdx.x >> 3, k = threadIdx.x & 7;
    const int* b = p.M[m].L[lvl].box;
    int v = (k & 2) ? ((k & 1) ? F.h - 1 : F.w - 1) : 0;
    if (b) v = (k & 2) ? -__ldg(b + k) : __ldg(b + k);
    sm.box[m][k] = v;
  }
  if (!F.staged) {
    if (threadIdx.x == 0) make_lvctx(lvl);
    __syncthreads();
    return;
  }
  const MLevel& L = p.M[0].L[lvl];
  const int x0 = (blockIdx.x % p.gx) * F.tw, y0 = (blockIdx.x / p.gx) * F.th;
  const int xf = floor_to(x0, 4), xs = floor_to(x0, 8), xb = floor_to(x0, 16);
  if (F.staged == 1) {
    mbar_wait(&sm.bar_frame[lvl], 0);
  } else {
    const size_t hw = (size_t)F.w * F.h;
    const int fplane = F.pf * F.th;
    for (int k = 0; k < 3; ++k) {
      fill_box(SM_F32(F.o_v) + k * fplane, F.vmap_curr + k * hw, F.w, F.h, xf, y0, F.pf, F.th);
      fill_box(SM_F32(F.o_n) + k * fplane, F.nmap_curr + k * hw, F.w, F.h, xf, y0, F.pf, F.th);
    }
    fill_box(SM_S16(F.o_dx), F.dIdx, F.w, F.h, xs, y0, F.ps, F.th);
    fill_box(SM_S16(F.o_dy), F.dIdy, F.w, F.h, xs, y0, F.ps, F.th);
    fill_box(SM_U8(F.o_img), F.nextImage, F.w, F.h, xb, y0, F.pb, F.th);
    fill_box(SM_F32(F.o_d1), L.nextDepth, F.w, F.h, xf, y0, F.pf, F.th);
    fill_box(SM_U8(F.o_cand), L.cand, F.w, F.h, xb, y0, F.pb, F.th);
  }
  if (threadIdx.x < 3) sm.winacc[threadIdx.x] = 0;
  __syncthreads();
  // mean displacement of the tile's photometric candidates under the current estimate of the camera model
  {
    const RgbWarp& Wp = sm.S[0].warp;
    const float* kk = Wp.krkinv.m;
    const float* sD1 = SM_F32(F.o_d1);
    const unsigned char* sC = SM_U8(F.o_cand);
    const int shf = x0 - xf, shb = x0 - xb;
    int sx = 0, sy = 0, n = 0;
    for (int i = threadIdx.x; i < F.npx; i += kT) {
      const int ly = i / F.tw, lx = i - ly * F.tw, x = x0 + lx, y = y0 + ly;
      if (x < F.w && y < F.h && sC[ly * F.pb + lx + shb]) {
        const float d1 = sD1[ly * F.pf + lx + shf];
        const float td1 = d1 * (kk[6] * x + kk[7] * y + kk[8]) + Wp.kt[2];
        const int u0 = __float2int_rn((d1 * (kk[0] * x + kk[1] * y + kk[2]) + Wp.kt[0]) / td1);
        const int v0 = __float2int_rn((d1 * (kk[3] * x + kk[4] * y + kk[5]) + Wp.kt[1]) / td1);
        const int dx = u0 - x, dy = v0 - y;
        if (abs(dx) < 64 && abs(dy) < 64) {
          sx += dx;
          sy += dy;
          n += 1;
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sx += __shfl_xor_sync(0xffffffffu, sx, o);
      sy += __shfl_xor_sync(0xffffffffu, sy, o);
      n += __shfl_xor_sync(0xffffffffu, n, o);
    }
    if ((threadIdx.x & 31) == 0 && n) {
      atomicAdd(&sm.winacc[0], sx);
      atomicAdd(&sm.winacc[1], sy);
      atomicAdd(&sm.winacc[2], n);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int n = sm.winacc[2];
    const int mx = n ? __float2int_rn((float)sm.winacc[0] / (float)n) : 0;
    const int my = n ? __float2int_rn((float)sm.winacc[1] / (float)n) : 0;
    const int wx0 = x0 + mx - F.halo, wy0 = y0 + my - F.halo;
    sm.win_x0 = wx0;
    sm.win_y0 = wy0;
    make_lvctx(lvl);
    if (F.staged == 1) {
      // the window region was read by the previous level through the generic proxy
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(&sm.bar_win, F.win_bytes);
      const int wxf = floor_to(wx0, 4), wxb = floor_to(wx0, 16);
      tma_load_3d(dyn_smem_raw + F.o_pv, L.tm_pv, wxf, wy0, 0, &sm.bar_win);
      tma_load_3d(dyn_smem_raw + F.o_pn, L.tm_pn, wxf, wy0, 0, &sm.bar_win);
      tma_load_2d(dyn_smem_raw + F.o_ld, L.tm_ld, wxf, wy0, &sm.bar_win);
      tma_load_2d(dyn_smem_raw + F.o_li, L.tm_li, wxb, wy0, &sm.bar_win);
    }
  }
  __syncthreads();
  if (F.staged == 1) {
    mbar_wait(&sm.bar_win, win_phase);
    win_phase ^= 1u;
  } else {
    const int wx0 = sm.win_x0, wy0 = sm.win_y0, wplane = F.wpf * F.wh;
    const int wxf = floor_to(wx0, 4), wxb = floor_to(wx0, 16);
    const size_t hw = (size_t)F.w * F.h;
    for (int k = 0; k < 3; ++k) {
      fill_box(SM_F32(F.o_pv) + k * wplane, L.vmap_g_prev + k * hw, F.w, F.h, wxf, wy0, F.wpf, F.wh);
      fill_box(SM_F32(F.o_pn) + k * wplane, L.nmap_g_prev + k * hw, F.w, F.h, wxf, wy0, F.wpf, F.wh);
    }
    fill_box(SM_F32(F.o_ld), L.lastDepth, F.w, F.h, wxf, wy0, F.wpf, F.wh);
    fill_box(SM_U8(F.o_li), L.lastImage, F.w, F.h, wxb, wy0, F.wpb, F.wh);
    __syncthreads();
  }
}

// --------------------------------------------------------------------------------- the iterations
// GENERAL = false: one model, every level staged -- the phases of object models and of unstaged levels are not even
// compiled in (the lean kernel is 10 % faster: a third less code around the same hot loop)
template <bool GENERAL, bool DBGT>
__device__ __noinline__ void run_level(int lvl, int q0, int nit, unsigned round0) {
  TSMEM();
  const int NM = GENERAL ? p.nmodels : 1, G = gridDim.x;  // the lean kernel: loops over one model fold away
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool FS = p.F[lvl].staged != 0;
  int wbuf = 0;
  for (int it = 0; it < nit; ++it) {
    const int q = q0 + it;
    const unsigned round = round0 + it;
    const bool last_of_l0 = (lvl == 0 && it + 1 == nit);
    DBG_MARK(8 + q * 8 + 0);
    DBG_CTA(q, 0);

    // -------- phase 1: photometric correspondences of every model, then arrive at barrier A
    for (int m = 0; m < NM; ++m) {
      if (FS && m == 0)
        phase1<true, true>(lvl, m);
      else if (GENERAL && FS)
        phase1_obj(lvl, m);
      else if (GENERAL)
        phase1<false, false>(lvl, m);
    }
    __syncthreads();
    if ((int)warp < NM) {  // integer sums commute exactly; the payload rides on the arrival itself (warp m: model m)
      unsigned cc = lane < kNW ? (unsigned)sm.cntw[warp][lane] : 0u, ss = lane < kNW ? (unsigned)sm.sigw[warp][lane] : 0u;
      cc = __reduce_add_sync(0xffffffffu, cc);
      ss = __reduce_add_sync(0xffffffffu, ss);
      if (lane == 0)
        red_add_u64(&p.acnt[round * kMaxM + warp], 1ull | ((unsigned long long)cc << 8) | ((unsigned long long)ss << 32));
    }
    DBG_MARK(8 + q * 8 + 1);
    DBG_CTA(q, 1);

    // -------- phase 2: ICP rows (independent of the counts: hides barrier A)
    for (int m = 0; m < NM; ++m, wbuf ^= 1) {
      float* const err = last_of_l0 ? p.M[m].err : nullptr;
      if (FS && m == 0)
        phase2<true, true>(lvl, m, err, wbuf);
      else if (GENERAL && FS)
        phase2_obj(lvl, m, err, wbuf);
      else if (GENERAL)
        phase2<false, false>(lvl, m, err, wbuf);
      if (GENERAL) {  // (one model: both sets of rows are folded by the publishing threads, see publish_sums)
        __syncthreads();
        fold_warp_rows(wbuf, m, 0, 29);
      }
    }
    DBG_MARK(8 + q * 8 + 2);
    DBG_CTA(q, 2);
    if ((int)threadIdx.x < NM) {  // wait for barrier A: all G arrivals carry the global count / sigma
      unsigned long long v;
      do {
        v = ld_u64_relaxed(&p.acnt[round * kMaxM + threadIdx.x]);
      } while ((int)(v & 0xffull) != G);
      sm.tot[threadIdx.x][0] = (int)((v >> 8) & 0xffffffull);
      sm.tot[threadIdx.x][1] = (int)(unsigned)(v >> 32);
    }
    __syncthreads();
    DBG_MARK(8 + q * 8 + 3);

    // -------- phase 3: RGB rows weighted with the global count
    for (int m = 0; m < NM; ++m) {
      float tmpErr;
      const float sigma = rgb_sigma_from_counts(sm.tot[m][0], sm.tot[m][1], &tmpErr);
      if (threadIdx.x == 0) sm.tmpErr[m] = tmpErr;
      if (FS && m == 0)
        phase3<true, true>(lvl, m, sigma, wbuf);
      else if (GENERAL && FS)
        phase3_obj(lvl, m, sigma, wbuf);
      else if (GENERAL)
        phase3<false, false>(lvl, m, sigma, wbuf);
      __syncthreads();
      if (GENERAL) fold_warp_rows(wbuf, m, 1, 29);
      wbuf ^= 1;
    }
    if (GENERAL) __syncthreads();
    DBG_MARK(8 + q * 8 + 4);
    DBG_CTA(q, 3);

    // -------- add this CTA's sums to the grid accumulators, read the totals, solve
    if ((int)threadIdx.x < NM * kSums) publish_sums<kSums>(round, !GENERAL);
    DBG_MARK(8 + q * 8 + 5);
    collect_sums<kSums>(round, NM * kSums);
    DBG_MARK(8 + q * 8 + 6);
    DBG_CTA(q, 4);
    const int is_last = (q + 1 == sm.nsched);
    if ((int)warp < NM) {
      const int m = (int)warp;
      if (lane < 29) sm.S[m].icp_result[lane] = (float)reinterpret_cast<const double*>(dyn_smem_raw + p.o_out)[m * 64 + lane];
      gn_solve_warp(m, is_last ? sm.sched[q] : sm.sched[q + 1], is_last, sm.tmpErr[m], sm.tot[m][0]);
    }
    __syncthreads();
    DBG_MARK(8 + q * 8 + 7);
  }
}

// SO(3) pre-alignment of every model on level 2 (RGBDOdometry.cpp:239-310); returns the rounds used
template <bool GENERAL>
__device__ __noinline__ unsigned run_so3() {
  TSMEM();
  const int NM = GENERAL ? p.nmodels : 1;
  const FLevel& F = p.F[2];
  const int x0 = (blockIdx.x % p.gx) * F.tw, y0 = (blockIdx.x / p.gx) * F.th;
  const unsigned warp = threadIdx.x >> 5;
  unsigned round = 0;
  int wbuf = 0;
  for (int it = 0; it < 10; ++it) {
    bool all_done = true;  // identical in every CTA
    for (int m = 0; m < NM; ++m) all_done = all_done && sm.S[m].so3_done;
    if (all_done) break;
    for (int m = 0; m < NM; ++m) {
      float acc[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = 0.f;
      bool work = false;
      if (!sm.S[m].so3_done) {  // a finished model contributes zeros (its words still count every CTA)
        const GNState& S = sm.S[m];
        for (int i = threadIdx.x; i < F.npx; i += kT) {
          const int ly = i / F.tw, lx = i - ly * F.tw, x = x0 + lx, y = y0 + ly;
          if (x < F.w && y < F.h) {
            so3_pixel(p.M[m].so3_last, p.M[m].so3_next, (size_t)F.w, F.w, F.h, S.so3_imageBasis, S.so3_kinv, S.so3_krlr, x, y, acc);
            work = true;
          }
        }
      }
      store_warp_row(wbuf, work, acc);
      __syncthreads();
      fold_warp_rows(wbuf, m, 0, 11);
      wbuf ^= 1;
    }
    __syncthreads();
    if ((int)threadIdx.x < NM * 11) publish_sums<11>(round, false);
    collect_sums<11>(round, NM * 11);
    if ((int)warp < NM && !sm.S[warp].so3_done) so3_update_warp((int)warp, it);
    __syncthreads();
    ++round;
  }
  return round;
}

template <bool GENERAL, bool DBGT>
__global__ void __launch_bounds__(kT, 1) gn_tiled_kernel(const TParams kp) {
  extern __shared__ __align__(128) unsigned char dyn_smem_raw[];
  TFixed& sm = *reinterpret_cast<TFixed*>(dyn_smem_raw);
  {  // parameters -> shared memory (the phase functions are not inlined)
    const int* src = reinterpret_cast<const int*>(&kp);
    int* dst = reinterpret_cast<int*>(&sm.prm);
    for (int i = threadIdx.x; i < (int)(sizeof(TParams) / 4); i += kT) dst[i] = src[i];
  }
  if (threadIdx.x == 0) {
    int n = 0;
    for (int i = 2; i >= 0; --i)
      for (int j = 0; j < kp.iters[i] && n < 19; ++j) sm.sched[n++] = i;
    sm.nsched = n;
    for (int l = 0; l < 3; ++l) mbar_init(&sm.bar_frame[l], 1);
    mbar_init(&sm.bar_win, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (threadIdx.x >= 32 && threadIdx.x < 35) {
    const int l = threadIdx.x - 32;
    const LevelK k = kp.F[l].k;
    gn::make_K(k.fx, k.fy, k.cx, k.cy, sm.K[l], sm.Kinv[l]);
  }
  __syncthreads();
  const TParams& p = sm.prm;
  const int NM = GENERAL ? p.nmodels : 1;
  const unsigned warp = threadIdx.x >> 5;
  DBG_MARK(0);
  // every level's frame tiles are requested now; the finer levels land while the coarser ones iterate
  if (threadIdx.x == 0)
    for (int l = 2; l >= 0; --l)
      if (p.F[l].staged == 1) issue_frame_tma(l);
  if ((int)warp < NM) {
    gn_init_warp((int)warp);
    if (!p.use_so3) gn_begin_warp(&sm.S[warp], 0, sm.nsched ? sm.sched[0] : 0);
  }
  __syncthreads();
  DBG_MARK(1);
  unsigned round = 0;
  if (p.use_so3) round = run_so3<GENERAL>();
  DBG_MARK(2);
  // ---- Gauss-Newton iterations, coarse to fine (RGBDOdometry.cpp:331-461)
  unsigned win_phase = 0;
  int q0 = 0;
  for (int lvl = 2; lvl >= 0; --lvl) {
    int nit = p.iters[lvl];
    if (q0 + nit > sm.nsched) nit = sm.nsched - q0;
    if (nit <= 0) continue;
    level_begin(lvl, win_phase);
    run_level<GENERAL, DBGT>(lvl, q0, nit, round);
    q0 += nit;
    round += nit;
  }
  // the kernels that follow on the stream (launched with the programmatic-dependency attribute, cfb_common.cuh) may
  // start launching now: they wait for this grid to complete before they touch anything
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // ---- CTA 0 publishes pose + stats of every model
  if (blockIdx.x == 0)
    for (int m = 0; m < NM; ++m) {
      const float* src = (const float*)&sm.S[m];
      float* dst = (float*)p.M[m].g;
      for (int i = threadIdx.x; i < (int)(sizeof(GNState) / 4); i += kT) dst[i] = src[i];
    }
  // pose, inverse, previous pose and fusion weight for the fuse / clean / predict kernels of this frame
  // (pose_math.cuh: the same expressions as the host's, bit for bit)
  if (blockIdx.x == 0 && (int)threadIdx.x < NM && p.M[threadIdx.x].pd) {
    pose_block_update(p.M[threadIdx.x].pd, sm.S[threadIdx.x].out_trans, sm.S[threadIdx.x].out_rot);
    // the statistics follow the block (Model::PoseReadback): the host fetches both with one copy
    *reinterpret_cast<TrackStats*>(p.M[threadIdx.x].pd + 1) = sm.S[threadIdx.x].stats;
  }
  DBG_MARK(3);
}

// sobel + candidate gates for all three levels in one launch; also clears the barrier words of the
// tracker launch that follows
struct PrepLevel {
  const unsigned char* img;
  const float* nextDepth;
  short *dx, *dy;
  unsigned char* cand;
  int w, h;
  float minScale;
  const float* vx;  // x plane of the model's global vertex map (extent of the valid vertices), with `box`
  int* box;         // 8 ints, preset to a large value, or null (camera model: no extents kept)
};
struct PrepParams {
  PrepLevel L[3];
  unsigned long long* sync_words;  // barrier A words (kMaxRounds x kMaxM) then the accumulator slots, or null
  int nacc;                        // accumulator words in use: kMaxRounds x nmodels x kXWords
};
constexpr size_t kSyncBytes = 8ull * (kMaxRounds * kMaxM + (size_t)kMaxRounds * kMaxM * kXWords * kXStride);  // barrier A + accumulator slots
__global__ void rgb_prepare_tiled_kernel(const PrepParams pp) {
  pdl_prologue();
  int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (pp.sync_words) {
    if (q < kMaxRounds * kMaxM) pp.sync_words[q] = 0ull;
    if (q < pp.nacc) pp.sync_words[kMaxRounds * kMaxM + (size_t)q * kXStride] = 0ull;
  }
#pragma unroll
  for (int l = 0; l < 3; ++l) {
    const PrepLevel& L = pp.L[l];
    const int n = L.w * L.h;
    if (q < n) {
      int y = q / L.w, x = q - y * L.w;
      rgb_prepare_pixel(L.img, L.w, L.h, L.nextDepth, L.minScale, L.dx, L.dy, L.cand, x, y);
      if (L.box) {  // extents [minx, miny, -maxx, -maxy]: candidates, valid vertices
        const bool cf = L.cand[q] != 0, vf = !isnan(__ldg(L.vx + q));
        const int big = 0x7f7f7f7f;
        if (__any_sync(__activemask(), cf || vf)) {
          const unsigned am = __activemask();
          int v[8] = {cf ? x : big, cf ? y : big, cf ? -x : big, cf ? -y : big, vf ? x : big, vf ? y : big, vf ? -x : big, vf ? -y : big};
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const int r = __reduce_min_sync(am, v[k]);
            if (r != big && (threadIdx.x & 31) == (__ffs(am) - 1)) atomicMin(L.box + k, r);
          }
        }
      }
      return;
    }
    q -= n;
  }
}

// ------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qr) == cudaSuccess &&
        qr == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)f;
    cudaGetLastError();
  }
  return fn;
}

// planar image of `planes` planes of w x h elements -> tensor map with box (bw, bh[, planes]); false when the
// image does not meet the TMA constraints (16-byte rows) or the driver refuses
bool encode_map(CUtensorMap* out, const void* base, CUtensorMapDataType dt, int esize, int w, int h, int planes, int bw, int bh) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  if (((size_t)w * esize) % 16 || ((size_t)bw * esize) % 16 || bw > 256 || bh > 256 || ((uintptr_t)base & 15)) return false;
  cuuint64_t gdim[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)planes};
  cuuint64_t gstr[2] = {(cuuint64_t)w * esize, (cuuint64_t)w * h * esize};
  cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)planes};
  cuuint32_t estr[3] = {1, 1, 1};
  const int rank = planes > 1 ? 3 : 2;
  return fn(out, dt, rank, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int round_up(int a, int b) { return (a + b - 1) / b * b; }
unsigned align128(unsigned a) { return (a + 127u) & ~127u; }
// row pitch of a box that covers `n` elements starting anywhere inside an `a`-element alignment unit
int box_pitch(int n, int a, bool origin_aligned) { return origin_aligned ? round_up(n, a) : round_up(n + a - 1, a); }

}  // namespace

#define RET_IF(e)                       \
  do {                                  \
    cudaError_t e__ = (e);              \
    if (e__ != cudaSuccess) return e__; \
  } while (0)

// Tile plan + tensor maps of one odometry object (fixed buffers: built once, on first use).
struct RGBDOdometry::TiledState {
  int gx = 1, gy = 1;
  FLevel F[3];          // plan part of the frame levels (pointers filled per launch)
  unsigned smem_bytes = 0;
  unsigned o_wrow = 0, o_blk = 0, o_out = 0, o_corr = 0;
  // device copies of the tensor maps: [level][which]; image / depth maps exist for both buffers they can name
  enum { TM_V, TM_N, TM_DX, TM_DY, TM_IMG_A, TM_IMG_B, TM_D1_NEXT, TM_D1_LAST, TM_CAND, TM_PV, TM_PN, TM_LD, TM_LI, TM_COUNT };
  CUtensorMap* d_maps = nullptr;  // [3][TM_COUNT]
  const unsigned char* img_a[3] = {nullptr, nullptr, nullptr};  // the buffer TM_IMG_A describes
  int attr_set = 0;  // bit v: the shared-memory attribute of kernel variant v is set
  int nmodels_planned = 0;
};

namespace {
// choose the tile grid and the shared-memory layout for `nm` models on `sms` CTAs
void plan_tiles(int W, int H, int sms, int nm, RGBDOdometry::TiledState& ts) {
  const int maxG = sms < 255 ? sms : 255;  // barrier A counts arrivals in 8 bits
  long best = -1;
  for (int gx = 1; gx <= maxG; ++gx) {
    const int gy = maxG / gx;
    const int tw = (W + gx - 1) / gx, th = (H + gy - 1) / gy;
    const int gxe = (W + tw - 1) / tw, gye = (H + th - 1) / th;  // tiles actually needed
    const long frame = (long)tw * th;
    const long win = (long)(tw + 2 * kMaxHalo + 3) * (th + 2 * kMaxHalo);
    long cost = frame * 4 + win;                 // pixel work dominates, the window only costs shared memory
    if (tw % 16) cost += frame / 4;              // unaligned f32 tiles at the coarser levels need wider boxes
    if (frame > kPP * kT) cost += 1000000L;      // level 0 would not fit a shared-memory tile
    if (best < 0 || cost < best) {
      best = cost;
      ts.gx = gxe;
      ts.gy = gye;
    }
  }
  unsigned off = align128((unsigned)sizeof(TFixed));
  ts.o_wrow = off;
  off = align128(off + 2u * kNW * 32 * 4);
  ts.o_blk = off;
  off = align128(off + (unsigned)nm * 64 * 4);
  ts.o_out = off;
  off = align128(off + (unsigned)nm * 64 * 8);
  ts.o_corr = off;
  off = align128(off + 2 * kPP * kT * 4);
  const unsigned cap = 227u * 1024u;
  auto window_bytes = [](const FLevel& F) {
    return align128(3u * F.wpf * F.wh * 4) * 2 + align128((unsigned)F.wpf * F.wh * 4) + align128((unsigned)F.wpb * F.wh);
  };
  const unsigned off0 = off;
  unsigned wmax = 0;
  for (int halo = kMaxHalo; halo >= 2; --halo) {  // shrink the window halo until the finest level fits too
    off = off0;
    wmax = 0;
    for (int l = 2; l >= 0; --l) {  // coarse to fine: frame tiles of every staged level + one window
      FLevel& F = ts.F[l];
      F.w = W >> l;
      F.h = H >> l;
      F.tw = (F.w + ts.gx - 1) / ts.gx;
      F.th = (F.h + ts.gy - 1) / ts.gy;
      F.npx = F.tw * F.th;
      F.pf = box_pitch(F.tw, 4, F.tw % 4 == 0);
      F.ps = box_pitch(F.tw, 8, F.tw % 8 == 0);
      F.pb = box_pitch(F.tw, 16, F.tw % 16 == 0);
      F.halo = halo;
      F.wwl = F.tw + 2 * halo;
      F.wh = F.th + 2 * halo;
      F.wpf = box_pitch(F.wwl, 4, false);
      F.wpb = box_pitch(F.wwl, 16, false);
      F.staged = 0;
      unsigned o = off;
      F.o_v = o;
      o = align128(o + 3u * F.pf * F.th * 4);
      F.o_n = o;
      o = align128(o + 3u * F.pf * F.th * 4);
      F.o_dx = o;
      o = align128(o + (unsigned)F.ps * F.th * 2);
      F.o_dy = o;
      o = align128(o + (unsigned)F.ps * F.th * 2);
      F.o_img = o;
      o = align128(o + (unsigned)F.pb * F.th);
      F.o_d1 = o;
      o = align128(o + (unsigned)F.pf * F.th * 4);
      F.o_cand = o;
      o = align128(o + (unsigned)F.pb * F.th);
      F.frame_bytes = 7u * F.pf * F.th * 4 + 2u * F.ps * F.th * 2 + 2u * F.pb * F.th;
      const unsigned wb = window_bytes(F), wnew = wb > wmax ? wb : wmax;
      if (!getenv("CFB_TILED_NOSTAGE") && F.npx <= kPP * kT && F.w < 2048 && F.h < 2048 && F.pf <= 256 && F.pb <= 256 &&
          F.th <= 256 && F.wpb <= 256 && F.wh <= 256 && o + wnew <= cap) {
        F.staged = 1;
        off = o;
        wmax = wnew;
      }  // a global-memory level keeps the same pixel enumeration: the pixel -> thread map, and with it the
         // summation order, does not depend on where a level's data lives
    }
    if (ts.F[0].staged || ts.F[0].npx > kPP * kT) break;  // level 0 staged, or it never can be
  }
  for (int l = 0; l < 3; ++l) {  // the window region is shared by the staged levels, after all frame tiles
    FLevel& F = ts.F[l];
    if (!F.staged) continue;
    unsigned o = off;
    F.o_pv = o;
    o += align128(3u * F.wpf * F.wh * 4);
    F.o_pn = o;
    o += align128(3u * F.wpf * F.wh * 4);
    F.o_ld = o;
    o += align128((unsigned)F.wpf * F.wh * 4);
    F.o_li = o;
    F.win_bytes = 7u * F.wpf * F.wh * 4 + (unsigned)F.wpb * F.wh;
  }
  ts.smem_bytes = off + wmax;
  ts.nmodels_planned = nm;
}
}  // namespace

void RGBDOdometry::destroyTiled() {
  if (tiled_) {
    cudaFree(tiled_->d_maps);
    delete tiled_;
    tiled_ = nullptr;
  }
}

// (re)build plan + tensor maps of this object for launches with `nm` models
cudaError_t RGBDOdometry::prepareTiled(int nm) {
  if (tiled_ && tiled_->nmodels_planned == nm) return cudaSuccess;
  destroyTiled();
  tiled_ = new TiledState();
  TiledState& ts = *tiled_;
  plan_tiles(width, height, num_sms(), nm, ts);
  RET_IF(cudaMalloc((void**)&ts.d_maps, sizeof(CUtensorMap) * 3 * TiledState::TM_COUNT));
  CUtensorMap h[3][TiledState::TM_COUNT];
  memset(h, 0, sizeof(h));
  for (int l = 0; l < 3; ++l) {
    FLevel& F = ts.F[l];
    if (!F.staged) continue;
    const int w = F.w, hh = F.h;
    bool ok = true;
    const CUtensorMapDataType f32 = CU_TENSOR_MAP_DATA_TYPE_FLOAT32, u16 = CU_TENSOR_MAP_DATA_TYPE_UINT16, u8 = CU_TENSOR_MAP_DATA_TYPE_UINT8;
    ok = ok && encode_map(&h[l][TiledState::TM_V], vmaps_curr_[l], f32, 4, w, hh, 3, F.pf, F.th);
    ok = ok && encode_map(&h[l][TiledState::TM_N], nmaps_curr_[l], f32, 4, w, hh, 3, F.pf, F.th);
    ok = ok && encode_map(&h[l][TiledState::TM_DX], nextdIdx[l], u16, 2, w, hh, 1, F.ps, F.th);
    ok = ok && encode_map(&h[l][TiledState::TM_DY], nextdIdy[l], u16, 2, w, hh, 1, F.ps, F.th);
    ok = ok && encode_map(&h[l][TiledState::TM_IMG_A], nextImage[l], u8, 1, w, hh, 1, F.pb, F.th);
    ok = ok && encode_map(&h[l][TiledState::TM_IMG_B], lastNextImage[l], u8, 1, w, hh, 1, F.pb, F.th);
    ok = ok && encode_map(&h[l][TiledState::TM_D1_NEXT], nextDepth[l], f32, 4, w, hh, 1, F.pf, F.th);
    ok = ok && encode_map(&h[l][TiledState::TM_D1_LAST], lastDepth[l], f32, 4, w, hh, 1, F.pf, F.th);
    ok = ok && encode_map(&h[l][TiledState::TM_CAND], rgbCand[l], u8, 1, w, hh, 1, F.pb, F.th);
    ok = ok && encode_map(&h[l][TiledState::TM_PV], vmaps_g_prev_[l], f32, 4, w, hh, 3, F.wpf, F.wh);
    ok = ok && encode_map(&h[l][TiledState::TM_PN], nmaps_g_prev_[l], f32, 4, w, hh, 3, F.wpf, F.wh);
    ok = ok && encode_map(&h[l][TiledState::TM_LD], lastDepth[l], f32, 4, w, hh, 1, F.wpf, F.wh);
    ok = ok && encode_map(&h[l][TiledState::TM_LI], lastImage[l], u8, 1, w, hh, 1, F.wpb, F.wh);
    if (getenv("CFB_TILED_NOTMA")) ok = false;  // debugging aid: fill the tiles with ordinary loads
    ts.img_a[l] = nextImage[l];
    F.staged = ok ? 1 : 2;
  }
  RET_IF(cudaMemcpy(ts.d_maps, h, sizeof(h), cudaMemcpyHostToDevice));
  if (getenv("CFB_TILED_DEBUG")) {
    fprintf(stderr, "[cfb tiled] %dx%d, %d models: grid %d x %d, %u bytes of shared memory\n", width, height, nm, ts.gx, ts.gy,
            ts.smem_bytes);
    for (int l = 0; l < 3; ++l)
      fprintf(stderr, "[cfb tiled]   level %d: %dx%d tile %dx%d (pitches %d/%d/%d) staged %d window %dx%d (pitches %d/%d) frame %u B window %u B\n",
              l, ts.F[l].w, ts.F[l].h, ts.F[l].tw, ts.F[l].th, ts.F[l].pf, ts.F[l].ps, ts.F[l].pb, ts.F[l].staged, ts.F[l].wwl,
              ts.F[l].wh, ts.F[l].wpf, ts.F[l].wpb, ts.F[l].staged ? ts.F[l].frame_bytes : 0u, ts.F[l].staged ? ts.F[l].win_bytes : 0u);
  }
  return cudaSuccess;
}

size_t RGBDOdometry::tiledScratchBytes() { return kSyncBytes + 256; }

bool RGBDOdometry::canBatch(int n) const { return n >= 1 && n <= kMaxM && width < 2048 && height < 2048; }

cudaError_t RGBDOdometry::enqueuePrepare(cudaStream_t s, void* sync_words, int nmodels, bool extents) {
  PrepParams pp;
  int total = 0;
  if (extents) {
    if (!d_box_) RET_IF(cudaMalloc((void**)&d_box_, 24 * sizeof(int)));
    RET_IF(cudaMemsetAsync(d_box_, 0x7f, 24 * sizeof(int), s));  // atomicMin targets
  }
  for (int i = 0; i < NUM_PYRS; ++i) {
    const int w = width >> i, h = height >> i;
    pp.L[i] = PrepLevel{nextImage[i], (next_is_last_ ? lastDepth[i] : nextDepth[i]), nextdIdx[i], nextdIdy[i], rgbCand[i], w, h,
                        (float)(pow(minimumGradientMagnitudes[i], 2.0) / pow(sobelScale, 2.0)), vmaps_g_prev_[i],
                        extents ? d_box_ + 8 * i : nullptr};
    total += w * h;
  }
  pp.sync_words = (unsigned long long*)sync_words;
  pp.nacc = kMaxRounds * nmodels * kXWords;
  CFB_PDL(launch_pdl(rgb_prepare_tiled_kernel, (total + 255) / 256, 256, 0, s, pp));
  return cudaGetLastError();
}

// All odometry objects belong to one frame (same geometry, same frame-side inputs, initAll() done on
// stream s); od[0] is the camera model whose tiles are staged.  trans / rot: n x 3 / n x 9 host arrays,
// in/out.  scratch: tiledScratchBytes() of zero-initialised device memory owned by the caller.
cudaError_t RGBDOdometry::trackTiled(RGBDOdometry* const* od, int n, float (*trans)[3], float (*rot)[9], float icpWeight,
                                     bool pyramid, bool fastOdom, bool so3, float* const* err, size_t err_pitch,
                                     void* scratch, cudaStream_t s, PoseDev* const* pd, bool async, bool prepared) {
  if (n < 1 || n > kMaxM || !scratch) return cudaErrorInvalidValue;
  if (async && !pd) return cudaErrorInvalidValue;  // without a host round trip the pose must live on the device
  struct Out {
    float trans[3];
    float rot[9];
    TrackStats st;
  };
  RGBDOdometry& f = *od[0];
  RET_IF(f.prepareTiled(n));
  TiledState& ts = *f.tiled_;
  TParams p;
  memset(&p, 0, sizeof(p));
  p.acnt = (unsigned long long*)scratch;
  p.xacc = p.acnt + kMaxRounds * kMaxM;
  for (int m = 0; m < n; ++m) {
    RGBDOdometry& o = *od[m];
    if (!(pd && pd[m])) {
      float* h_in = (float*)((char*)o.h_pinned + 1536);
      memcpy(h_in, trans[m], 3 * sizeof(float));
      memcpy(h_in + 3, rot[m], 9 * sizeof(float));
      RET_IF(cudaMemcpyAsync(o.d_pose_in, h_in, 12 * sizeof(float), cudaMemcpyHostToDevice, s));
    }
    // Sobel images + candidate gates of this model (a caller that spreads the models over streams has done it)
    if (!prepared) RET_IF(o.enqueuePrepare(s, m == 0 ? scratch : nullptr, n, m > 0));
    MParams& M = p.M[m];
    for (int i = 0; i < NUM_PYRS; ++i) {
      MLevel& L = M.L[i];
      L.vmap_g_prev = o.vmaps_g_prev_[i];
      L.nmap_g_prev = o.nmaps_g_prev_[i];
      L.lastDepth = o.lastDepth[i];
      L.nextDepth = o.next_is_last_ ? o.lastDepth[i] : o.nextDepth[i];
      L.lastImage = o.lastImage[i];
      L.cand = o.rgbCand[i];
      L.box = m > 0 ? o.d_box_ + 8 * i : nullptr;  // object models: see enqueuePrepare
      if (m == 0) {
        const CUtensorMap* tm = ts.d_maps + i * TiledState::TM_COUNT;
        L.tm_d1 = tm + (o.next_is_last_ ? TiledState::TM_D1_LAST : TiledState::TM_D1_NEXT);
        L.tm_cand = tm + TiledState::TM_CAND;
        L.tm_pv = tm + TiledState::TM_PV;
        L.tm_pn = tm + TiledState::TM_PN;
        L.tm_ld = tm + TiledState::TM_LD;
        L.tm_li = tm + TiledState::TM_LI;
      }
    }
    M.so3_last = o.lastNextImage[2];
    M.so3_next = o.nextImage[2];
    M.g = o.gn;
    M.pd = pd ? pd[m] : nullptr;
    M.pose_in = M.pd ? M.pd->tr : o.d_pose_in;
    M.err = err ? err[m] : nullptr;
    if (m > 0) {  // correspondences handed from phase 1 to phase 3 (phase1_obj)
      const size_t words = (size_t)kPP * ts.gx * ts.gy * kT;
      if (o.corr_words_ < words) {
        cudaFree(o.d_corr_);
        o.d_corr_ = nullptr;
        RET_IF(cudaMalloc(&o.d_corr_, words * 8));
        RET_IF(cudaMemsetAsync(o.d_corr_, 0, words * 8, s));
        o.corr_words_ = words;
      }
      M.corrZ = (unsigned*)o.d_corr_;
      M.corrD = (float*)o.d_corr_ + words;
    }
  }
  for (int i = 0; i < NUM_PYRS; ++i) {
    FLevel& F = p.F[i];
    F = ts.F[i];
    const Intr k = f.intr.level(i);
    F.vmap_curr = f.vmaps_curr_[i];
    F.nmap_curr = f.nmaps_curr_[i];
    F.nextImage = f.nextImage[i];
    F.dIdx = f.nextdIdx[i];
    F.dIdy = f.nextdIdy[i];
    F.k = LevelK{k.fx, k.fy, k.cx, k.cy};
    const CUtensorMap* tm = ts.d_maps + i * TiledState::TM_COUNT;
    F.tm_v = tm + TiledState::TM_V;
    F.tm_n = tm + TiledState::TM_N;
    F.tm_dx = tm + TiledState::TM_DX;
    F.tm_dy = tm + TiledState::TM_DY;
    F.tm_img = tm + (f.nextImage[i] == ts.img_a[i] ? TiledState::TM_IMG_A : TiledState::TM_IMG_B);
  }
  p.nmodels = n;
  p.gx = ts.gx;
  p.gy = ts.gy;
  p.err_pitch = err_pitch;
  p.distThres = f.distThres_;
  p.angleThres = f.angleThres_;
  p.maxDepthDelta = f.maxDepthDeltaRGB;
  p.sobelScale = f.sobelScale;
  p.icpWeight = icpWeight;
  p.use_so3 = so3 ? 1 : 0;
  p.iters[0] = fastOdom ? 3 : 10;
  p.iters[1] = pyramid ? 5 : 0;
  p.iters[2] = pyramid ? 4 : 0;
  p.o_wrow = ts.o_wrow;
  p.o_blk = ts.o_blk;
  p.o_out = ts.o_out;
  p.o_corr = ts.o_corr;
  p.dbg = (unsigned long long*)f.dbg_trace_;
  // four instantiations: lean (one model, every level staged) / general, each with and without the trace
  bool general = n > 1;
  for (int i = 0; i < NUM_PYRS; ++i) general = general || (p.iters[i] > 0 && ts.F[i].staged == 0);
  const int variant = (general ? 1 : 0) | (p.dbg ? 2 : 0);
  const void* kernels[4] = {(const void*)gn_tiled_kernel<false, false>, (const void*)gn_tiled_kernel<true, false>,
                            (const void*)gn_tiled_kernel<false, true>, (const void*)gn_tiled_kernel<true, true>};
  if (!(ts.attr_set & (1 << variant))) {
    // all four at once: setting the attribute also loads the kernel (lazy module loading), so the first frame with a
    // second model does not pay for loading the general instantiation
    for (int v = 0; v < 4; ++v)
      RET_IF(cudaFuncSetAttribute(kernels[v], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ts.smem_bytes));
    ts.attr_set = 15;
  }
  void* args[] = {(void*)&p};
  if (f.time_kernel_) RET_IF(cudaEventRecord(f.ev_k0_, s));
  // (a plain launch with the programmatic-dependency attribute instead of the cooperative one was measured: no gain)
  RET_IF(cudaLaunchCooperativeKernel(kernels[variant], dim3(ts.gx * ts.gy), dim3(kT), args, ts.smem_bytes, s));
  if (f.time_kernel_) {
    RET_IF(cudaEventRecord(f.ev_k1_, s));
    f.ev_pending_ = true;
  }
  auto swap_so3_images = [&](RGBDOdometry& o) {
    if (!so3) return;
    for (int i = 0; i < NUM_PYRS; i++) {
      unsigned char* t = o.lastNextImage[i];
      o.lastNextImage[i] = o.nextImage[i];
      o.nextImage[i] = t;
    }
  };
  if (async) {  // the caller reads pose / stats later (device pose block, statsDevice()); nothing to wait for
    for (int m = 0; m < n; ++m) swap_so3_images(*od[m]);
    return cudaSuccess;
  }
  for (int m = 0; m < n; ++m) {
    RGBDOdometry& o = *od[m];
    Out* ho = (Out*)((char*)o.h_pinned + 2048);
    RET_IF(cudaMemcpyAsync(ho->trans, o.gn->out_trans, 12 * sizeof(float), cudaMemcpyDeviceToHost, s));
    RET_IF(cudaMemcpyAsync(&ho->st, &o.gn->stats, sizeof(TrackStats), cudaMemcpyDeviceToHost, s));
  }
  RET_IF(cudaStreamSynchronize(s));
  if (f.time_kernel_) f.kernelTiming(nullptr, nullptr, false);
  for (int m = 0; m < n; ++m) {
    RGBDOdometry& o = *od[m];
    Out* ho = (Out*)((char*)o.h_pinned + 2048);
    memcpy(trans[m], ho->trans, sizeof(float) * 3);
    memcpy(rot[m], ho->rot, sizeof(float) * 9);
    o.stats_ = ho->st;
    swap_so3_images(o);
  }
  return cudaSuccess;
}

void RGBDOdometry::enableKernelTiming(bool on) {
  if (on && !ev_k0_) {
    cudaEventCreate(&ev_k0_);
    cudaEventCreate(&ev_k1_);
  }
  time_kernel_ = on && ev_k0_ && ev_k1_;
}

void RGBDOdometry::kernelTiming(double* sum_ms, int* launches, bool reset) {
  if (ev_pending_ && cudaEventSynchronize(ev_k1_) == cudaSuccess) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ev_k0_, ev_k1_) == cudaSuccess) {
      kernel_ms_sum_ += ms;
      kernel_launches_++;
    }
    ev_pending_ = false;
  }
  if (sum_ms) *sum_ms = kernel_ms_sum_;
  if (launches) *launches = kernel_launches_;
  if (reset) {
    kernel_ms_sum_ = 0;
    kernel_launches_ = 0;
  }
}

}  // namespace cfb
