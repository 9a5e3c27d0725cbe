// Shared device/host declarations of the pcop CUDA library (sm_100a only).
//
// Layout in HBM ("wave" = the frames processed by one set of launches):
//   every per-point array is frame-strided: frame f owns [f*cap, (f+1)*cap), cap = max points
//   per frame; every per-frame scalar is an int32/uint32 array of B entries that lives on the
//   device, so no stage needs a host round-trip to learn the previous stage's count.
//   A point is a float4 {x,y,z,w} (pcl::PointXYZ), one 16-byte vector load.
//
// All float arithmetic that feeds an integer decision uses the __f*_rn intrinsics (never
// contracted into FMA) in the operation order written in oracle/pcop_oracle.cpp's
// specification comments; the library is also compiled with -fmad=false.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pcop.h"

namespace pcop {

constexpr unsigned FULL = 0xffffffffu;

// ---- tiles -----------------------------------------------------------------
constexpr int CT_THREADS = 256;  // stream-compaction / per-point kernels
constexpr int CT_ITEMS = 4;
constexpr int CT_TILE = CT_THREADS * CT_ITEMS;  // 1024 points
constexpr int BT_ITEMS = 16;                     // big-tile compactions (crop, voxel heads, plane extract)
constexpr int BT_TILE = CT_THREADS * BT_ITEMS;   // 4096 points
constexpr int RS_THREADS = 256;  // radix sort
constexpr int RS_ITEMS = 8;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;  // 2048 keys
constexpr int RS_RADIX_BITS = 8;
constexpr int RS_BINS = 1 << RS_RADIX_BITS;
constexpr int RS_MAX_PASSES = 4;
constexpr int TS_CHUNK = 2048;  // canonical tree-sum chunk (oracle "CT2048")
constexpr int MAX_HYP = PCOP_MAX_HYPOTHESES;
constexpr int RNG_TABLE = 4096;  // rnd() values precomputed per handle

__host__ __device__ inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// ---- deterministic float helpers --------------------------------------------
__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }

// squared distance in FLANN L2_Simple order: ((dx*dx)+(dy*dy))+(dz*dz)
__device__ __forceinline__ float dist2(float ax, float ay, float az, float bx, float by, float bz) {
  const float dx = fsub(ax, bx), dy = fsub(ay, by), dz = fsub(az, bz);
  return fadd(fadd(fmul(dx, dx), fmul(dy, dy)), fmul(dz, dz));
}

// |((a*x + b*y) + (c*z + d))|
__device__ __forceinline__ float plane_dist(const float4 co, float x, float y, float z) {
  return fabsf(fadd(fadd(fmul(co.x, x), fmul(co.y, y)), fadd(fmul(co.z, z), co.w)));
}

// static_cast<int>(float) with x86 cvttss2si semantics (NaN / out of range -> INT_MIN)
__device__ __forceinline__ int cvt_f2i(float v) {
  if (v != v || v >= 2147483648.0f || v < -2147483648.0f) return (int)0x80000000;
  return __float2int_rz(v);
}
__device__ __forceinline__ long long cvt_f2l(float v) {
  if (v != v || v >= 9223372036854775808.0f || v < -9223372036854775808.0f) return (long long)0x8000000000000000ull;
  return __float2ll_rz(v);
}

// order-preserving float <-> uint mapping for atomicMin/atomicMax
__device__ __forceinline__ unsigned f2ord(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
constexpr unsigned ORD_POS_FLT_MAX = 0xff7fffffu;  // f2ord(+FLT_MAX)
constexpr unsigned ORD_NEG_FLT_MAX = 0x00800000u;  // f2ord(-FLT_MAX)

// ---- per-frame records --------------------------------------------------------
struct MinMax {  // ordered-uint encoded
  unsigned mn[3], mx[3];
};

struct VoxelFrame {
  float inv;
  int min_b[3];
  unsigned mul1, mul2;
  int overflow;
};

struct EceFrame {
  float mn[3];
  float inv[3];
  int dim[3];
  int mode;  // 0: clique cells (edge < tol/sqrt(3)), union-find over cells; 1: cells >= tol, per-point neighbour scan
};

struct PlaneFrame {  // state of the plane loop of one frame
  int active;        // still looping
  int cur;           // which ping-pong buffer holds the current cloud
  int nr_points;     // size when the loop started (od.cpp:376)
  int n;             // current size
  int n_passes;
  int n_hyp;         // hypotheses generated this pass
  int gen_end;       // generator stopped early: 0 no, 1 empty sample / skip limit, 2 rng table exhausted
  int n_inliers_last;
  double log_prob;   // det_log(1 - probability), evaluated once per frame
  float4 coeff_sel;  // RANSAC winner
  float4 coeff_ref;  // after refinement
  float4 hyp[MAX_HYP];
  int hyp_valid[MAX_HYP];  // isModelValid
  int pass_points[PCOP_MAX_PLANE_PASSES_RECORDED];
  int pass_inliers[PCOP_MAX_PLANE_PASSES_RECORDED];
  float4 pass_coeff[PCOP_MAX_PLANE_PASSES_RECORDED];
};

struct PlaneConst {
  float thr;
  double eps_angle, cos_eps;
  double axis[3];
  double keep_fraction;
  int max_iterations;
  double log_probability;  // det_log(1 - probability), evaluated on the device side spec
  double probability;
  int optimize;
};

// host-visible error helper
#define PCOP_CUDA_TRY(expr)                                                     \
  do {                                                                          \
    cudaError_t _e = (expr);                                                    \
    if (_e != cudaSuccess) return ::pcop::fail_cuda(h, _e, #expr, __FILE__, __LINE__); \
  } while (0)

}  // namespace pcop
