// RANSAC plane-removal loop (reference: segment_plane_and_extract_indices od.cpp:342-428 ->
// pcl::SACSegmentation<SACMODEL_PERPENDICULAR_PLANE, SAC_RANSAC> + pcl::ExtractIndices,
// SURVEY 8a-4).
//
// PCL draws samples sequentially but the draws never depend on the scores, so per pass and per
// frame: (1) one warp replays boost::mt19937(12345) + the persistent index shuffle sparsely and
// emits all <= 51 hypotheses; (2) one sweep over the points scores every hypothesis (warp
// ballots -> integer counts); (3) one thread replays PCL's adaptive-k loop over the counts;
// (4) the nine inlier moments are accumulated in double in the canonical tree order;
// (5) one thread runs PCL's closed-form eigen33 and validates the refined model; (6) a stable
// compaction removes the refined inliers; (7) the while(size > 0.3*nr) rule is evaluated per
// frame.  Frames of a wave run their passes in lock-step; finished frames idle.
#include "det_math.cuh"
#include <cstdio>
#include "internal.cuh"
#include "primitives.cuh"

namespace pcop {
#ifdef PCOP_PLANE_DEBUG_CLK
__device__ long long g_plane_loop_clk[16];  // phase timestamps of frame 0 / CTA 0 (tools/plane_phases.py)
#define PL_CLK(k)                                                                  \
  do {                                                                             \
    if (blockIdx.y == 0 && rank == 0 && threadIdx.x == 0) g_plane_loop_clk[k] = clock64(); \
  } while (0)
#else
#define PL_CLK(k) \
  do {            \
  } while (0)
#endif

namespace {

constexpr int MAP_CAP = RNG_TABLE + 8;
constexpr double kHalfPi = 1.57079632679489661923;

struct BufPair {
  float4* p[2];
  int* s[2];
};

__device__ bool model_valid(const PlaneConst& pc, const float4 co) {
  if (!(pc.eps_angle > 0.0)) return true;
  if (pc.eps_angle >= kHalfPi) return true;
  const double nx = co.x, ny = co.y, nz = co.z;
  const double dot = dadd(dadd(dmul(nx, pc.axis[0]), dmul(ny, pc.axis[1])), dmul(nz, pc.axis[2]));
  const double nn = __dsqrt_rn(dadd(dadd(dmul(nx, nx), dmul(ny, ny)), dmul(nz, nz)));
  const double na = __dsqrt_rn(dadd(dadd(dmul(pc.axis[0], pc.axis[0]), dmul(pc.axis[1], pc.axis[1])),
                                    dmul(pc.axis[2], pc.axis[2])));
  const double cosang = ddiv(fabs(dot), dmul(nn, na));
  return !(cosang < pc.cos_eps);
}

__device__ __forceinline__ bool collinear_ratio_test(const float4 p0, const float4 p1, const float4 p2) {
  const float ax = fdiv(fsub(p1.x, p0.x), fsub(p2.x, p0.x));
  const float ay = fdiv(fsub(p1.y, p0.y), fsub(p2.y, p0.y));
  const float az = fdiv(fsub(p1.z, p0.z), fsub(p2.z, p0.z));
  return (ax == ay) && (az == ay);
}

__device__ float4 compute_model(const float4 p0, const float4 p1, const float4 p2) {
  const float ax = fsub(p1.x, p0.x), ay = fsub(p1.y, p0.y), az = fsub(p1.z, p0.z);
  const float bx = fsub(p2.x, p0.x), by = fsub(p2.y, p0.y), bz = fsub(p2.z, p0.z);
  float nx = fsub(fmul(ay, bz), fmul(az, by));
  float ny = fsub(fmul(az, bx), fmul(ax, bz));
  float nz = fsub(fmul(ax, by), fmul(ay, bx));
  const float norm = __fsqrt_rn(fadd(fadd(fmul(nx, nx), fmul(ny, ny)), fmul(nz, nz)));
  nx = fdiv(nx, norm);
  ny = fdiv(ny, norm);
  nz = fdiv(nz, norm);
  const float d = -fadd(fadd(fmul(nx, p0.x), fmul(ny, p0.y)), fmul(nz, p0.z));
  return make_float4(nx, ny, nz, d);
}

// Scratch of the hypothesis generator (one warp).  The frame-resident loop kernel overlays it on its point slices.
struct GenScratch {
  int mpos[MAP_CAP];
  int mval[MAP_CAP];
  int trip[MAX_HYP][3];
  int srng[3 * MAX_HYP];  // the random numbers of the fast path, fetched by all lanes at once
  int sq[3 * MAX_HYP], sA[3 * MAX_HYP], sT[3 * MAX_HYP];
  int sLq[3 * MAX_HYP];
};

// one warp: hypothesis generation (getSamples/drawIndexSample/isSampleGood/computeModelCoefficients) for a cloud
// of n points.  shuffled_indices_ is simulated sparsely: positions 0..2 live in registers, every other touched
// position in a (pos,val) list searched by the 32 lanes.  Writes hyp[0..nh) / hyp_valid[0..nh) (any memory space the
// warp can write); the points are read with ld.global.cg (the loop kernel reads clouds that other CTAs of the cluster
// wrote during the same launch, so no L1 line may be trusted); returns nh and gen_end (0 no early stop, 1 empty sample / skip limit, 2 rng table exhausted) in
// every lane.
__device__ __forceinline__ void plane_gen_warp(const float4* __restrict__ pts, const int n, const int* __restrict__ rng,
                                               const PlaneConst& pc, GenScratch& G, float4* hyp, int* hyp_valid, int& nh_out,
                                               int& gen_end_out) {
  const int lane = threadIdx.x & 31;
  int* mpos = G.mpos;
  int* mval = G.mval;
  int ne = 0;
  int s[3] = {0, 1, 2};
  int t = 0;
  int nh = 0;
  int gen_end = 0;
  // Fast path: the draws never depend on the points unless a sample fails isSampleGood (collinear, rare).  So first
  // replay the index draws of all hypotheses assuming every first draw is good (no memory traffic), then let the
  // lanes fetch and fit the hypotheses in parallel; one bad sample sends the frame through the sequential replay
  // below, which is PCL's loop verbatim.
  int(*trip)[3] = G.trip;
  bool fast_done = false;
  const int want = min(pc.max_iterations + 1, MAX_HYP);
  if (n >= 3 && 3 * want <= RNG_TABLE && 3 * want <= MAP_CAP) {
    // Draw replay in O(1) per draw (no search list).  Step j (i = j % 3) swaps shuf[i] with shuf[q_j],
    // q_j = i + rnd_j % (n - i).  A_j / T_j = values at positions i / q_j before the step; afterwards position i
    // holds T_j and position q_j holds A_j, and sample h = (T_3h, T_3h+1, T_3h+2).  The value at a position is what
    // its latest earlier writer left there: positions 0..2 are rewritten every three steps (so only steps j-1..j-3
    // matter), a position >= 3 only by an earlier step with the same target (Lq, found by all lanes in parallel).
    int* srng = G.srng;
    int *sq = G.sq, *sA = G.sA, *sT = G.sT, *sLq = G.sLq;
    const int J = 3 * want;
    for (int k = lane; k < J; k += 32) {
      srng[k] = rng[k];
      const int i = k % 3;
      sq[k] = i + (int)((unsigned)srng[k] % (unsigned)(n - i));
    }
    __syncwarp();
    // Lq[j] = latest k < j with the same target.  Lane l owns the steps k = l, l+32, ... (their targets in registers);
    // per j one broadcast load, a few register compares and, on the rare match, a warp max.
    int myq[(3 * MAX_HYP + 31) / 32];
#pragma unroll
    for (int c = 0; c < (3 * MAX_HYP + 31) / 32; ++c) myq[c] = (lane + 32 * c < J) ? sq[lane + 32 * c] : -1;
    for (int j = 0; j < J; ++j) {
      const int qj = sq[j];
      int best = -1;
#pragma unroll
      for (int c = 0; c < (3 * MAX_HYP + 31) / 32; ++c) {
        const int k = lane + 32 * c;
        if (k < j && myq[c] == qj) best = k;
      }
      int lq = -1;
      if (__any_sync(FULL, best >= 0)) lq = __reduce_max_sync(FULL, best);
      if (lane == 0) sLq[j] = lq;
    }
    __syncwarp();
    if (lane == 0) {
      // one hypothesis (three steps, slots 0, 1, 2) per iteration: the six shared-memory loads are issued up front, the
      // values of the last three steps stay in registers; shared memory is only read again for a repeated target
      int a1 = 0, a2 = 0, t3 = 0, t2 = 0, t1 = 0;  // A_{j-1}, A_{j-2}, T_{j-3}, T_{j-2}, T_{j-1}
      int q1 = -1, q2 = -1, q3 = -1;              // q_{j-1}, q_{j-2}, q_{j-3}
      for (int j0 = 0; j0 < J; j0 += 3) {
        const int qs[3] = {sq[j0], sq[j0 + 1], sq[j0 + 2]};
        const int ls[3] = {sLq[j0], sLq[j0 + 1], sLq[j0 + 2]};
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int j = j0 + i, qj = qs[i], lq = ls[i];
          int a;
          if (j >= 1 && q1 == i) a = a1;
          else if (j >= 2 && q2 == i) a = a2;
          else if (j >= 3) a = t3;
          else a = i;
          int tt;
          if (qj == i) {
            tt = a;
          } else if (qj < 3) {
            // position qj in 1..2 (> i): its latest writer among steps j-1, j-2, j-3 (slots i1, i2, i3 = i)
            tt = qj;
            const int i1 = (i + 2) % 3, i2 = (i + 1) % 3;
            if (j >= 1 && q1 == qj && i1 != qj) tt = a1;
            else if (j >= 1 && i1 == qj) tt = t1;
            else if (j >= 2 && q2 == qj && i2 != qj) tt = a2;
            else if (j >= 2 && i2 == qj) tt = t2;
            else if (j >= 3 && q3 == qj) tt = sA[j - 3];
          } else {
            tt = (lq >= 0) ? sA[lq] : qj;
          }
          sA[j] = a;
          sT[j] = tt;
          a2 = a1;
          a1 = a;
          t3 = t2;
          t2 = t1;
          t1 = tt;
          q3 = q2;
          q2 = q1;
          q1 = qj;
        }
      }
    }
    __syncwarp();
    for (int k = lane; k < J; k += 32) trip[k / 3][k % 3] = sT[k];
    t = J;
    __syncwarp();
    bool bad = false;
    for (int h = lane; h < want; h += 32) {
      const float4 p0 = __ldcg(pts + trip[h][0]), p1 = __ldcg(pts + trip[h][1]), p2 = __ldcg(pts + trip[h][2]);
      if (collinear_ratio_test(p0, p1, p2)) {
        bad = true;
      } else {
        const float4 co = compute_model(p0, p1, p2);
        hyp[h] = co;
        hyp_valid[h] = model_valid(pc, co) ? 1 : 0;
      }
    }
    if (!__any_sync(FULL, bad)) {
      fast_done = true;
      nh = want;
    } else {  // restart from PCL's initial state
      ne = 0;
      s[0] = 0;
      s[1] = 1;
      s[2] = 2;
      t = 0;
    }
    __syncwarp();
  }
  if (fast_done) {
    // nothing left to do
  } else if (n < 3) {
    gen_end = 1;  // getSamples: fewer points than the sample size -> empty selection
  } else {
    while (nh <= pc.max_iterations && nh < MAX_HYP) {
      bool good = false;
      float4 p0, p1, p2;
      for (int check = 0; check < 1000; ++check) {
        if (t + 3 > RNG_TABLE) {
          gen_end = 2;
          break;
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int r = rng[t++];
          const int j = i + (int)((unsigned)r % (unsigned)(n - i));
          const int vi = s[i];
          if (j < 3) {
            // j >= i always; swap two register slots
            const int vj = (j == 0) ? s[0] : ((j == 1) ? s[1] : s[2]);
            if (j == 0) s[0] = vi;
            else if (j == 1) s[1] = vi;
            else s[2] = vi;
            s[i] = vj;
          } else {
            int found = -1;
            for (int e = lane; e < ne; e += 32)
              if (mpos[e] == j) found = e;
            const unsigned b = __ballot_sync(FULL, found >= 0);
            int vj = j;
            if (b) {
              const int idx = __shfl_sync(FULL, found, __ffs(b) - 1);
              vj = mval[idx];
              __syncwarp();
              if (lane == 0) mval[idx] = vi;
            } else {
              if (lane == 0) {
                mpos[ne] = j;
                mval[ne] = vi;
              }
              ++ne;
            }
            __syncwarp();
            s[i] = vj;
          }
        }
        p0 = __ldcg(pts + s[0]);
        p1 = __ldcg(pts + s[1]);
        p2 = __ldcg(pts + s[2]);
        if (!collinear_ratio_test(p0, p1, p2)) {  // isSampleGood
          good = true;
          break;
        }
      }
      if (!good) {
        if (!gen_end) gen_end = 1;
        break;
      }
      // computeModelCoefficients repeats the same collinearity test, so it cannot fail here
      const float4 co = compute_model(p0, p1, p2);
      if (lane == 0) {
        hyp[nh] = co;
        hyp_valid[nh] = model_valid(pc, co) ? 1 : 0;
      }
      ++nh;
    }
  }
  __syncwarp();
  nh_out = nh;
  gen_end_out = gen_end;
}

// RandomSampleConsensus::computeModel's loop, replayed over the precomputed counts.
// `navail` hypotheses have been scored so far: if the loop asks for a later one it returns true ("need more") and
// decides nothing (the remaining hypotheses are scored, then this runs again).  count(h) = inliers of hypothesis h.
template <class CountFn>
__device__ __forceinline__ bool plane_select_replay(const PlaneConst& pc, double log_probability, int n, int nh, int navail,
                                                    const int* hyp_valid, CountFn count, int& sel_out) {
  const double one_over_indices = ddiv(1.0, (double)n);
  const double eps = 2.220446049250313e-16;
  int best = -2147483647;
  int sel = -1;
  double k = 1.0;
  for (int h = 0; h < nh; ++h) {
    if (!((double)h < k)) break;
    if (h >= navail) return true;
    const int c = hyp_valid[h] ? count(h) : 0;
    if (c > best) {
      best = c;
      sel = h;
      const double w = dmul((double)best, one_over_indices);
      double p_no = dsub(1.0, dmul(dmul(w, w), w));
      p_no = (eps < p_no) ? p_no : eps;
      p_no = (p_no < dsub(1.0, eps)) ? p_no : dsub(1.0, eps);
      k = ddiv(log_probability, det_log(p_no));
    }
    if (h + 1 > pc.max_iterations) break;
  }
  sel_out = sel;
  return false;
}

__device__ void compute_roots2(double b, double c, double* r) {
  r[0] = 0.0;
  double d = dsub(dmul(b, b), dmul(4.0, c));
  if (d < 0.0) d = 0.0;
  const double sd = __dsqrt_rn(d);
  r[2] = dmul(0.5, dadd(b, sd));
  r[1] = dmul(0.5, dsub(b, sd));
}

__device__ void compute_roots(const double* m, double* r) {
  const double m00 = m[0], m01 = m[1], m02 = m[2], m11 = m[4], m12 = m[5], m22 = m[8];
  double c0 = dmul(dmul(m00, m11), m22);
  c0 = dadd(c0, dmul(dmul(dmul(2.0, m01), m02), m12));
  c0 = dsub(c0, dmul(dmul(m00, m12), m12));
  c0 = dsub(c0, dmul(dmul(m11, m02), m02));
  c0 = dsub(c0, dmul(dmul(m22, m01), m01));
  double c1 = dsub(dmul(m00, m11), dmul(m01, m01));
  c1 = dadd(c1, dmul(m00, m22));
  c1 = dsub(c1, dmul(m02, m02));
  c1 = dadd(c1, dmul(m11, m22));
  c1 = dsub(c1, dmul(m12, m12));
  const double c2 = dadd(dadd(m00, m11), m22);
  if (fabs(c0) < 2.220446049250313e-16) {
    compute_roots2(c2, c1, r);
    return;
  }
  const double s_inv3 = ddiv(1.0, 3.0);
  const double s_sqrt3 = __dsqrt_rn(3.0);
  const double c2_over_3 = dmul(c2, s_inv3);
  double a_over_3 = dmul(dsub(c1, dmul(c2, c2_over_3)), s_inv3);
  if (a_over_3 > 0.0) a_over_3 = 0.0;
  const double half_b =
      dmul(0.5, dadd(c0, dmul(c2_over_3, dsub(dmul(dmul(2.0, c2_over_3), c2_over_3), c1))));
  double q = dadd(dmul(half_b, half_b), dmul(dmul(a_over_3, a_over_3), a_over_3));
  if (q > 0.0) q = 0.0;
  const double rho = __dsqrt_rn(-a_over_3);
  const double theta = dmul(det_atan2_ypos(__dsqrt_rn(-q), half_b), s_inv3);
  const double cos_theta = det_cos(theta);
  const double sin_theta = det_sin(theta);
  r[0] = dadd(c2_over_3, dmul(dmul(2.0, rho), cos_theta));
  r[1] = dsub(c2_over_3, dmul(rho, dadd(cos_theta, dmul(s_sqrt3, sin_theta))));
  r[2] = dsub(c2_over_3, dmul(rho, dsub(cos_theta, dmul(s_sqrt3, sin_theta))));
  double t;
  if (r[0] >= r[1]) {
    t = r[0];
    r[0] = r[1];
    r[1] = t;
  }
  if (r[1] >= r[2]) {
    t = r[1];
    r[1] = r[2];
    r[2] = t;
    if (r[0] >= r[1]) {
      t = r[0];
      r[0] = r[1];
      r[1] = t;
    }
  }
  if (r[0] <= 0.0) compute_roots2(c2, c1, r);
}

__device__ __forceinline__ void cross3(const double* a, const double* b, double* o) {
  o[0] = dsub(dmul(a[1], b[2]), dmul(a[2], b[1]));
  o[1] = dsub(dmul(a[2], b[0]), dmul(a[0], b[2]));
  o[2] = dsub(dmul(a[0], b[1]), dmul(a[1], b[0]));
}

__device__ void eigen33_smallest(const double* mat, double* evec) {
  double scale = 0.0;
  for (int i = 0; i < 9; ++i) scale = fabs(mat[i]) > scale ? fabs(mat[i]) : scale;
  if (scale <= 2.2250738585072014e-308) scale = 1.0;
  double sm[9];
  for (int i = 0; i < 9; ++i) sm[i] = ddiv(mat[i], scale);
  double r[3];
  compute_roots(sm, r);
  sm[0] = dsub(sm[0], r[0]);
  sm[4] = dsub(sm[4], r[0]);
  sm[8] = dsub(sm[8], r[0]);
  double v1[3], v2[3], v3[3];
  cross3(&sm[0], &sm[3], v1);
  cross3(&sm[0], &sm[6], v2);
  cross3(&sm[3], &sm[6], v3);
  const double l1 = dadd(dadd(dmul(v1[0], v1[0]), dmul(v1[1], v1[1])), dmul(v1[2], v1[2]));
  const double l2 = dadd(dadd(dmul(v2[0], v2[0]), dmul(v2[1], v2[1])), dmul(v2[2], v2[2]));
  const double l3 = dadd(dadd(dmul(v3[0], v3[0]), dmul(v3[1], v3[1])), dmul(v3[2], v3[2]));
  const double* v;
  double l;
  if (l1 >= l2 && l1 >= l3) {
    v = v1;
    l = l1;
  } else if (l2 >= l1 && l2 >= l3) {
    v = v2;
    l = l2;
  } else {
    v = v3;
    l = l3;
  }
  const double s = __dsqrt_rn(l);
  evec[0] = ddiv(v[0], s);
  evec[1] = ddiv(v[1], s);
  evec[2] = ddiv(v[2], s);
}

// optimizeModelCoefficients from the nine summed moments (xx, xy, xz, yy, yz, zz, x, y, z) and the inlier count:
// eigen33, validity check.  Returns true (and the refined model in `out`) when the model is replaced.
__device__ bool plane_refine_model(const PlaneConst& pc, const double* sums, double cntd, float4& out) {
  if (cntd < 4.0) return false;  // fewer than 4 inliers: keep the RANSAC model
  double a[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) a[k] = ddiv(sums[k], cntd);
  double cov[9];
  cov[0] = dsub(a[0], dmul(a[6], a[6]));
  cov[1] = dsub(a[1], dmul(a[6], a[7]));
  cov[2] = dsub(a[2], dmul(a[6], a[8]));
  cov[4] = dsub(a[3], dmul(a[7], a[7]));
  cov[5] = dsub(a[4], dmul(a[7], a[8]));
  cov[8] = dsub(a[5], dmul(a[8], a[8]));
  cov[3] = cov[1];
  cov[6] = cov[2];
  cov[7] = cov[5];
  double vec[3];
  eigen33_smallest(cov, vec);
  float4 o;
  o.x = (float)vec[0];
  o.y = (float)vec[1];
  o.z = (float)vec[2];
  const float cx = (float)a[6], cy = (float)a[7], cz = (float)a[8];
  o.w = -fadd(fadd(fmul(o.x, cx), fmul(o.y, cy)), fmul(o.z, cz));
  if (!model_valid(pc, o)) return false;
  out = o;
  return true;
}


// =====================================================================================================================
// Frame-resident plane loop: ONE thread-block cluster per frame runs every pass of od.cpp:376-399 without the host.
//
//   k_plane_gen0   (one warp per frame) initialises the frame's loop state and generates the hypotheses of pass 0;
//   k_plane_loop   (cluster of PL_CL CTAs per frame): every CTA keeps a contiguous slice of the current cloud in its
//                  shared memory (x, y, z planes), so one pass reads the cloud from HBM once: score the first 8
//                  hypotheses -> replay the adaptive-k loop -> [score the rest] -> CT2048 moments -> eigen33 refinement ->
//                  stable extraction -> while (size > 0.3 * nr).  The CTAs exchange only counts and chunk partials,
//                  pushed into every peer's shared memory (DSMEM) in front of a cluster barrier; every CTA then takes
//                  the (deterministic) decisions redundantly, which saves the broadcast barrier.  The pass that ends the
//                  loop writes the remaining cloud straight into the stage output (no finalize copy); a frame that
//                  needs another pass generates its hypotheses in-kernel and reloads its slices from L2.
// Frames above 8 slices take the windowed instantiation: a CTA whose part of the frame is longer than its slice reloads
// it in windows (see k_plane_loop); the chunk sums and the compaction order do not depend on the window size.
constexpr int PL_CL = 8;
constexpr int PL_MAX_THREADS = 1024;
constexpr int PL_MAX_WARPS = PL_MAX_THREADS / 32;
constexpr int PL_MAX_GROUPS = PL_MAX_THREADS / 256;  // 256-thread groups, one CT2048 chunk at a time each
// Hypotheses are scored in batches: the adaptive-k replay of a frame whose first hypotheses already hold the dominant
// plane stops after k = log(0.01) / log(1 - w^3) of them (3.5 for an inlier ratio w = 0.9), so most frames are
// decided by the first four
constexpr int PL_N_BATCHES = 3;
__constant__ const int PL_BATCH_END[PL_N_BATCHES] = {4, 8, MAX_HYP};

struct PlShared {
  float4 hyp[MAX_HYP];
  int hyp_valid[MAX_HYP];
  int cnt[MAX_HYP];              // this CTA's inlier counts
  int cnt_all[PL_CL][MAX_HYP];   // every CTA's counts (pushed by the peers)
  int kept_all[PL_CL];           // every CTA's kept-point total of the extraction
  int warp_excl[PL_MAX_WARPS];
  double msh[PL_MAX_GROUPS][8][9];   // per-warp moment sums of the chunk in flight
  int mcnt[PL_MAX_GROUPS][8];
  double log_prob;  // det_log(1 - probability), from k_plane_gen0
  float4 coeff_sel, coeff_ref;
  int model_ok, need_more, nh, gen_end;
};

// barrier 1 + g for the 256 threads of group g (immediate ids, so that ptxas reserves only the barriers in use:
// the barrier file is shared by the CTAs resident on an SM)
template <int GROUPS>
__device__ __forceinline__ void group_bar_sync(int g) {
  if (g == 0) asm volatile("bar.sync 1, 256;" ::: "memory");
  else if (g == 1) asm volatile("bar.sync 2, 256;" ::: "memory");
  else if (GROUPS > 2 && g == 2) asm volatile("bar.sync 3, 256;" ::: "memory");
  else if (GROUPS > 2) asm volatile("bar.sync 4, 256;" ::: "memory");
}
__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of `p` (a generic pointer into this CTA's shared memory) in CTA `rank` of the cluster
template <class T>
__device__ __forceinline__ T* dsmem_ptr(T* p, unsigned rank) {
  unsigned long long out;
  asm volatile("mapa.u64 %0, %1, %2;" : "=l"(out) : "l"((unsigned long long)p), "r"(rank));
  return reinterpret_cast<T*>(out);
}

__global__ void __launch_bounds__(32)
    k_plane_gen0(PlaneFrame* __restrict__ pf, const float4* __restrict__ in, size_t in_stride, const int* __restrict__ n_in,
                 int* __restrict__ n_in_copy, const int* __restrict__ rng, PlaneConst pc, uint32_t* __restrict__ warnings) {
  const int f = blockIdx.x;
  const int lane = threadIdx.x;
  PlaneFrame& P = pf[f];
  const int n = n_in[f];
  const int active = ((double)n > dmul(pc.keep_fraction, (double)n)) ? 1 : 0;  // od.cpp:379
  if (lane == 0) {
    if (n_in_copy) n_in_copy[f] = n;
    P.cur = -1;
    P.nr_points = n;
    P.n = n;
    P.n_passes = 0;
    P.n_inliers_last = 0;
    P.coeff_sel = make_float4(0.f, 0.f, 0.f, 0.f);
    P.coeff_ref = make_float4(0.f, 0.f, 0.f, 0.f);
    P.active = active;
  }
  if (lane == 1) P.log_prob = det_log(dsub(1.0, pc.probability));  // (constant of the adaptive-k rule, once per frame)
  for (int k = lane; k < PCOP_MAX_PLANE_PASSES_RECORDED; k += 32) {
    P.pass_points[k] = 0;
    P.pass_inliers[k] = 0;
    P.pass_coeff[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  int nh = 0, gen_end = 0;
  if (active) {
    __shared__ GenScratch G;
    plane_gen_warp(in + (size_t)f * in_stride, n, rng, pc, G, P.hyp, P.hyp_valid, nh, gen_end);
  }
  if (lane == 0) {
    P.n_hyp = nh;
    P.gen_end = gen_end;
    if (gen_end == 2) atomicOr(&warnings[f], (uint32_t)PCOP_WARN_RNG_TABLE_EXHAUSTED);
  }
}

// inlier counts of hypotheses [h_begin, h_end) over this CTA's slice -> S.cnt, G hypotheses per sweep of the slice
// (h_end - h_begin is a multiple of G or runs into NaN planes, which count nothing)
template <int G, int THREADS>
__device__ __forceinline__ void pl_score(PlShared& S, const float* __restrict__ sx, const float* __restrict__ sy,
                                         const float* __restrict__ sz, int sn, float thr, int h_begin, int h_end) {
  const int lane = threadIdx.x & 31;
  for (int h0 = h_begin; h0 < h_end; h0 += G) {
    int c[G];
    float4 co[G];
#pragma unroll
    for (int j = 0; j < G; ++j) {
      c[j] = 0;
      co[j] = S.hyp[h0 + j];  // (MAX_HYP is a multiple of 8)
    }
    for (int i = threadIdx.x; i < sn; i += THREADS) {
      const float x = sx[i], y = sy[i], z = sz[i];
#pragma unroll
      for (int j = 0; j < G; ++j) c[j] += (plane_dist(co[j], x, y, z) < thr) ? 1 : 0;
    }
#pragma unroll
    for (int j = 0; j < G; ++j) {
      const int s = __reduce_add_sync(FULL, c[j]);
      if (lane == 0 && s) atomicAdd(&S.cnt[h0 + j], s);
    }
  }
}

// every CTA's counts of [h_begin, h_end) -> every CTA's cnt_all (followed by a cluster barrier at the call site)
template <int THREADS>
__device__ __forceinline__ void pl_push_counts(PlShared& S, unsigned rank, int h_begin, int h_end) {
  const int nhh = h_end - h_begin;
  for (int k = threadIdx.x; k < PL_CL * nhh; k += THREADS) {
    const unsigned r = (unsigned)(k / nhh);
    const int h = h_begin + k % nhh;
    *dsmem_ptr(&S.cnt_all[rank][h], r) = S.cnt[h];
  }
}

// thread 0: adaptive-k replay over the cluster-wide counts
__device__ __forceinline__ void pl_select(PlShared& S, const PlaneConst& pc, int n, int navail) {
  int sel = -1;
  const PlShared* Sp = &S;
  const bool more = plane_select_replay(pc, S.log_prob, n, S.nh, navail, S.hyp_valid,
                                        [Sp](int h) {
                                          int c = 0;
#pragma unroll
                                          for (int r = 0; r < PL_CL; ++r) c += Sp->cnt_all[r][h];
                                          return c;
                                        },
                                        sel);
  S.need_more = more ? 1 : 0;
  if (more) return;
  S.model_ok = (sel >= 0 && S.hyp_valid[sel]) ? 1 : 0;
  S.coeff_sel = (sel >= 0) ? S.hyp[sel] : make_float4(0.f, 0.f, 0.f, 0.f);
  S.coeff_ref = S.coeff_sel;
}

// ExtractIndices(negative) classification of a window of wn points in the slice planes: warp w takes the points
// [w * per_warp, (w + 1) * per_warp) row by row, bit r of keepmask = the point of row r is kept.  S.warp_excl[w] = base
// (warp 0's value) + the kept points of the warps before w.  Warp 0 adds the window's kept total to `total`.
template <int WARPS>
__device__ __forceinline__ unsigned pl_keep_scan(PlShared& S, const float* __restrict__ sx, const float* __restrict__ sy,
                                                 const float* __restrict__ sz, int wn, float4 co, bool ok, float thr,
                                                 int base, int& total) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per_warp = cdiv(cdiv(wn, WARPS), 32) * 32;  // <= 512: windows hold at most 16384 points
  const int rows = per_warp / 32;
  const int wb = warp * per_warp;
  unsigned keepmask = 0u;
  for (int r = 0; r < rows; ++r) {
    const int i = wb + r * 32 + lane;
    if (i < wn) {
      const bool inl = ok && plane_dist(co, sx[i], sy[i], sz[i]) < thr;
      if (!inl) keepmask |= 1u << r;
    }
  }
  const unsigned wtotal = __reduce_add_sync(FULL, (unsigned)__popc(keepmask));
  if (lane == 0) S.warp_excl[warp] = (int)wtotal;
  __syncthreads();
  if (warp == 0) {
    const int v = (lane < WARPS) ? S.warp_excl[lane] : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += up;
    }
    if (lane < WARPS) S.warp_excl[lane] = base + incl - v;
    total += __shfl_sync(FULL, incl, 31);
  }
  return keepmask;
}

// the kept points of a window classified by pl_keep_scan -> dpts / dsrc from slot wbase on (warp's share, row by row);
// its inliers -> inl[i - kept_before_i] (inl: nullptr when the inlier list is not wanted)
template <int WARPS>
__device__ __forceinline__ void pl_write(unsigned keepmask, unsigned wbase, int wlo, int wn, const float4* pts,
                                         const int* srcidx, float4* dpts, int* dsrc, int* inl) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per_warp = cdiv(cdiv(wn, WARPS), 32) * 32;
  const int wb = warp * per_warp;
  for (int r = 0; r < per_warp / 32; ++r) {
    const int i = wb + r * 32 + lane;
    const bool keep = (keepmask >> r) & 1u;
    const unsigned m = __ballot_sync(FULL, keep);
    const unsigned pos = wbase + __popc(m & lanemask_lt());
    const int gi = wlo + i;
    if (keep) {
      dpts[pos] = __ldcg(pts + gi);
      dsrc[pos] = srcidx ? __ldcg(srcidx + gi) : gi;
    } else if (i < wn && inl) {
      inl[gi - (int)pos] = gi;
    }
    wbase += __popc(m);
  }
}

// THREADS = 512: two CTAs (of different frames) per SM, so one frame's barriers and single-thread phases overlap the
// other's sweeps; needs slices of at most 8192 points.  THREADS = 1024: one CTA per SM, slices up to 16384 points.
// WINDOWS (1024 threads, frames of any size): a CTA whose range of the frame is longer than its slice walks it in
// windows of slice_cap points.  (A separate instantiation: its extra live state costs the frames that fit 7 % of their
// time in spills, so waves whose frames all fit take the one without.)  Each launch takes the frames with n_lo < n <= n_hi points (the host does not know the sizes: it
// launches the small tier for everything and the larger ones only if the wave's largest input frame could need them).
// gpart: [B][cdiv(cap, TS_CHUNK)][10] chunk partials of the frames with more chunks than nch_max (WINDOWS only).
template <int THREADS, bool WINDOWS>
__global__ void __cluster_dims__(PL_CL, 1, 1) __launch_bounds__(THREADS, THREADS == 512 ? 2 : 1)
    k_plane_loop(PlaneFrame* __restrict__ pf, const float4* __restrict__ in, size_t in_stride, BufPair bp, PlaneConst pc,
                 const int* __restrict__ rng, int* __restrict__ inlier_idx, float4* __restrict__ out,
                 int* __restrict__ out_src, int* __restrict__ n_out, uint32_t* __restrict__ warnings, int cap,
                 int slice_cap, int nch_max, int n_lo, int n_hi, double* __restrict__ gpart) {
  constexpr int PL_THREADS = THREADS, PL_WARPS = THREADS / 32, PL_GROUPS = THREADS / 256;
  const unsigned rank = cluster_ctarank();
  const int f = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  extern __shared__ __align__(16) unsigned char pl_smem[];
  PlShared& S = *reinterpret_cast<PlShared*>(pl_smem);
  double* part = reinterpret_cast<double*>(pl_smem + sizeof(PlShared));  // [nch_max][10] chunk partials of the whole frame
  float* sx = reinterpret_cast<float*>(pl_smem + sizeof(PlShared) + (size_t)nch_max * 80);
  float* sy = sx + slice_cap;
  float* sz = sy + slice_cap;
  GenScratch& G = *reinterpret_cast<GenScratch*>(sx);  // (only live between two passes, when the slices are dead)

  PlaneFrame& P = pf[f];
  // loop state: read once, then carried in registers by every thread of every CTA (all decisions are deterministic
  // functions of cluster-wide data, so the copies never diverge); CTA 0 / thread 0 writes it back
  int n = P.n, cur = P.cur, active = P.active, n_passes = P.n_passes;
  const int nr = P.nr_points;
  if (n <= n_lo || n > n_hi) return;  // another tier's frame (uniform over the cluster)
  bool first = true;

  if (!active) {  // the loop never starts (empty cloud, keep_fraction >= 1): planar_cloud_y = the input
    const float4* pts = in + (size_t)f * in_stride;
    for (int i = (int)rank * PL_THREADS + tid; i < n; i += PL_CL * PL_THREADS) {
      out[(size_t)f * cap + i] = __ldg(pts + i);
      out_src[(size_t)f * cap + i] = i;
    }
    if (rank == 0 && tid == 0) n_out[f] = n;
    return;
  }

  while (true) {
    PL_CLK(0);
    const float4* pts = (cur < 0) ? (in + (size_t)f * in_stride) : (bp.p[cur] + (size_t)f * cap);
    const int* srcidx = (cur < 0) ? nullptr : (bp.s[cur] + (size_t)f * cap);
    // CTA ranges: whole CT2048 chunks, so that a chunk never spans two CTAs.  A range longer than the slice (WINDOWS
    // only) is walked in windows of slice_cap points, whole chunks as well: a CTA with one window loads it once per pass,
    // one with more reloads every window in each phase that reads the cloud (scoring batch, moments, extraction)
    const int SLf = cdiv(cdiv(n, PL_CL), TS_CHUNK) * TS_CHUNK;
    const int SL = WINDOWS ? SLf : min(slice_cap, SLf);
    const int lo = min((int)rank * SL, n), hi = min(lo + SL, n), sn = hi - lo;
    const bool multi = WINDOWS && SL > slice_cap;  // (uniform over the cluster: more chunks than nch_max)
    const int nwin = multi ? max(1, cdiv(sn, slice_cap)) : 1;
    // Pass 0 reads the stage input (written by an earlier kernel); later passes read a cloud that other CTAs of the
    // cluster wrote during this launch: ld.global.cg, an earlier pass may have left stale L1 lines.
    const bool fresh = !first;
    // points [w0, w0 + wn) -> the slice planes, eight 16-byte loads in flight per thread (the load is latency-bound: four
    // in flight took 12 k cycles, and cp.async with 4-byte elements -- three per point straight into the planes -- is
    // bound by the LDGSTS issue rate at 11.5 k)
    auto load = [=](int w0, int wn) {
      for (int i0 = tid; i0 < wn; i0 += 8 * PL_THREADS) {
        float4 p[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = i0 + u * PL_THREADS;
          p[u] = (i < wn) ? (fresh ? __ldcg(pts + w0 + i) : __ldg(pts + w0 + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = i0 + u * PL_THREADS;
          if (i < wn) {
            sx[i] = p[u].x;
            sy[i] = p[u].y;
            sz[i] = p[u].z;
          }
        }
      }
    };
    // window w of this CTA's range in the slice planes; returns its size
    auto window = [=](int w) {
      if (nwin == 1) return sn;
      const int wlo = lo + w * slice_cap, wn = min(slice_cap, hi - wlo);
      __syncthreads();
      load(wlo, wn);
      __syncthreads();
      return wn;
    };
    if (nwin == 1) load(lo, sn);
    if (first) {  // pass 0: hypotheses from k_plane_gen0 (later passes: generated below, already in shared memory)
      if (tid == 0) {
        S.nh = P.n_hyp;
        S.gen_end = P.gen_end;
        S.log_prob = P.log_prob;
      }
      if (tid < MAX_HYP) {
        S.hyp[tid] = P.hyp[tid];
        S.hyp_valid[tid] = P.hyp_valid[tid];
      }
      first = false;
    }
    __syncthreads();
    if (tid < MAX_HYP) {
      // hypotheses past nh are NaN planes: |NaN| < thr is false, so they count nothing
      const float qnan = __uint_as_float(0x7fc00000u);
      if (tid >= S.nh) S.hyp[tid] = make_float4(qnan, qnan, qnan, qnan);
      S.cnt[tid] = 0;
    }
    __syncthreads();
    const int nh = S.nh;
    PL_CLK(1);

    // ---- RANSAC: score a batch of hypotheses, replay the adaptive-k loop, go on only if the replay ran past them -----
    for (int ph = 0, scored = 0; ph < PL_N_BATCHES; ++ph) {
      const int end = PL_BATCH_END[ph];
      for (int w = 0; w < nwin; ++w) {
        const int wn = window(w);
        if (end - scored <= 4) pl_score<4, PL_THREADS>(S, sx, sy, sz, wn, pc.thr, scored, min(nh, end));
        else pl_score<8, PL_THREADS>(S, sx, sy, sz, wn, pc.thr, scored, min(nh, end));
      }
      __syncthreads();
      pl_push_counts<PL_THREADS>(S, rank, scored, end);
      PL_CLK(2);
      cluster_sync_all();
      PL_CLK(3);
      if (tid == 0) pl_select(S, pc, n, end);
      __syncthreads();
      PL_CLK(4);
      if (!S.need_more) break;  // (uniform over the cluster: every CTA replays the same counts)
      scored = end;
    }
    const bool ok = S.model_ok != 0;
    PL_CLK(5);

    // ---- optimizeModelCoefficients: CT2048 moments of the RANSAC inliers, eigen33 ----------------------------------
    if (pc.optimize && ok) {
      const float4 co = S.coeff_sel;
      const int g = tid >> 8, t = tid & 255, gw = (tid >> 5) & 7;
      // the chunk partials of the whole frame: in shared memory, or (more chunks than nch_max) in global memory
      double* fpart = multi ? gpart + (size_t)f * cdiv(cap, TS_CHUNK) * 10 : part;
      for (int wi = 0; wi < nwin; ++wi) {
        const int wn = window(wi);
        const int nlc = cdiv(wn, TS_CHUNK);
        const int gc0 = (lo + wi * slice_cap) / TS_CHUNK;  // first chunk of the window
        for (int lc = g; lc < nlc; lc += PL_GROUPS) {
          double a[9];
#pragma unroll
          for (int k = 0; k < 9; ++k) a[k] = 0.0;
          int cnt = 0;
#pragma unroll
          for (int r = 0; r < TS_CHUNK / 256; ++r) {
            const int i = lc * TS_CHUNK + r * 256 + t;
            double e[9];
#pragma unroll
            for (int k = 0; k < 9; ++k) e[k] = 0.0;
            if (i < wn) {
              const float px = sx[i], py = sy[i], pz = sz[i];
              if (plane_dist(co, px, py, pz) < pc.thr) {
                const double x = px, y = py, z = pz;
                e[0] = dmul(x, x);
                e[1] = dmul(x, y);
                e[2] = dmul(x, z);
                e[3] = dmul(y, y);
                e[4] = dmul(y, z);
                e[5] = dmul(z, z);
                e[6] = x;
                e[7] = y;
                e[8] = z;
                ++cnt;
              }
            }
#pragma unroll
            for (int k = 0; k < 9; ++k) a[k] = dadd(a[k], e[k]);
          }
#pragma unroll
          for (int k = 0; k < 9; ++k) a[k] = tree_butterfly(a[k]);
          cnt = __reduce_add_sync(FULL, cnt);
          if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 9; ++k) S.msh[g][gw][k] = a[k];
            S.mcnt[g][gw] = cnt;
          }
          group_bar_sync<PL_GROUPS>(g);
          double* o = fpart + (size_t)(gc0 + lc) * 10;
          if (t < 9) {
            double s = S.msh[g][0][t];
            for (int w = 1; w < 8; ++w) s = dadd(s, S.msh[g][w][t]);
            o[t] = s;
          } else if (t == 9) {
            int c = 0;
            for (int w = 0; w < 8; ++w) c += S.mcnt[g][w];
            o[9] = (double)c;
          }
          group_bar_sync<PL_GROUPS>(g);
        }
      }
      __syncthreads();
      if (multi) {
        __threadfence();  // (the partials are read back by warp 0 of every CTA after the barrier)
      } else {
        // this CTA's chunk partials -> every peer
        const int nv = cdiv(sn, TS_CHUNK) * 10;
        for (int k = tid; k < (PL_CL - 1) * nv; k += PL_THREADS) {
          const unsigned r = (rank + 1u + (unsigned)(k / nv)) % PL_CL;
          double* mine = part + (size_t)(lo / TS_CHUNK) * 10 + k % nv;
          *dsmem_ptr(mine, r) = *mine;
        }
      }
      PL_CLK(6);
      cluster_sync_all();
      PL_CLK(7);
      if (warp == 0) {
        const int nch = cdiv(n, TS_CHUNK);
        double tot = 0.0;
        if (lane < 10) {  // (in chunk order: the same sum for any slice and window size)
          if (multi) {
#pragma unroll 8
            for (int c = 0; c < nch; ++c) tot = dadd(tot, __ldcg(fpart + (size_t)c * 10 + lane));
          } else {
            for (int c = 0; c < nch; ++c) tot = dadd(tot, part[(size_t)c * 10 + lane]);
          }
        }
        double a[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) a[k] = __shfl_sync(FULL, tot, k);
        const double cntd = __shfl_sync(FULL, tot, 9);
        if (lane == 0) {
          float4 o;
          if (plane_refine_model(pc, a, cntd, o)) S.coeff_ref = o;
        }
      }
      __syncthreads();
    }

    // ---- ExtractIndices(negative) with the refined model: stable compaction over the cluster -----------------------
    PL_CLK(8);
    const float4 co = S.coeff_ref;
    // The output order is CTA rank, window, warp, row.  A CTA with one window classifies it once (keep mask in
    // registers); one with more counts its kept points in a sweep over its windows here and classifies every window
    // again in the write sweep below.
    const int per_warp = cdiv(cdiv(sn, PL_WARPS), 32) * 32;  // <= 1024: slices hold at most 32768 points
    const int rows = per_warp / 32;
    const int wb = warp * per_warp;
    unsigned keepmask = 0u;
    if (nwin > 1) {
      int kept = 0;  // (warp 0)
      for (int w = 0; w < nwin; ++w) pl_keep_scan<PL_WARPS>(S, sx, sy, sz, window(w), co, ok, pc.thr, 0, kept);
      if (warp == 0 && lane < PL_CL) *dsmem_ptr(&S.kept_all[rank], (unsigned)lane) = kept;
    } else {
      for (int r = 0; r < rows; ++r) {
        const int i = wb + r * 32 + lane;
        if (i < sn) {
          const bool inl = ok && plane_dist(co, sx[i], sy[i], sz[i]) < pc.thr;
          if (!inl) keepmask |= 1u << r;
        }
      }
      const unsigned wtotal = __reduce_add_sync(FULL, (unsigned)__popc(keepmask));
      if (lane == 0) S.warp_excl[warp] = (int)wtotal;
      __syncthreads();
      if (warp == 0) {
        const int v = (lane < PL_WARPS) ? S.warp_excl[lane] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int up = __shfl_up_sync(FULL, incl, o);
          if (lane >= o) incl += up;
        }
        if (lane < PL_WARPS) S.warp_excl[lane] = incl - v;
        const int total = __shfl_sync(FULL, incl, 31);
        if (lane < PL_CL) *dsmem_ptr(&S.kept_all[rank], (unsigned)lane) = total;
      }
    }
    PL_CLK(9);
    cluster_sync_all();
    PL_CLK(10);
    int base = 0, remaining = 0;
#pragma unroll
    for (int r = 0; r < PL_CL; ++r) {
      const int k = S.kept_all[r];
      base += (r < (int)rank) ? k : 0;
      remaining += k;
    }
    const int inliers = n - remaining;
    const bool go_on = inliers != 0 && ((double)remaining > dmul(pc.keep_fraction, (double)nr));  // od.cpp:379, 383-387
    const int dst = (cur < 0) ? 0 : (1 - cur);
    float4* dpts = go_on ? (bp.p[dst] + (size_t)f * cap) : (out + (size_t)f * cap);
    int* dsrc = go_on ? (bp.s[dst] + (size_t)f * cap) : (out_src + (size_t)f * cap);
    if (nwin > 1) {
      int run = 0;  // (warp 0) kept points of this CTA's earlier windows
      for (int w = 0; w < nwin; ++w) {
        const int wn = window(w), wlo = lo + w * slice_cap;
        const unsigned km = pl_keep_scan<PL_WARPS>(S, sx, sy, sz, wn, co, ok, pc.thr, run, run);
        __syncthreads();
        pl_write<PL_WARPS>(km, (unsigned)(base + S.warp_excl[warp]), wlo, wn, pts, srcidx, dpts, dsrc,
                           inlier_idx ? inlier_idx + (size_t)f * cap : nullptr);
      }
    } else {
      unsigned wbase = (unsigned)(base + S.warp_excl[warp]);
      for (int r = 0; r < rows; ++r) {
        const int i = wb + r * 32 + lane;
        const bool keep = (keepmask >> r) & 1u;
        const unsigned m = __ballot_sync(FULL, keep);
        const unsigned pos = wbase + __popc(m & lanemask_lt());
        const int gi = lo + i;
        if (keep) {
          dpts[pos] = __ldcg(pts + gi);  // (the padding word travels with the point)
          dsrc[pos] = srcidx ? __ldcg(srcidx + gi) : gi;
        } else if (i < sn && inlier_idx) {
          inlier_idx[(size_t)f * cap + (gi - (int)pos)] = gi;
        }
        wbase += __popc(m);
      }
    }

    // ---- od.cpp:379-399 bookkeeping ----------------------------------------------------------------------------------
    PL_CLK(11);
    if (inliers == 0) {  // od.cpp:383-387: "Couldn't estimate a planar model", break; the cloud is unchanged
      if (rank == 0 && tid == 0) {
        P.n_inliers_last = 0;
        P.active = 0;
        P.coeff_sel = S.coeff_sel;
        P.coeff_ref = S.coeff_ref;
        atomicOr(&warnings[f], (uint32_t)PCOP_WARN_PLANE_BREAK);
        n_out[f] = n;
      }
      return;
    }
    if (rank == 0 && tid == 0) {
      if (n_passes < PCOP_MAX_PLANE_PASSES_RECORDED) {
        P.pass_points[n_passes] = n;
        P.pass_inliers[n_passes] = inliers;
        P.pass_coeff[n_passes] = S.coeff_ref;
      }
      P.n_passes = n_passes + 1;
      P.n_inliers_last = inliers;
      P.n = remaining;
      P.coeff_sel = S.coeff_sel;
      P.coeff_ref = S.coeff_ref;
      P.active = go_on ? 1 : 0;
      if (!go_on) n_out[f] = remaining;
    }
    if (!go_on) return;
    n_passes += 1;
    cur = dst;  // planar_cloud.swap(cloud_f)
    n = remaining;

    // ---- another pass: the new cloud must be visible to the whole cluster, then every CTA generates the (same)
    // hypotheses into its own shared memory; the scratch overlays the slices, which are dead until the reload
    __threadfence();
    cluster_sync_all();
    if (warp == 0) {
      int gnh, gen_end;
      plane_gen_warp(bp.p[cur] + (size_t)f * cap, n, rng, pc, G, S.hyp, S.hyp_valid, gnh, gen_end);
      if (lane == 0) {
        S.nh = gnh;
        S.gen_end = gen_end;
        if (gen_end == 2 && rank == 0) atomicOr(&warnings[f], (uint32_t)PCOP_WARN_RNG_TABLE_EXHAUSTED);
      }
    }
    __syncthreads();
  }
}

}  // namespace

// slice sizes in points: the large tier's frames above 8 x PL_SLICE_MAX points are walked in windows of that size
constexpr int PL_SLICE_MAX = 16384;
constexpr int PL_SLICE_SMALL = 8192;

int plane_small_tier_max() { return PL_CL * PL_SLICE_SMALL; }

cudaError_t run_plane(const Ctx& c, const PlaneArgs& a) {
  BufPair bp;
  bp.p[0] = a.buf[0];
  bp.p[1] = a.buf[1];
  bp.s[0] = a.src[0];
  bp.s[1] = a.src[1];
  KL(c, "k_plane_gen0", k_plane_gen0<<<c.B, 32, 0, c.stream>>>(a.pf, a.in, a.in_stride, a.n_in, a.n_in_copy, a.rng, a.pc, a.warnings));
  count_launch(c);
  static_assert(sizeof(GenScratch) <= 4096 * 12, "the generator scratch overlays the smallest slice planes");
  static_assert(sizeof(PlShared) % 16 == 0, "alignment of the regions behind PlShared");
  auto smem_bytes = [](int slice_cap) { return sizeof(PlShared) + (size_t)(PL_CL * slice_cap / TS_CHUNK) * 80 + (size_t)slice_cap * 12; };
  // small tier: slices of at most 8192 points (two CTAs per SM)
  const int bound = std::min(c.grid_cap, PL_CL * PL_SLICE_MAX);
  const int small_slice = std::min(PL_SLICE_SMALL, std::max(4096, cdiv(cdiv(bound, PL_CL), TS_CHUNK) * TS_CHUNK));
  const int small_max = PL_CL * small_slice;
  {
    const size_t smem = smem_bytes(small_slice);
    cudaFuncSetAttribute(k_plane_loop<512, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  // per device, idempotent
    KL(c, "k_plane_loop", k_plane_loop<512, false><<<dim3(PL_CL, c.B), 512, smem, c.stream>>>(
                              a.pf, a.in, a.in_stride, bp, a.pc, a.rng, a.inlier_idx, a.out, a.out_src, a.n_out, a.warnings,
                              c.cap, small_slice, PL_CL * small_slice / TS_CHUNK, -1, small_max, a.partial));
    count_launch(c);
  }
  // Larger frames take the one-CTA-per-SM tier.  The host does not know the sizes of the clouds that reach the plane
  // stage, so the tier is launched only when the caller expects such frames (a.large_tier: a frame of an earlier wave was
  // that large, or the stage is being repeated because one of this wave turned out to be); frames it would have taken
  // are left untouched by the small tier and reported through plane_small_tier_max().  A wave whose input frames could
  // reach the plane stage with more than 8 slices takes the windowed instantiation for all of its large frames (one
  // launch: the frames of the wave run side by side); otherwise the one without windows, which spills less.
  if (c.grid_cap > small_max && a.large_tier) {
    const int slice_cap = cdiv(cdiv(bound, PL_CL), TS_CHUNK) * TS_CHUNK;
    const size_t smem = smem_bytes(slice_cap);
    if (c.grid_cap > PL_CL * slice_cap) {
      cudaFuncSetAttribute(k_plane_loop<1024, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      KL(c, "k_plane_loop_windows", k_plane_loop<1024, true><<<dim3(PL_CL, c.B), 1024, smem, c.stream>>>(
                                        a.pf, a.in, a.in_stride, bp, a.pc, a.rng, a.inlier_idx, a.out, a.out_src, a.n_out,
                                        a.warnings, c.cap, slice_cap, PL_CL * slice_cap / TS_CHUNK, small_max, INT_MAX,
                                        a.partial));
    } else {
      cudaFuncSetAttribute(k_plane_loop<1024, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      KL(c, "k_plane_loop_large", k_plane_loop<1024, false><<<dim3(PL_CL, c.B), 1024, smem, c.stream>>>(
                                      a.pf, a.in, a.in_stride, bp, a.pc, a.rng, a.inlier_idx, a.out, a.out_src, a.n_out,
                                      a.warnings, c.cap, slice_cap, PL_CL * slice_cap / TS_CHUNK, small_max,
                                      PL_CL * slice_cap, a.partial));
    }
    count_launch(c);
  }
  return cudaGetLastError();
}

}  // namespace pcop

#ifdef PCOP_PLANE_DEBUG_CLK
extern "C" int pcop_debug_plane_loop_cycles(long long* out16) {
  return (int)cudaMemcpyFromSymbol(out16, pcop::g_plane_loop_clk, sizeof(long long) * 16);
}
#endif
