// Obstacle footprints (PCOP_OUT_FOOTPRINTS): per cluster, the axis-aligned box of its members and the 2-D convex hull
// of the members projected along z.
//
// Box: {min x, min y, min z, 0, max x, max y, max z, 0} in IEEE totalOrder (-0 < +0), reduced on the order-preserving
// uint32 of every float, so the result does not depend on the reduction order.  A singleton (the only cluster that can
// hold a non-finite point: the ECE kernels give such a point a private cell without neighbours) copies its member.
//
// Hull: the strictly extreme projected members, counter-clockwise from the lexicographically smallest (x, y); members
// with equal (x, y) (float ==) count once, as their smallest remaining-cloud index.  Every orientation is Shewchuk's
// orient2d: the double evaluation with the ccwerrboundA filter, then an exact expansion.  The answer is therefore unique
// and any hull algorithm reaches it; this one works on pieces of at most FP_PIECE members:
//   k_fp_piece    one block per piece (a persistent grid per frame walks the pieces of all clusters): gather the
//                 members into shared memory, the box, an Akl-Toussaint octagon prefilter (points strictly inside the
//                 octagon of eight extreme members are dropped, by the exact predicate), a bitonic sort by (x, y, index)
//                 and Andrew's monotone chain.  A single-piece cluster is finished here; a piece of a larger one leaves
//                 its hull in the staging at the piece's first member slot.
//   k_fp_combine  one block per multi-piece cluster: the box over all members, then the hull of the union of the piece
//                 hulls, in shared memory when the union fits FP_PIECE points, else in global scratch (the cluster's
//                 slots of `work`) with the same sort and chain -- the path of clusters whose members are mostly extreme.
//   k_fp_csr      one block per frame: hull sizes -> CSR offsets, the staged vertices -> hull_indices.
// Launch counts per call: k_fp_piece + k_fp_csr, and k_fp_combine when a frame may hold a cluster above FP_PIECE.
#include "internal.cuh"
#include "primitives.cuh"

namespace pcop {
namespace {

constexpr int FP_PIECE = 4096;    // members per piece (one shared-memory tile)
constexpr int FP_THREADS = 512;
constexpr int FP_GRID = 32;       // blocks per frame of k_fp_piece
constexpr int FP_COMBINE_GRID = 4;   // blocks per frame of k_fp_combine (most frames have no multi-piece cluster)
constexpr size_t FP_SMEM = (size_t)FP_PIECE * sizeof(float4) + (size_t)FP_PIECE * sizeof(int);

// ---- Shewchuk's orient2d (Adaptive Precision Floating-Point Arithmetic and Fast Robust Geometric Predicates, 1997):
// > 0 when c lies left of a -> b.  Every operation is an explicitly rounded double op; TwoProduct uses the FMA.
__device__ __forceinline__ void two_sum(double a, double b, double& x, double& y) {
  x = __dadd_rn(a, b);
  const double bv = __dsub_rn(x, a);
  const double av = __dsub_rn(x, bv);
  y = __dadd_rn(__dsub_rn(a, av), __dsub_rn(b, bv));
}
__device__ __forceinline__ void two_diff(double a, double b, double& x, double& y) {
  x = __dsub_rn(a, b);
  const double bv = __dsub_rn(a, x);
  const double av = __dadd_rn(x, bv);
  y = __dadd_rn(__dsub_rn(a, av), __dsub_rn(bv, b));
}
__device__ __forceinline__ void two_product(double a, double b, double& x, double& y) {
  x = __dmul_rn(a, b);
  y = __fma_rn(a, b, -x);
}

// the sign of (acx + acxt)(bcy + bcyt) - (acy + acyt)(bcx + bcxt), exactly: 16 products summed into a nonoverlapping
// expansion (Grow-Expansion), whose largest nonzero component carries the sign
__device__ __noinline__ double orient2d_exact(double acx, double acxt, double bcy, double bcyt, double acy, double acyt,
                                              double bcx, double bcxt) {
  double e[17];
  int n = 0;
  const double l[4] = {acx, acx, acxt, acxt}, r[4] = {bcy, bcyt, bcy, bcyt};
  const double l2[4] = {acy, acy, acyt, acyt}, r2[4] = {bcx, bcxt, bcx, bcxt};
  for (int t = 0; t < 8; ++t) {
    double hi, lo;
    if (t < 4) two_product(l[t], r[t], hi, lo);
    else two_product(-l2[t - 4], r2[t - 4], hi, lo);
    const double parts[2] = {lo, hi};
    for (int s = 0; s < 2; ++s) {
      double q = parts[s];
      int m = 0;
      for (int i = 0; i < n; ++i) {  // Grow-Expansion with zero elimination
        double x, y;
        two_sum(q, e[i], x, y);
        q = x;
        if (y != 0.0) e[m++] = y;
      }
      if (q != 0.0) e[m++] = q;
      n = m;
    }
  }
  return n ? e[n - 1] : 0.0;
}

__device__ __forceinline__ double orient2d(float ax, float ay, float bx, float by, float cx, float cy) {
  const double acx = __dsub_rn((double)ax, (double)cx), bcx = __dsub_rn((double)bx, (double)cx);
  const double acy = __dsub_rn((double)ay, (double)cy), bcy = __dsub_rn((double)by, (double)cy);
  const double detleft = __dmul_rn(acx, bcy), detright = __dmul_rn(acy, bcx);
  const double det = __dsub_rn(detleft, detright);
  double detsum;
  if (detleft > 0.0) {
    if (detright <= 0.0) return det;
    detsum = __dadd_rn(detleft, detright);
  } else if (detleft < 0.0) {
    if (detright >= 0.0) return det;
    detsum = __dsub_rn(-detleft, detright);
  } else {
    return det;
  }
  const double ccwerrboundA = 3.3306690738754716e-16;  // (3 + 16 eps) eps, eps = 2^-53
  const double errbound = __dmul_rn(ccwerrboundA, detsum);
  if (det >= errbound || -det >= errbound) return det;
  double acxt, bcxt, acyt, bcyt, t0, t1;
  two_diff((double)ax, (double)cx, t0, acxt);
  two_diff((double)bx, (double)cx, t1, bcxt);
  two_diff((double)ay, (double)cy, t0, acyt);
  two_diff((double)by, (double)cy, t1, bcyt);
  return orient2d_exact(acx, acxt, bcy, bcyt, acy, acyt, bcx, bcxt);
}

// candidates: {x, y, remaining-cloud index (bits), 0 (monotone_chain marks the lower chain there)}
__device__ __forceinline__ bool cand_less(const float4& a, const float4& b) {
  if (a.x != b.x) return a.x < b.x;
  if (a.y != b.y) return a.y < b.y;
  return __float_as_int(a.z) < __float_as_int(b.z);
}
__device__ __forceinline__ bool same_xy(const float4& a, const float4& b) { return a.x == b.x && a.y == b.y; }
__device__ __forceinline__ double orient_c(const float4& a, const float4& b, const float4& c) {
  return orient2d(a.x, a.y, b.x, b.y, c.x, c.y);
}

// Sorts buf[0, n) by (x, y, index) with the whole block: a bitonic network over the next power of two in which every
// compare-exchange is ascending (the first step of each merge compares mirrored positions), so the positions past n
// act as +inf and never move.  buf may be shared or global memory.
__device__ void block_sort(float4* buf, int n) {
  int n2 = 1;
  while (n2 < n) n2 <<= 1;
  for (int k = 2; k <= n2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < n2 / 2; t += blockDim.x) {
        // t-th pair of this step: i has bit j clear
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int l = (j == (k >> 1)) ? (i ^ (k - 1)) : (i | j);
        if (l < n) {
          const float4 a = buf[i], b = buf[l];
          if (cand_less(b, a)) {
            buf[i] = b;
            buf[l] = a;
          }
        }
      }
      __syncthreads();
    }
  }
}

// Andrew's monotone chain over the sorted candidates buf[0, n) (n >= 1) by one thread: strictly convex turns only,
// each (x, y) once (the first of a run: the smallest index).  Leaves the hull's candidate positions in st and returns
// the vertex count.  The upper pass skips the vertices of the lower chain (marked in buf[].w, which the candidates
// carry as 0): they lie strictly below the segment from the first to the last point, so they are no upper-hull
// vertices, and without them the stack never holds more than the distinct points (it would hold one more when the
// second point is a lower-chain vertex and every point is extreme).  st has room for the distinct points.
__device__ int monotone_chain(float4* buf, int n, int* st) {
  int k = 0;
  for (int i = 0; i < n; ++i) {
    if (i > 0 && same_xy(buf[i], buf[i - 1])) continue;
    while (k >= 2 && orient_c(buf[st[k - 2]], buf[st[k - 1]], buf[i]) <= 0.0) --k;
    st[k++] = i;
  }
  if (k == 1) return 1;
  const int lower = k;
  const int last = st[k - 1];
  for (int j = 1; j < lower - 1; ++j) buf[st[j]].w = 1.0f;
  for (int i = last - 1; i >= 0; --i) {
    if (i > 0 && (same_xy(buf[i], buf[i - 1]) || buf[i].w != 0.0f)) continue;
    while (k > lower && orient_c(buf[st[k - 2]], buf[st[k - 1]], buf[i]) <= 0.0) --k;
    if (i > 0) st[k++] = i;  // (the first point closes the chain; it is st[0] already)
  }
  return k;
}

// the box keys of one member (order-preserving uint32 of x, y, z)
struct BoxKeys {
  unsigned mn[3], mx[3];
};
__device__ __forceinline__ void box_init(BoxKeys& b) {
  for (int a = 0; a < 3; ++a) {
    b.mn[a] = 0xffffffffu;
    b.mx[a] = 0u;
  }
}
__device__ __forceinline__ void box_add(BoxKeys& b, const float4& p) {
  const unsigned k[3] = {f2ord(p.x), f2ord(p.y), f2ord(p.z)};
  for (int a = 0; a < 3; ++a) {
    b.mn[a] = min(b.mn[a], k[a]);
    b.mx[a] = max(b.mx[a], k[a]);
  }
}
// block reduction of the box into sh (6 words), written to out[8] by thread 0
__device__ void box_finish(BoxKeys& b, unsigned* sh, float* out) {
  for (int a = 0; a < 3; ++a) {
    b.mn[a] = __reduce_min_sync(FULL, b.mn[a]);
    b.mx[a] = __reduce_max_sync(FULL, b.mx[a]);
  }
  if ((threadIdx.x & 31) == 0)
    for (int a = 0; a < 3; ++a) {
      atomicMin(&sh[a], b.mn[a]);
      atomicMax(&sh[3 + a], b.mx[a]);
    }
  __syncthreads();
  if (threadIdx.x == 0) {
    reinterpret_cast<float4*>(out)[0] = make_float4(ord2f(sh[0]), ord2f(sh[1]), ord2f(sh[2]), 0.0f);
    reinterpret_cast<float4*>(out)[1] = make_float4(ord2f(sh[3]), ord2f(sh[4]), ord2f(sh[5]), 0.0f);
  }
}

// Akl-Toussaint prefilter of buf[0, n) in shared memory: the members extreme along +-x, +-y, +-(x + y), +-(x - y)
// (any choice of members is safe: a point strictly left of every non-degenerate edge of a closed chain of members
// winds inside it, hence lies strictly inside the members' hull); survivors are compacted to the front.
// Returns the survivor count.  sel: 8 x u64 shared scratch.
__device__ int octagon_filter(float4* buf, int n, unsigned long long* sel, int* count) {
  // keys: (order of the directional value) << 32 | position; min over 8 directions (max = min of the complement)
  unsigned long long best[8];
  for (int d = 0; d < 8; ++d) best[d] = ~0ull;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float4 p = buf[i];
    const float s = __fadd_rn(p.x, p.y), t = __fsub_rn(p.x, p.y);
    // CCW order of the outward directions: -y, +(x - y), +x, +(x + y), +y, -(x - y), -x, -(x + y)
    const unsigned v[8] = {f2ord(p.y), ~f2ord(t), ~f2ord(p.x), ~f2ord(s), ~f2ord(p.y), f2ord(t), f2ord(p.x), f2ord(s)};
    for (int d = 0; d < 8; ++d) best[d] = min(best[d], ((unsigned long long)v[d] << 32) | (unsigned)i);
  }
  for (int d = 0; d < 8; ++d) {
    for (int o = 16; o >= 1; o >>= 1) best[d] = min(best[d], __shfl_xor_sync(FULL, best[d], o));
    if ((threadIdx.x & 31) == 0) atomicMin(&sel[d], best[d]);
  }
  __syncthreads();
  float4 oct[8];
  for (int d = 0; d < 8; ++d) oct[d] = buf[(int)(sel[d] & 0xffffffffu)];
  // each thread keeps its survivors in registers (static indices) until everyone has read buf
  constexpr int PER = FP_PIECE / FP_THREADS;
  float4 keep[PER];
  unsigned kept = 0u;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const int i = threadIdx.x + k * FP_THREADS;
    if (i >= n) continue;
    keep[k] = buf[i];
    bool inside = false;
    for (int d = 0; d < 8; ++d) {
      const float4& a = oct[d];
      const float4& b = oct[(d + 1) & 7];
      if (same_xy(a, b)) continue;
      inside = orient_c(a, b, keep[k]) > 0.0;
      if (!inside) break;
    }
    if (!inside) kept |= 1u << k;
  }
  __syncthreads();
  int pos = kept ? atomicAdd(count, __popc(kept)) : 0;
#pragma unroll
  for (int k = 0; k < PER; ++k)
    if (kept & (1u << k)) buf[pos++] = keep[k];
  __syncthreads();
  return *count;
}

// the hull of buf[0, n) (n >= 1): sort, chain (thread 0, stack in st), vertices' indices to out.  Returns the vertex
// count (every thread).
__device__ int hull_of(float4* buf, int n, int* st, int* out, int* sh_h) {
  block_sort(buf, n);
  if (threadIdx.x == 0) *sh_h = monotone_chain(buf, n, st);
  __syncthreads();
  const int h = *sh_h;
  for (int k = threadIdx.x; k < h; k += blockDim.x) out[k] = __float_as_int(buf[st[k]].z);
  __syncthreads();
  return h;
}

struct FpShared {
  unsigned box[6];
  unsigned long long sel[8];
  int count, h;
};
__device__ __forceinline__ void fp_shared_reset(FpShared& s) {
  if (threadIdx.x < 6) s.box[threadIdx.x] = threadIdx.x < 3 ? 0xffffffffu : 0u;
  if (threadIdx.x < 8) s.sel[threadIdx.x] = ~0ull;
  if (threadIdx.x == 0) s.count = 0;
}

__global__ void __launch_bounds__(FP_THREADS, 1)
    k_fp_piece(FootprintArgs a, int cap) {
  extern __shared__ __align__(16) unsigned char fp_smem[];
  float4* buf = reinterpret_cast<float4*>(fp_smem);
  int* st = reinterpret_cast<int*>(fp_smem + (size_t)FP_PIECE * sizeof(float4));
  __shared__ FpShared s;
  const int f = blockIdx.y;
  const int C = a.n_clusters[f];
  const float4* src = a.in + (size_t)f * a.in_stride;
  const int* offs = a.offsets + (size_t)f * (cap + 1);
  const int* idx = a.indices + (size_t)f * cap;
  float* boxes = a.boxes + (size_t)f * cap * 8;
  int* count = a.hull_count + (size_t)f * (cap + 1);
  int* stage = a.stage + (size_t)f * cap;
  int* pcount = a.hull_indices + (size_t)f * cap;  // (piece hull sizes at the piece's first slot; k_fp_csr overwrites)
  // items: the pieces of every cluster in cluster order; the walk resumes where the block's previous item was found
  int c = 0, first_item = 0;
  for (int item = blockIdx.x;; item += gridDim.x) {
    int pieces = 0;
    while (c < C) {
      pieces = max(1, cdiv(offs[c + 1] - offs[c], FP_PIECE));
      if (item < first_item + pieces) break;
      first_item += pieces;
      ++c;
    }
    if (c >= C) break;
    const int piece = item - first_item;
    const int b = offs[c] + piece * FP_PIECE, e = min(offs[c + 1], b + FP_PIECE), n = e - b;
    if (pieces == 1 && n <= 1) {  // a singleton: its member, whatever its coordinates (an empty cluster: zeros)
      if (threadIdx.x == 0) {
        const float4 p = n ? __ldg(src + idx[b]) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        reinterpret_cast<float4*>(boxes + (size_t)c * 8)[0] = make_float4(p.x, p.y, p.z, 0.0f);
        reinterpret_cast<float4*>(boxes + (size_t)c * 8)[1] = make_float4(p.x, p.y, p.z, 0.0f);
        if (n) stage[b] = idx[b];
        count[c] = n;
      }
      continue;
    }
    __syncthreads();  // (shared state of the previous item)
    fp_shared_reset(s);
    BoxKeys bk;
    box_init(bk);
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      const int i = idx[b + j];
      const float4 p = __ldg(src + i);
      if (pieces == 1) box_add(bk, p);
      buf[j] = make_float4(p.x, p.y, __int_as_float(i), 0.0f);
    }
    __syncthreads();
    if (pieces == 1) box_finish(bk, s.box, boxes + (size_t)c * 8);
    const int m = (n >= 16) ? octagon_filter(buf, n, s.sel, &s.count) : n;
    const int h = hull_of(buf, m, st, stage + b, &s.h);
    if (threadIdx.x == 0) {
      if (pieces == 1) count[c] = h;
      else pcount[b] = h;
    }
  }
}

__global__ void __launch_bounds__(FP_THREADS, 1)
    k_fp_combine(FootprintArgs a, int cap) {
  extern __shared__ __align__(16) unsigned char fp_smem[];
  float4* sbuf = reinterpret_cast<float4*>(fp_smem);
  int* sst = reinterpret_cast<int*>(fp_smem + (size_t)FP_PIECE * sizeof(float4));
  __shared__ FpShared s;
  const int f = blockIdx.y;
  const int C = a.n_clusters[f];
  const float4* src = a.in + (size_t)f * a.in_stride;
  const int* offs = a.offsets + (size_t)f * (cap + 1);
  const int* idx = a.indices + (size_t)f * cap;
  float* boxes = a.boxes + (size_t)f * cap * 8;
  int* count = a.hull_count + (size_t)f * (cap + 1);
  int* stage = a.stage + (size_t)f * cap;
  int* pcount = a.hull_indices + (size_t)f * cap;
  int big = 0;  // multi-piece clusters seen so far; block k takes every gridDim.x-th, starting at the k-th
  for (int c = 0; c < C; ++c) {
    const int b = offs[c], n = offs[c + 1] - b;
    if (n <= FP_PIECE) continue;
    if (big++ % gridDim.x != blockIdx.x) continue;
    __syncthreads();
    fp_shared_reset(s);
    __syncthreads();
    BoxKeys bk;
    box_init(bk);
    for (int j = threadIdx.x; j < n; j += blockDim.x) box_add(bk, __ldg(src + idx[b + j]));
    box_finish(bk, s.box, boxes + (size_t)c * 8);
    int total = 0;
    for (int q = b; q < b + n; q += FP_PIECE) total += pcount[q];
    // the union of the piece hulls: in shared memory when it fits, else in the cluster's slots of the global scratch
    const bool fits = total <= FP_PIECE;
    float4* buf = fits ? sbuf : a.work + (size_t)f * cap + b;
    int* st = fits ? sst : pcount + b;  // (the piece sizes are read by then: the chain's stack takes their slots)
    int pos = 0;
    for (int q = b; q < b + n; q += FP_PIECE) {
      const int k = pcount[q];
      for (int j = threadIdx.x; j < k; j += blockDim.x) {
        const int i = stage[q + j];
        const float4 p = __ldg(src + i);
        buf[pos + j] = make_float4(p.x, p.y, __int_as_float(i), 0.0f);
      }
      pos += k;
    }
    __syncthreads();
    const int h = hull_of(buf, total, st, stage + b, &s.h);
    if (threadIdx.x == 0) count[c] = h;
  }
}

// one block per frame: exclusive scan of the hull sizes, then every cluster's staged vertices to its CSR slots
__global__ void __launch_bounds__(1024)
    k_fp_csr(FootprintArgs a, int cap) {
  __shared__ int warp_sum[32];
  __shared__ int carry;
  const int f = blockIdx.x;
  const int C = a.n_clusters[f];
  const int* offs = a.offsets + (size_t)f * (cap + 1);
  const int* count = a.hull_count + (size_t)f * (cap + 1);
  const int* stage = a.stage + (size_t)f * cap;
  int* hoff = a.hull_offsets + (size_t)f * (cap + 1);
  int* hidx = a.hull_indices + (size_t)f * cap;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < C; base += blockDim.x) {
    const int c = base + threadIdx.x;
    const int v = c < C ? count[c] : 0;
    int incl = v;
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += up;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      int w = warp_sum[lane];
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(FULL, w, o);
        if (lane >= o) w += up;
      }
      warp_sum[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const int before = carry + (warp ? warp_sum[warp - 1] : 0);
    if (c < C) hoff[c] = before + incl - v;
    __syncthreads();
    if (threadIdx.x == 0) carry += warp_sum[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    hoff[C] = carry;
    a.n_hull[f] = carry;
  }
  __syncthreads();
  for (int c = warp; c < C; c += blockDim.x >> 5) {
    const int o = hoff[c], k = count[c], b = offs[c];
    for (int j = lane; j < k; j += 32) hidx[o + j] = stage[b + j];
  }
}

}  // namespace

cudaError_t run_footprints(const Ctx& c, const FootprintArgs& a) {
  // (the shared-memory opt-in is a property of the current device's context: set on every call)
  cudaError_t e = cudaFuncSetAttribute(k_fp_piece, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FP_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_fp_combine, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FP_SMEM);
  if (e != cudaSuccess) return e;
  KL(c, "k_fp_piece", k_fp_piece<<<dim3(FP_GRID, c.B), FP_THREADS, FP_SMEM, c.stream>>>(a, c.cap));
  count_launch(c);
  if (c.grid_cap > FP_PIECE) {  // some cluster may be larger than one piece
    KL(c, "k_fp_combine", k_fp_combine<<<dim3(FP_COMBINE_GRID, c.B), FP_THREADS, FP_SMEM, c.stream>>>(a, c.cap));
    count_launch(c);
  }
  KL(c, "k_fp_csr", k_fp_csr<<<c.B, 1024, 0, c.stream>>>(a, c.cap));
  count_launch(c);
  return cudaGetLastError();
}

}  // namespace pcop
