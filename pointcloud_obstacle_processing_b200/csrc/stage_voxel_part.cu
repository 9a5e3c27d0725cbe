// Fused crop + VoxelGrid, partition variant (reference: the crop of od.cpp:195-215 followed by downsample_cloud
// od.cpp:271-296 -> pcl::VoxelGrid::applyFilter, SURVEY 8a-1/8a-2).  Same composite key as stage_voxel_fused.cu
// ((F_z - B_z) * ny * nx + (F_y - B_y) * nx + (F_x - B_x), the lexicographic order PCL's own keys have), but the
// global four-pass LSD sort of (key, index) pairs is replaced by ONE partition pass on the key's top bits and a
// block-local direct-address step on the low bits:
//
//   k_vp_hist      crop predicate + key of every point; per-(chunk, bucket) counts (bucket = key >> S, <= 16384 buckets
//                  per frame, 16-bit shared-memory counters), min/max of the survivors, the NaN-y/z flag;
//   k_vp_scan      per frame: bucket starts (exclusive scan), per-chunk offsets inside each bucket, M, and the work
//                  list of the reduce kernel: consecutive non-empty buckets are grouped greedily up to 2048 elements
//                  or the bitmap's range (262144 keys);
//   k_vp_scatter   second read of the input: every survivor goes to a slot of its (chunk, bucket) range -- slot taken
//                  with a shared-memory atomic -- as {x, y, z, original index};
//   k_vp_reduce    one block per group (<= 2048 elements), everything in shared memory: a bitmap over the group's key
//                  range gives every voxel its rank (popcount prefix) -- i.e. its sorted position, without sorting; a
//                  counting pass groups the elements by voxel; every element finds its place inside its voxel's run by
//                  counting the smaller original indices (runs are ~2 points); one thread per voxel then sums its run
//                  sequentially (PCL's order: ORACLE CHOICE "ascending original index"), divides by the float count and
//                  writes the centroid at (voxels of earlier groups: decoupled look-back) + rank.
//
// Per survivor the kernels issue ~150 instructions where the LSD path issues ~560, and the survivors make one round
// trip through HBM instead of four.  The order inside a bucket range depends on the atomics, but nothing observable
// does: every voxel's points are put in ascending original index before they are summed.
//
// Declined frames (internal flags, the host repeats the wave): a survivor with a NaN y or z (bit 0: generic path, as
// in stage_voxel_fused.cu), a bucket above 2048 points (bit 1: LSD path), more groups than the launch covered (bit 2:
// this path again with the worst-case grid).
#include <cmath>
#include <cstddef>
#include <cstdlib>

#include "internal.cuh"
#include "primitives.cuh"

namespace pcop {
#ifdef PCOP_VP_DEBUG_CLK
// phase timestamps of one block in [0, 10); [12, 16): groups, groups on the binary search, groups of more than 64
// buckets, elements, summed over the blocks since the last read (tools/vp_phases.py)
__device__ long long g_vp_reduce_clk[16];
#define VP_CLK(k)                                                                          \
  do {                                                                                     \
    if (blockIdx.x == 5 && blockIdx.y == 20 && threadIdx.x == 0) g_vp_reduce_clk[k] = clock64(); \
  } while (0)
#else
#define VP_CLK(k) \
  do {            \
  } while (0)
#endif

namespace {

constexpr int VP_THREADS = 256;
constexpr int VP_WARPS = VP_THREADS / 32;
constexpr int VP_NB_MAX = 16384;        // buckets per frame
constexpr int VP_MAX_CHUNKS = 8;        // histogram / scatter blocks per frame
constexpr int VP_EMAX = 2048;           // elements per group (and per bucket)
constexpr int VPR_THREADS = 512;        // reduce kernel: 16 warps per group, 4 elements per thread, all kept in registers
constexpr int VPR_WARPS = VPR_THREADS / 32;
constexpr int VP_EPT = VP_EMAX / VPR_THREADS;
constexpr int VP_BITMAP_WORDS = 8192;   // 262144 keys per group (128 buckets at S = 11)
constexpr int VP_KMAX = 256;            // buckets per group (<= VP_BITMAP_WORDS * 32 >> S)
constexpr int VP_SCAN_THREADS = 512;
constexpr int VP_SCAN_WARPS = VP_SCAN_THREADS / 32;
constexpr int VP_MAX_ROUNDS = VP_NB_MAX / 32;

__device__ __forceinline__ bool vp_keep(const float4 p, const VoxFusedPlan& pl) {
  // od.cpp:197-199, literal: drop iff isnan(x) || x<x_min || x>x_max || z<z_min || z>z_max || y<y_min || y>y_max
  return !((p.x != p.x) || p.x < pl.lim[0] || p.x > pl.lim[1] || p.z < pl.lim[4] || p.z > pl.lim[5] || p.y < pl.lim[2] ||
           p.y > pl.lim[3]);
}
__device__ __forceinline__ uint32_t vp_key(float x, float y, float z, const VoxFusedPlan& pl) {
  const int cx = __float2int_rz(floorf(fmul(x, pl.inv))) - pl.b0[0];
  const int cy = __float2int_rz(floorf(fmul(y, pl.inv))) - pl.b0[1];
  const int cz = __float2int_rz(floorf(fmul(z, pl.inv))) - pl.b0[2];
  return (uint32_t)cx + pl.nx * ((uint32_t)cy + pl.ny * (uint32_t)cz);
}
// chunk c of a frame of n points: [i0, i1), multiples of 4 * VP_THREADS so that the unrolled loops stay aligned
// (a chunk holds fewer than 65536 points: the per-chunk counters are 16 bits wide, see vox_part_plan)
__device__ __forceinline__ void vp_chunk(int n, int chunks, int c, int& i0, int& i1) {
  const int cs = cdiv(cdiv(n, chunks), 4 * VP_THREADS) * (4 * VP_THREADS);
  i0 = min(c * cs, n);
  i1 = min(i0 + cs, n);
}

// Per (frame, chunk) the histogram kernel leaves a record of VP_CHUNK_TAIL words behind the chunk's counters: min / max
// of its survivors (6 floats) and its NaN-y/z flag.  The scan kernel combines the chunks, so nothing has to be zeroed or
// initialised before the histogram runs (round 2 first spent a launch per wave on that).
constexpr int VP_CHUNK_TAIL = 8;

template <bool NEED_MINMAX>
__global__ void __launch_bounds__(VP_THREADS)
    k_vp_hist(const float4* __restrict__ in, size_t in_stride, const int* __restrict__ n_in, VoxFusedPlan pl,
              uint32_t* __restrict__ ghist, int chunks) {
  const int c = blockIdx.x, f = blockIdx.y;
  extern __shared__ uint32_t vp_sh[];  // [nb_pad / 2]: two 16-bit counters per word
  __shared__ float shmm[VP_WARPS][6];
  const int nwords = pl.nb_pad >> 1;
  for (int w = threadIdx.x; w < nwords; w += VP_THREADS) vp_sh[w] = 0u;
  __syncthreads();
  const int n = n_in[f];
  int i0, i1;
  vp_chunk(n, chunks, c, i0, i1);
  const float4* src = in + (size_t)f * in_stride;
  float mn[3] = {3.402823466e+38f, 3.402823466e+38f, 3.402823466e+38f};
  float mx[3] = {-3.402823466e+38f, -3.402823466e+38f, -3.402823466e+38f};
  bool odd = false;  // a survivor whose y or z is not finite
  for (int b0 = i0 + threadIdx.x; b0 < i1; b0 += 4 * VP_THREADS) {
    float4 p[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = b0 + u * VP_THREADS;
      const float qnan = __uint_as_float(0x7fc00000u);
      p[u] = (i < i1) ? __ldg(src + i) : make_float4(qnan, 0.f, 0.f, 0.f);  // (a NaN x is dropped by the predicate)
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (vp_keep(p[u], pl)) {
        odd = odd || !(fabsf(p[u].y) <= 3.0e38f) || !(fabsf(p[u].z) <= 3.0e38f);
        if (NEED_MINMAX) {
          const float v[3] = {p[u].x, p[u].y, p[u].z};
#pragma unroll
          for (int a = 0; a < 3; ++a) {  // compare-based: NaN never updates (oracle voxel_setup)
            if (v[a] < mn[a]) mn[a] = v[a];
            if (v[a] > mx[a]) mx[a] = v[a];
          }
        }
        // (the clamp only matters for NaN y / z survivors, whose frame is declined anyway)
        const uint32_t bucket = min(vp_key(p[u].x, p[u].y, p[u].z, pl) >> pl.part_shift, (uint32_t)pl.nb - 1u);
        atomicAdd(&vp_sh[bucket >> 1], 1u << ((bucket & 1u) * 16u));
      }
    }
  }
  const int any_odd = __syncthreads_or(odd ? 1 : 0);
  uint32_t* gh = ghist + ((size_t)f * chunks + c) * (nwords + VP_CHUNK_TAIL);
  if (NEED_MINMAX) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {
        mn[a] = fminf(mn[a], __shfl_xor_sync(FULL, mn[a], o));
        mx[a] = fmaxf(mx[a], __shfl_xor_sync(FULL, mx[a], o));
      }
    }
    if (lane_id() == 0) {
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        shmm[warp_id()][a] = mn[a];
        shmm[warp_id()][3 + a] = mx[a];
      }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
      const int a = threadIdx.x;
      float v = shmm[0][a];
      for (int w = 1; w < VP_WARPS; ++w) v = (a < 3) ? fminf(v, shmm[w][a]) : fmaxf(v, shmm[w][a]);
      gh[nwords + a] = __float_as_uint(v);
    }
  }
  if (threadIdx.x == 6) gh[nwords + 6] = any_odd ? 1u : 0u;
  for (int w = threadIdx.x; w < nwords; w += VP_THREADS) gh[w] = vp_sh[w];
}

// PCL's voxel frame from the min/max of the survivors (same arithmetic as stage_voxel.cu's k_voxel_setup; the host
// has proven that the overflow guard cannot fire)
__device__ void vp_setup_one(const float (&mnv)[3], const float (&mxv)[3], float leaf, VoxelFrame* __restrict__ vf, int f) {
  VoxelFrame v;
  v.inv = fdiv(1.0f, leaf);
  unsigned div_b[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    v.min_b[a] = cvt_f2i(floorf(fmul(mnv[a], v.inv)));
    const int max_b = cvt_f2i(floorf(fmul(mxv[a], v.inv)));
    div_b[a] = (unsigned)max_b - (unsigned)v.min_b[a] + 1u;
  }
  v.overflow = 0;
  v.mul1 = div_b[0];
  v.mul2 = div_b[0] * div_b[1];
  vf[f] = v;
}

__device__ __forceinline__ unsigned warp_incl_scan(unsigned v) {
  const int lane = lane_id();
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned up = __shfl_up_sync(FULL, v, o);
    if (lane >= o) v += up;
  }
  return v;
}

// warp 0: exclusive scan, in place, of the n <= 32 * PER entries of `a` (shared memory); returns the total in every lane
template <int PER>
__device__ __forceinline__ unsigned warp0_excl_scan(uint32_t* a, int n) {
  const int lane = lane_id();
  unsigned v[PER];
  unsigned sum = 0u;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int i = lane * PER + j;
    v[j] = (i < n) ? a[i] : 0u;
    sum += v[j];
  }
  const unsigned incl = warp_incl_scan(sum);
  unsigned run = incl - sum;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int i = lane * PER + j;
    if (i < n) a[i] = run;
    run += v[j];
  }
  return __shfl_sync(FULL, incl, 31);
}

// per-(chunk, bucket) 16-bit counts of the four buckets b0 .. b0 + 3 (b0 % 4 == 0: one 8-byte load per chunk)
__device__ __forceinline__ void vp_unpack4(const uint2 w, unsigned (&v)[4]) {
  v[0] = w.x & 0xffffu;
  v[1] = w.x >> 16;
  v[2] = w.y & 0xffffu;
  v[3] = w.y >> 16;
}
// t[k] = the buckets' totals over the chunks
__device__ __forceinline__ void vp_bucket_totals4(const unsigned short* gh16, size_t chunk_stride16, int chunks, int b0,
                                                  unsigned (&t)[4]) {
#pragma unroll
  for (int k = 0; k < 4; ++k) t[k] = 0u;
#pragma unroll
  for (int c = 0; c < VP_MAX_CHUNKS; ++c) {
    if (c < chunks) {
      unsigned v[4];
      vp_unpack4(*reinterpret_cast<const uint2*>(gh16 + (size_t)c * chunk_stride16 + b0), v);
#pragma unroll
      for (int k = 0; k < 4; ++k) t[k] += v[k];
    }
  }
}

__global__ void __launch_bounds__(VP_SCAN_THREADS, 2)
    k_vp_scan(const uint32_t* __restrict__ ghist, uint32_t* __restrict__ chunk_start, unsigned short* __restrict__ ne_bucket,
              uint32_t* __restrict__ ne_start,
              uint2* __restrict__ grec, int* __restrict__ n_groups, int* __restrict__ n_crop,
              uint32_t* __restrict__ flags, uint32_t* __restrict__ warnings, float leaf, VoxelFrame* __restrict__ vf,
              VoxFusedPlan pl, int chunks, int want_keys, int gmax, int gstride) {
  const int f = blockIdx.x, tid = threadIdx.x, lane = lane_id(), warp = warp_id();
  __shared__ uint32_t s_rt[VP_MAX_ROUNDS / 4 + 1];  // elements before each round of 128 buckets
  __shared__ uint32_t s_rn[VP_MAX_ROUNDS / 4 + 1];  // non-empty buckets before each round
  __shared__ unsigned s_total[2];
  const int nwords = pl.nb_pad >> 1;
  const uint32_t* gh = ghist + (size_t)f * chunks * (nwords + VP_CHUNK_TAIL);
  const size_t chunk_stride16 = 2 * (size_t)(nwords + VP_CHUNK_TAIL);
  const unsigned short* gh16 = reinterpret_cast<const unsigned short*>(gh);
  if (tid == 0) {  // the chunks' min / max and NaN flags (see VP_CHUNK_TAIL); this is also where the frame's flag word starts
    float mnv[3] = {3.402823466e+38f, 3.402823466e+38f, 3.402823466e+38f};
    float mxv[3] = {-3.402823466e+38f, -3.402823466e+38f, -3.402823466e+38f};
    uint32_t odd = 0u;
    for (int c = 0; c < chunks; ++c) {
      const uint32_t* tail = gh + (size_t)c * (nwords + VP_CHUNK_TAIL) + nwords;
      odd |= tail[6];
      if (want_keys) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          mnv[a] = fminf(mnv[a], __uint_as_float(tail[a]));
          mxv[a] = fmaxf(mxv[a], __uint_as_float(tail[3 + a]));
        }
      }
    }
    flags[f] = odd;
    if (warnings) warnings[f] = 0u;
    if (want_keys) vp_setup_one(mnv, mxv, leaf, vf, f);
  }
  __syncthreads();  // (the flag word is written before anyone ORs into it)
  uint32_t* cs_out = chunk_start + (size_t)f * chunks * pl.nb_pad;
  unsigned short* ne_out = ne_bucket + (size_t)f * VP_NB_MAX;
  uint32_t* ns_out = ne_start + (size_t)f * (VP_NB_MAX + 1);  // element start of every non-empty bucket, then M
  const int nrounds = (pl.nb_pad + 127) >> 7;  // rounds of 128 buckets: four consecutive buckets per lane
  // ---- pass 1: per round, elements and non-empty buckets ----------------------------------------------------------------
  bool too_big = false;
  for (int r = warp; r < nrounds; r += VP_SCAN_WARPS) {
    const int b0 = 128 * r + 4 * lane;
    unsigned t[4] = {0u, 0u, 0u, 0u};
    if (b0 < pl.nb_pad) vp_bucket_totals4(gh16, chunk_stride16, chunks, b0, t);  // (buckets past nb hold zeros)
    unsigned nz = 0u;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      too_big = too_big || t[k] > (unsigned)VP_EMAX;
      nz += (t[k] != 0u) ? 1u : 0u;
    }
    const unsigned sum = __reduce_add_sync(FULL, t[0] + t[1] + t[2] + t[3]);
    const unsigned ne = __reduce_add_sync(FULL, nz);
    if (lane == 0) {
      s_rt[r] = sum;
      s_rn[r] = ne;
    }
  }
  if (too_big) atomicOr(&flags[f], 2u);
  __syncthreads();
  if (warp == 0) {
    const unsigned m = warp0_excl_scan<(VP_MAX_ROUNDS / 4 + 31) / 32>(s_rt, nrounds);
    const unsigned ne = warp0_excl_scan<(VP_MAX_ROUNDS / 4 + 31) / 32>(s_rn, nrounds);
    if (lane == 0) {
      s_total[0] = m;
      s_total[1] = ne;
      n_crop[f] = (int)m;
    }
  }
  __syncthreads();
  const unsigned M = s_total[0];
  const int NE = (int)s_total[1];
  // ---- pass 2: bucket starts, per-chunk offsets inside each bucket, the list of non-empty buckets -----------------------
  for (int r = warp; r < nrounds; r += VP_SCAN_WARPS) {
    const int b0 = 128 * r + 4 * lane;
    unsigned t[4] = {0u, 0u, 0u, 0u};
    const bool in_range = b0 < pl.nb_pad;
    if (in_range) vp_bucket_totals4(gh16, chunk_stride16, chunks, b0, t);
    const unsigned mine = t[0] + t[1] + t[2] + t[3];
    const unsigned incl = warp_incl_scan(mine);
    unsigned nz = 0u;
#pragma unroll
    for (int k = 0; k < 4; ++k) nz += (t[k] != 0u) ? 1u : 0u;
    const unsigned nz_incl = warp_incl_scan(nz);
    unsigned start[4];  // the buckets' starts (buckets past nb are empty: start = M)
    start[0] = s_rt[r] + incl - mine;
    start[1] = start[0] + t[0];
    start[2] = start[1] + t[1];
    start[3] = start[2] + t[2];
    if (in_range) {
      unsigned run[4] = {start[0], start[1], start[2], start[3]};
#pragma unroll
      // absolute first slot of every (chunk, bucket) range, for the scatter kernel (the counts are read a second time --
      // cache hits -- rather than kept: 32 registers less, two blocks per SM)
      for (int c = 0; c < chunks; ++c) {
        *reinterpret_cast<uint4*>(cs_out + (size_t)c * pl.nb_pad + b0) = make_uint4(run[0], run[1], run[2], run[3]);
        unsigned v[4];
        vp_unpack4(*reinterpret_cast<const uint2*>(gh16 + (size_t)c * chunk_stride16 + b0), v);
#pragma unroll
        for (int k = 0; k < 4; ++k) run[k] += v[k];
      }
      unsigned o = s_rn[r] + nz_incl - nz;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (t[k] != 0u) {
          ne_out[o] = (unsigned short)(b0 + k);
          ns_out[o] = start[k];
          ++o;
        }
      }
    }
  }
  if (tid == 0) ns_out[NE] = M;
  __syncthreads();  // (the block's global writes are visible to the block)
  // ---- groups (warp 0): greedy -- a group takes consecutive non-empty buckets while it stays within VP_EMAX elements and
  // K buckets (the bitmap's key range), so most groups are nearly full.  32 ordinals per step: the lanes hold the END
  // positions of ordinals o .. o + 31; the group that starts at position gs / ordinal go closes in front of the first of
  // them that would break a limit (the scan's global writes above are visible: __syncthreads). ---------------------------------------------------------------------------------------
  if (warp != 0) return;
  const int K = min(VP_KMAX, (VP_BITMAP_WORDS * 32) >> pl.part_shift);
  uint2* gf = grec + (size_t)f * gstride;  // {element start, first non-empty ordinal} of every group, then {M, NE}
  int ng = 0;
  if (NE > 0) {
    unsigned gs = 0u;  // element start of the open group
    int go = 0;        // its first ordinal
    if (lane == 0) gf[0] = make_uint2(0u, 0u);
    ng = 1;
    for (int base = 0; base < NE; base += 32) {
      const int o = base + lane;
      const unsigned st = (o < NE) ? ns_out[o] : 0u, en = (o < NE) ? ns_out[o + 1] : 0u;
      while (true) {
        // (o > go: the bucket that opens a group always fits -- a larger one has already declined the frame)
        const bool breaks = (o < NE) && (o > go) && (en - gs > (unsigned)VP_EMAX || o - go >= K);
        const unsigned m = __ballot_sync(FULL, breaks);
        if (!m) break;
        const int l = __ffs(m) - 1;  // ordinal base + l opens the next group
        go = base + l;
        gs = __shfl_sync(FULL, st, l);
        if (lane == 0 && ng < gmax) gf[ng] = make_uint2(gs, (unsigned)go);
        ++ng;
      }
    }
  }
  if (lane == 0) {
    n_groups[f] = ng;
    if (ng <= gmax) gf[ng] = make_uint2(M, (unsigned)NE);
    else atomicOr(&flags[f], 4u);
  }
}

// (512 threads: the kernel waits on its input loads -- 60 % of its stall samples -- and the 50 KB of cursors allow four
// blocks per SM, so the wider block doubles the loads in flight)
constexpr int VPS_THREADS = 512;
__global__ void __launch_bounds__(VPS_THREADS)
    k_vp_scatter(const float4* __restrict__ in, size_t in_stride, const int* __restrict__ n_in, VoxFusedPlan pl,
                 const uint32_t* __restrict__ chunk_start, const uint32_t* __restrict__ flags, float4* __restrict__ part,
                 int cap, int chunks) {
  const int c = blockIdx.x, f = blockIdx.y;
  if (flags[f]) return;  // a declined frame: the wave is repeated by another path
  extern __shared__ uint32_t vp_sh[];  // [nb_pad] next free slot of every (this chunk, bucket) range
  const uint32_t* cs = chunk_start + ((size_t)f * chunks + c) * pl.nb_pad;
  for (int b = threadIdx.x; b < pl.nb_pad; b += VPS_THREADS) vp_sh[b] = cs[b];
  __syncthreads();
  const int n = n_in[f];
  int i0, i1;
  vp_chunk(n, chunks, c, i0, i1);
  const float4* src = in + (size_t)f * in_stride;
  float4* dst = part + (size_t)f * cap;
  // software-pipelined: the next four loads are in flight while the current four points are placed
  const float qnan = __uint_as_float(0x7fc00000u);
  float4 nxt[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int i = i0 + threadIdx.x + u * VPS_THREADS;
    nxt[u] = (i < i1) ? __ldg(src + i) : make_float4(qnan, 0.f, 0.f, 0.f);
  }
  for (int b0 = i0 + threadIdx.x; b0 < i1; b0 += 4 * VPS_THREADS) {
    float4 p[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      p[u] = nxt[u];
      const int i = b0 + (4 + u) * VPS_THREADS;
      nxt[u] = (i < i1) ? __ldg(src + i) : make_float4(qnan, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (vp_keep(p[u], pl)) {
        const uint32_t bucket = vp_key(p[u].x, p[u].y, p[u].z, pl) >> pl.part_shift;
        const uint32_t pos = atomicAdd(&vp_sh[bucket], 1u);
        dst[pos] = make_float4(p[u].x, p[u].y, p[u].z, __int_as_float(b0 + u * VPS_THREADS));
      }
    }
  }
}

constexpr int VP_ORD_TAB = 4096;  // span of bucket ids a group may cover for the direct bucket -> ordinal table

struct alignas(16) VpReduceSmem {
  union {
    struct {                                    // setup .. pass 2
      uint32_t bitmap[VP_BITMAP_WORDS];         // one bit per key of the group's range
      unsigned short wprefix[VP_BITMAP_WORDS];  // voxels before each bitmap word, inside its round of 128 words
    } k;
    struct {                                    // pass 3 .. sums (first written after the last read of `k`)
      int sidx[VP_EMAX];                        // original indices, grouped by voxel (any order inside a run)
      float sx[VP_EMAX], sy[VP_EMAX], sz[VP_EMAX];  // coordinates, grouped by voxel, ascending original index inside a run
    } e;
  };
  uint32_t rtot[VP_BITMAP_WORDS / 128];     // voxels in each round of 128 bitmap words
  uint32_t start[VP_EMAX + 4];              // per voxel: point count, then first position of its run
  uint32_t srt[VP_EMAX / 128];              // run lengths in each round of 128 voxels
  uint32_t bkt_start[VP_KMAX + 1];          // element start of the group's buckets (binary-search groups only)
  unsigned char ord_tab[VP_ORD_TAB];        // bucket id - first bucket id -> ordinal inside the group
  unsigned vbase;
};

static_assert(offsetof(VpReduceSmem, start) % 16 == 0 && offsetof(VpReduceSmem, k.wprefix) % 8 == 0, "vector accesses");
static_assert(VP_BITMAP_WORDS / 128 <= 64 && VP_EMAX / 128 <= VPR_WARPS, "the block scans: two rounds per lane, one per warp");

// exclusive scan of four consecutive values per lane over a round of 128 values: returns the lane's exclusive prefix
// inside the round (of its first value) and the round's total (all lanes)
__device__ __forceinline__ unsigned vp_round_scan(const unsigned (&c)[4], unsigned& total) {
  const unsigned mine = c[0] + c[1] + c[2] + c[3];
  const unsigned incl = warp_incl_scan(mine);
  total = __shfl_sync(FULL, incl, 31);
  return incl - mine;
}

template <bool WITH_KEYS>
__global__ void __launch_bounds__(VPR_THREADS, 3)
    k_vp_reduce(const float4* __restrict__ part, const uint32_t* __restrict__ ne_start,
                const unsigned short* __restrict__ ne_bucket, const uint2* __restrict__ grec,
                const int* __restrict__ n_groups, const uint32_t* __restrict__ flags, VoxFusedPlan pl,
                const VoxelFrame* __restrict__ vf, float4* __restrict__ out, uint32_t* __restrict__ out_keys,
                int* __restrict__ n_out, unsigned* __restrict__ desc, int cap, int gstride) {
  const int f = blockIdx.x, g = blockIdx.y;  // frame-major dispatch (shallow look-back, see stage_voxel_fused.cu)
  const int tid = threadIdx.x, lane = lane_id(), warp = warp_id();
  // (four independent loads; the records of a frame that has fewer groups are stale but harmless)
  const int ng = n_groups[f];
  const uint32_t declined = flags[f];
  const uint2 r0 = grec[(size_t)f * gstride + g], r1 = grec[(size_t)f * gstride + g + 1];
  if (declined || g >= ng) {  // a declined frame, or no such group (ng == 0: no survivors)
    if (g == 0 && tid == 0) n_out[f] = 0;
    return;
  }
  VP_CLK(0);
  extern __shared__ __align__(16) unsigned char vp_raw[];
  VpReduceSmem& sm = *reinterpret_cast<VpReduceSmem*>(vp_raw);
  const uint32_t e0 = r0.x;
  const int E = (int)(r1.x - r0.x);  // <= VP_EMAX
  const int o0 = (int)r0.y, KB = (int)(r1.y - r0.y);
  const float4* src = part + (size_t)f * cap + e0;
  // the thread's elements ({x, y, z, original index}) stay in registers until they are staged in sorted order
  float4 p[VP_EPT];
#pragma unroll
  for (int k = 0; k < VP_EPT; ++k) {
    const int e = tid + k * VPR_THREADS;
    p[k] = (e < E) ? __ldg(src + e) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int S = pl.part_shift;
  const int wpb = (1 << S) >> 5;  // bitmap words per bucket (S >= 5)
  const int nwords = KB * wpb;    // <= VP_BITMAP_WORDS
  // every thread reads the group's first and last bucket ids itself: the table is filled without a barrier in front
  const unsigned short* nb = ne_bucket + (size_t)f * VP_NB_MAX + o0;
  const int b_first = nb[0];
  const bool direct = (int)nb[KB - 1] - b_first < VP_ORD_TAB;  // (else: binary search on the bucket starts)
  if (direct) {
    if (tid < KB) sm.ord_tab[nb[tid] - b_first] = (unsigned char)tid;
  } else if (tid <= KB) {
    sm.bkt_start[tid] = ne_start[(size_t)f * (VP_NB_MAX + 1) + o0 + tid];  // (entry NE holds M)
  }
  for (int w = 4 * tid; w < nwords; w += 4 * VPR_THREADS)  // (whole uint4s: the scans read them as such)
    *reinterpret_cast<uint4*>(&sm.k.bitmap[w]) = make_uint4(0u, 0u, 0u, 0u);
  for (int v = 4 * tid; v < E + 4; v += 4 * VPR_THREADS) *reinterpret_cast<uint4*>(&sm.start[v]) = make_uint4(0u, 0u, 0u, 0u);
#ifdef PCOP_VP_DEBUG_CLK
  if (tid == 0) {
    atomicAdd(reinterpret_cast<unsigned long long*>(&g_vp_reduce_clk[12]), 1ull);
    atomicAdd(reinterpret_cast<unsigned long long*>(&g_vp_reduce_clk[13]), direct ? 0ull : 1ull);
    atomicAdd(reinterpret_cast<unsigned long long*>(&g_vp_reduce_clk[14]), KB > 64 ? 1ull : 0ull);
    atomicAdd(reinterpret_cast<unsigned long long*>(&g_vp_reduce_clk[15]), (unsigned long long)E);
  }
#endif
  __syncthreads();
  VP_CLK(1);

  // ---- pass 1: every element sets the bit of its key ---------------------------------------------------------------------
  uint32_t slot[VP_EPT];  // position of the element's key in the bitmap; later (voxel rank << 16) | place inside its run
#pragma unroll
  for (int k = 0; k < VP_EPT; ++k) {
    const int e = tid + k * VPR_THREADS;
    slot[k] = 0u;
    if (e < E) {
      const uint32_t key = vp_key(p[k].x, p[k].y, p[k].z, pl);
      int ord;
      if (direct) {
        ord = sm.ord_tab[(int)(key >> S) - b_first];
      } else {  // the last bucket that starts at or before the element's position
        int lo = 0, hi = KB - 1;
        const uint32_t pos = e0 + (uint32_t)e;
        while (lo < hi) {
          const int mid = (lo + hi + 1) >> 1;
          if (sm.bkt_start[mid] <= pos) lo = mid;
          else hi = mid - 1;
        }
        ord = lo;
      }
      const uint32_t s = ((uint32_t)ord << S) | (key & ((1u << S) - 1u));
      slot[k] = s;
      atomicOr(&sm.k.bitmap[s >> 5], 1u << (s & 31u));
    }
  }
  __syncthreads();
  VP_CLK(2);
  // ---- voxel ranks: exclusive popcount prefix over the bitmap words; a warp takes a round of 128 words, four consecutive
  // words per lane (one 16-byte load) ----------------------------------------------------------------------------------------
  const int nr = cdiv(nwords, 128);  // <= 64
  for (int r = warp; r < nr; r += VPR_WARPS) {
    const int w = 128 * r + 4 * lane;
    const uint4 bw = (w < nwords) ? *reinterpret_cast<const uint4*>(&sm.k.bitmap[w]) : make_uint4(0u, 0u, 0u, 0u);  // (nwords % 4 == 0)
    const unsigned c[4] = {(unsigned)__popc(bw.x), (unsigned)__popc(bw.y), (unsigned)__popc(bw.z), (unsigned)__popc(bw.w)};
    unsigned total;
    const unsigned ex = vp_round_scan(c, total);
    if (w < nwords) {
      const unsigned a0 = ex, a1 = a0 + c[0], a2 = a1 + c[1], a3 = a2 + c[2];
      *reinterpret_cast<uint2*>(&sm.k.wprefix[w]) = make_uint2(a0 | (a1 << 16), a2 | (a3 << 16));
    }
    if (lane == 0) sm.rtot[r] = total;
  }
  __syncthreads();
  VP_CLK(3);
  // every warp scans the round totals itself (rounds 2 * lane and 2 * lane + 1 in lane `lane`) and keeps the voxels
  // before both rounds in one register (<= 2048 each); pass 2 takes a round's base from its lane by shuffle
  unsigned rbase2;
  int V;
  {
    const unsigned t0 = (2 * lane < nr) ? sm.rtot[2 * lane] : 0u, t1 = (2 * lane + 1 < nr) ? sm.rtot[2 * lane + 1] : 0u;
    const unsigned incl = warp_incl_scan(t0 + t1);
    const unsigned b0 = incl - t0 - t1;
    rbase2 = b0 | ((b0 + t0) << 16);
    V = (int)__shfl_sync(FULL, incl, 31);
  }
  unsigned* dd = desc + (size_t)f * gstride;
  if (tid == 0) st_volatile_u32(dd + g, ((g == 0) ? LB_PREFIX : LB_AGG) | (unsigned)V);  // early publish
  // ---- pass 2: a place for every element inside its voxel's run (any order), run lengths -------------------------------
#pragma unroll
  for (int k = 0; k < VP_EPT; ++k) {
    const int e = tid + k * VPR_THREADS;
    const uint32_t s = slot[k];
    const uint32_t rb = __shfl_sync(FULL, rbase2, (int)(s >> 13)) >> ((s >> 8) & 16u);  // round s >> 12
    if (e < E) {
      const uint32_t r = (rb & 0xffffu) + (uint32_t)sm.k.wprefix[s >> 5] +
                         (uint32_t)__popc(sm.k.bitmap[s >> 5] & ((1u << (s & 31u)) - 1u));
      const uint32_t j = atomicAdd(&sm.start[r], 1u);
      slot[k] = (r << 16) | j;
    }
  }
  __syncthreads();
  VP_CLK(4);
  {  // exclusive scan of the run lengths, in place: warp r takes the round of voxels 128 r .. 128 r + 127 (V <= 2048),
     // four consecutive voxels per lane
    const int vr = cdiv(V, 128);
    unsigned keep[4] = {0u, 0u, 0u, 0u};
    if (warp < vr) {
      const int v = 128 * warp + 4 * lane;
      const uint4 cw = *reinterpret_cast<const uint4*>(&sm.start[v]);  // (counts past E + 3 are stale: they only reach entries past V)
      const unsigned c[4] = {cw.x, cw.y, cw.z, cw.w};
      unsigned total;
      const unsigned ex = vp_round_scan(c, total);
      keep[0] = ex;
      keep[1] = ex + c[0];
      keep[2] = keep[1] + c[1];
      keep[3] = keep[2] + c[2];
      if (lane == 0) sm.srt[warp] = total;
    }
    // voxels of the earlier groups of this frame (decoupled look-back; the aggregates were published after the popcount,
    // the wait is on lower group ids only).  The last warp has no round unless V > 1920, so the L2 round trip hides
    // behind the run-length scan; `vbase` is read after the barriers below.
    if (warp == VPR_WARPS - 1 && g > 0) {
      unsigned excl = 0u;
      int look = g - 1;
      while (true) {
        const int idx = look - lane;
        unsigned d = LB_PREFIX;  // lanes past the first group read as "prefix 0"
        if (idx >= 0) {
          d = lookback_wait(dd + idx);
        }
        const unsigned is_prefix = __ballot_sync(FULL, (d >> 30) == 2u);
        const int first = is_prefix ? (__ffs(is_prefix) - 1) : 31;
        unsigned v = (lane <= first) ? (d & LB_VALUE) : 0u;
        v = __reduce_add_sync(FULL, v);
        excl += v;
        if (is_prefix) break;
        look -= 32;
      }
      if (lane == 0) {
        st_volatile_u32(dd + g, LB_PREFIX | (excl + (unsigned)V));
        sm.vbase = excl;
      }
    } else if (tid == 0 && g == 0) {
      sm.vbase = 0u;
    }
    __syncthreads();
    VP_CLK(5);
    if (warp < vr) {
      const unsigned base = __reduce_add_sync(FULL, (lane < warp) ? sm.srt[lane] : 0u);
      const int v = 128 * warp + 4 * lane;
      *reinterpret_cast<uint4*>(&sm.start[v]) = make_uint4(base + keep[0], base + keep[1], base + keep[2], base + keep[3]);
    }
    // (entry V is E: written above when a round holds it, the counts at V .. V + 3 being zero; here when none does)
    if (tid == 0 && (V & 127) == 0) sm.start[V] = (unsigned)E;
  }
  __syncthreads();
  VP_CLK(6);
  // ---- pass 3: original indices grouped by voxel; then every element counts the smaller indices of its run and puts its
  // coordinates at that place (runs are ~2 points; a dense blob costs its run length per element) -----------------------
#pragma unroll
  for (int k = 0; k < VP_EPT; ++k) {
    const int e = tid + k * VPR_THREADS;
    if (e < E) sm.e.sidx[sm.start[slot[k] >> 16] + (slot[k] & 0xffffu)] = __float_as_int(p[k].w);
  }
  __syncthreads();
  VP_CLK(7);
#pragma unroll
  for (int k = 0; k < VP_EPT; ++k) {
    const int e = tid + k * VPR_THREADS;
    if (e < E) {
      const uint32_t r = slot[k] >> 16;
      const int s0 = (int)sm.start[r], cnt = (int)sm.start[r + 1] - s0;
      // (a run of two needs no order: a + b == b + a; its elements keep the places they drew in pass 2)
      int rank = (int)(slot[k] & 0xffffu);
      if (cnt > 2) {
        const int mine = __float_as_int(p[k].w);
        rank = 0;
        for (int t = 0; t < cnt; ++t) rank += (sm.e.sidx[s0 + t] < mine) ? 1 : 0;
      }
      sm.e.sx[s0 + rank] = p[k].x;
      sm.e.sy[s0 + rank] = p[k].y;
      sm.e.sz[s0 + rank] = p[k].z;
    }
  }
  __syncthreads();
  VP_CLK(8);
  // ---- one thread per voxel: sequential sum of its run, centroid, stored at (voxels of the earlier groups) + rank -----
  VoxelFrame vfr;
  float fb0 = 0.f, fb1 = 0.f, fb2 = 0.f;
  if (WITH_KEYS) {
    vfr = vf[f];
    fb0 = (float)vfr.min_b[0];
    fb1 = (float)vfr.min_b[1];
    fb2 = (float)vfr.min_b[2];
  }
  const unsigned vbase = sm.vbase;
  if (g == ng - 1 && tid == 0) n_out[f] = (int)(vbase + (unsigned)V);
  constexpr int VPT = VP_EMAX / VPR_THREADS;  // voxels per thread
#pragma unroll
  for (int k = 0; k < VPT; ++k) {
    const int v = tid + k * VPR_THREADS;
    if (v < V) {
      const int s0 = (int)sm.start[v], s1 = (int)sm.start[v + 1];
      float ax = 0.0f, ay = 0.0f, az = 0.0f;
      for (int t = s0; t < s1; ++t) {
        ax = fadd(ax, sm.e.sx[t]);
        ay = fadd(ay, sm.e.sy[t]);
        az = fadd(az, sm.e.sz[t]);
      }
      const float c = (float)(s1 - s0);
      const size_t o = (size_t)f * cap + vbase + (unsigned)v;
      // (x / 1.0f == x exactly: the single-point voxels, more than half of them, skip the three divisions)
      out[o] = (s1 - s0 == 1) ? make_float4(ax, ay, az, 1.0f) : make_float4(fdiv(ax, c), fdiv(ay, c), fdiv(az, c), 1.0f);
      if (WITH_KEYS) {  // PCL's key of this voxel, from one of its points (voxel_grid.hpp: ijk = floor(p*inv) - min_b)
        const int i0 = cvt_f2i(fsub(floorf(fmul(sm.e.sx[s0], vfr.inv)), fb0));
        const int i1 = cvt_f2i(fsub(floorf(fmul(sm.e.sy[s0], vfr.inv)), fb1));
        const int i2 = cvt_f2i(fsub(floorf(fmul(sm.e.sz[s0], vfr.inv)), fb2));
        out_keys[o] = (uint32_t)i0 + (uint32_t)i1 * vfr.mul1 + (uint32_t)i2 * vfr.mul2;
      }
    }
  }
  VP_CLK(9);
}

}  // namespace

// Buckets of the partition path for a plan made by make_vox_fused_plan: S low key bits per bucket so that a frame has
// at most 2^nbits buckets, nbits = clamp(log2(max_points) - 3, 8, 14) (about 8 points per bucket on average when the
// survivors fill the box evenly; real frames are far from even, which is what the 2048-point bucket limit is for).
void vox_part_plan(VoxFusedPlan& pl, size_t max_points) {
  pl.part_ok = 0;
  if (!pl.ok) return;
  if (max_points > (size_t)VP_MAX_CHUNKS * 61440) return;  // a chunk's 16-bit counters: the LSD path takes larger frames
  int lg = 0;
  while (((size_t)1 << lg) < max_points) ++lg;
  const int nbits = std::min(14, std::max(8, lg - 3));
  const int shift = std::max(5, pl.bits - nbits);
  if (pl.bits - shift > 14 || shift > 16) return;  // too many buckets / a bucket wider than the bitmap: the LSD path
  const unsigned long long total = (unsigned long long)pl.nx * pl.ny * pl.nz;
  pl.part_shift = shift;
  pl.nb = (int)((total + (1ull << shift) - 1) >> shift);
  if (pl.nb < 1) pl.nb = 1;
  if (pl.nb > VP_NB_MAX) return;
  pl.nb_pad = (pl.nb + 31) & ~31;
  pl.part_ok = 1;
}

// histogram / scatter blocks per frame: chunks of ~24 576 points (measured: 8 / 4 / 3 chunks per 120 k-point frame 5.53 /
// 5.46 / 5.40 ms per step; fewer chunks, less per-(chunk, bucket) traffic, but fewer blocks to fill the GPU with)
// A call of a few frames cannot fill the GPU with four blocks per frame: twice the chunks (half the points per block)
// while the frames are fewer than 32 (single-frame latency: hist + scatter 54 -> 34 us).
int vox_part_chunks(int max_n, int B) {
  const int per = (B < 32) ? 12288 : 24576;
  return std::max(1, std::min(VP_MAX_CHUNKS, max_n / per));
}
// worst-case number of groups of a frame of max_n points
int vox_part_group_bound(const VoxFusedPlan& pl, int max_n) {
  const int K = std::min(VP_KMAX, (VP_BITMAP_WORDS * 32) >> pl.part_shift);
  const int ne = std::min(pl.nb, max_n);
  const long long b = 2ll * max_n / VP_EMAX + ne / K + 3;  // (two consecutive groups hold more than VP_EMAX elements or K buckets)
  return (int)std::min<long long>(b, 65535);
}
size_t vox_part_hist_elems(int B) { return (size_t)B * VP_MAX_CHUNKS * (VP_NB_MAX / 2 + VP_CHUNK_TAIL); }
size_t vox_part_start_elems(int B) { return (size_t)B * (VP_NB_MAX + 1); }
size_t vox_part_chunk_start_elems(int B) { return (size_t)B * VP_MAX_CHUNKS * VP_NB_MAX; }
size_t vox_part_bucket_elems(int B) { return (size_t)B * VP_NB_MAX; }

void run_voxel_part(const Ctx& c, const VoxelPartArgs& a) {
  const VoxFusedPlan& pl = a.plan;
  const int chunks = vox_part_chunks(c.grid_cap, c.B);
  const int gmax = std::max(1, std::min(a.group_launch, a.group_stride - 1));
  cudaMemsetAsync(a.desc, 0, (size_t)c.B * a.group_stride * sizeof(unsigned), c.stream);
  const size_t hsm = (size_t)(pl.nb_pad / 2) * sizeof(uint32_t);
  if (a.want_keys)
    KL(c, "k_vp_hist", k_vp_hist<true><<<dim3(chunks, c.B), VP_THREADS, hsm, c.stream>>>(a.in, a.in_stride, a.n_in, pl, a.ghist,
                                                                                        chunks));
  else
    KL(c, "k_vp_hist", k_vp_hist<false><<<dim3(chunks, c.B), VP_THREADS, hsm, c.stream>>>(a.in, a.in_stride, a.n_in, pl, a.ghist,
                                                                                         chunks));
  KL(c, "k_vp_scan", k_vp_scan<<<c.B, VP_SCAN_THREADS, 0, c.stream>>>(a.ghist, a.chunk_start, a.ne_bucket, a.ne_start, a.grec, a.n_groups,
                                                                      a.n_crop, a.flags, a.warnings, a.leaf, a.vf, pl, chunks,
                                                                      a.want_keys, gmax, a.group_stride));
  const size_t ssm = (size_t)pl.nb_pad * sizeof(uint32_t);  // (<= 64 KB)
  cudaFuncSetAttribute(k_vp_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssm);
  KL(c, "k_vp_scatter", k_vp_scatter<<<dim3(chunks, c.B), VPS_THREADS, ssm, c.stream>>>(a.in, a.in_stride, a.n_in, pl, a.chunk_start,
                                                                                       a.flags, a.part, c.cap, chunks));
  const size_t rsm = sizeof(VpReduceSmem);
  if (a.want_keys) {
    cudaFuncSetAttribute(k_vp_reduce<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsm);
    KL(c, "k_vp_reduce", k_vp_reduce<true><<<dim3(c.B, gmax), VPR_THREADS, rsm, c.stream>>>(
                             a.part, a.ne_start, a.ne_bucket, a.grec, a.n_groups, a.flags, pl, a.vf, a.out, a.out_keys,
                             a.n_out, a.desc, c.cap, a.group_stride));
  } else {
    cudaFuncSetAttribute(k_vp_reduce<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsm);
    KL(c, "k_vp_reduce", k_vp_reduce<false><<<dim3(c.B, gmax), VPR_THREADS, rsm, c.stream>>>(
                             a.part, a.ne_start, a.ne_bucket, a.grec, a.n_groups, a.flags, pl, a.vf, a.out, a.out_keys,
                             a.n_out, a.desc, c.cap, a.group_stride));
  }
  count_launch(c, 4);
}

}  // namespace pcop

#ifdef PCOP_VP_DEBUG_CLK
extern "C" int pcop_debug_vp_reduce_cycles(long long* out16) {
  cudaError_t e = cudaMemcpyFromSymbol(out16, pcop::g_vp_reduce_clk, sizeof(long long) * 16);
  static const long long zero[4] = {0, 0, 0, 0};
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(pcop::g_vp_reduce_clk, zero, sizeof(zero), sizeof(long long) * 12);
  return (int)e;
}
#endif
