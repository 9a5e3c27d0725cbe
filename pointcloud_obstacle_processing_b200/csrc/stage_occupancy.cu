// Occupancy grid of the reference node (od.cpp:134-157 + 175-269, 467-672, 817-833).
//
// Initial data set (build_initial_occupancy_grid_dataset, od.cpp:175-269):
//   k_occ_count          one frame: every crop survivor adds 1 to its cell (64-bit global atomics)
//   k_occ_count_wave     every frame of a wave, one block per (chunk, frame): the same predicate and cell search into
//                        a shared-memory histogram flushed into the frame's int32 counts; the counter width follows
//                        the grid size only (see occ_count_mode), grids too large for shared memory count in global
//                        memory directly
//   k_occ_finish         one block per (row, frame): integer row average (64-bit sum), then the threshold
// Shadow casting + obstacle marking (traceShadow od.cpp:467-538, calculate_shadow_cast od.cpp:540-582,
// handle_shadow_casting od.cpp:584-672, the per-cluster loop and the marking loop of cloud_cb od.cpp:817-833):
//   k_occ_shadow         blocks (k, frame) take the frame's clusters k, k + gridDim.x, ...: members into the sensor
//                        frame, the four extrema by a (value, position) reduction that keeps the sequential loop's
//                        "first occurrence wins" rule, the shadow geometry by one thread (double arithmetic,
//                        deterministic asin / tan), then the fan of lines is dealt to the threads; every line walks
//                        its pixels sequentially (the y intercept is a running float sum).  All lines store the same
//                        value, so their order does not matter.
//   k_occ_mark           every remaining point marks its cell 100 (after the shadows, as in the reference).
// Every per-frame quantity (point and cluster counts, CSR, poses, grid, warning word) is read on the device, so the
// batched call runs these kernels inside the wave without the host learning C or P; pcop_occupancy_shadows runs
// them with one frame.
//
// The arithmetic choices the reference leaves open (double overloads of fabs / sqrt / asin / tan / ceil, step cap of
// the cell search, 64-bit cell indices, the degenerate-fan guard, the bounds check of the marking) are the ones
// written in words in include/pcop.h (pcop_occupancy_shadows).
#include "det_math.cuh"
#include "internal.cuh"

namespace pcop {

namespace {

constexpr int OCC_COUNT_CAP = 1 << 20;
constexpr long long SHADOW_MAX_LINE = 65536;
constexpr int SH_THREADS = 256;
constexpr int OCC_CHUNK = 16384;         // points per block of k_occ_count_wave (32-bit and global counters)
constexpr int OCC_CHUNK16 = 65535;       // ... with 16-bit counters: no cell of a chunk can count past 65535
constexpr int OCC_COUNT_THREADS = 512;

// get_occupancy_grid_x_y's while-loops (od.cpp:139-147) in closed form: the smallest k >= 0 for which the loop
// condition fails.  The edge value fl(a +- fl((k+1)*bs)) is monotone in k, so a floor estimate followed by a walk of a
// few steps lands on exactly the k the reference's loop stops at.  CAPPED: the count stops at OCC_COUNT_CAP (the
// shadow geometry and the marks, whose points may lie anywhere); the initial data set only sees crop survivors.
template <bool CAPPED>
__device__ __forceinline__ int occ_up(float x_min, float bs, float x) {  // while (x_min + (k+1)*bs < x) k++
  if (!(x == x)) return 0;
  const float est = floorf(fdiv(fsub(x, x_min), bs));
  if (CAPPED && est >= (float)(OCC_COUNT_CAP + 8)) return OCC_COUNT_CAP;
  int k = (est > 2.0f) ? (int)(est - 2.0f) : 0;
  while (k > 0 && !(fadd(x_min, fmul((float)k, bs)) < x)) --k;  // the loop would already have stopped at k-1
  while ((!CAPPED || k < OCC_COUNT_CAP) && fadd(x_min, fmul((float)(k + 1), bs)) < x) ++k;
  return k;
}
template <bool CAPPED>
__device__ __forceinline__ int occ_down(float y_max, float bs, float y) {  // while (y_max - (k+1)*bs > y) k++
  if (!(y == y)) return 0;
  const float est = floorf(fdiv(fsub(y_max, y), bs));
  if (CAPPED && est >= (float)(OCC_COUNT_CAP + 8)) return OCC_COUNT_CAP;
  int k = (est > 2.0f) ? (int)(est - 2.0f) : 0;
  while (k > 0 && !(fsub(y_max, fmul((float)k, bs)) > y)) --k;
  while ((!CAPPED || k < OCC_COUNT_CAP) && fsub(y_max, fmul((float)(k + 1), bs)) > y) ++k;
  return k;
}

// od.cpp:197-205: the literal crop predicate, then the cell of a survivor; -1: dropped (outside the box or the grid)
__device__ __forceinline__ long long occ_cell(const float4 p, const OccGrid& g) {
  if ((p.x != p.x) || p.x < g.lim[0] || p.x > g.lim[1] || p.z < g.lim[4] || p.z > g.lim[5] || p.y < g.lim[2] ||
      p.y > g.lim[3])
    return -1;
  const int xc = occ_up<false>(g.lim[2], g.block_size, p.y);  // od.cpp:203: (x, y, x_min, y_max) := (point.y, point.x, y_min, x_max)
  const int yc = occ_down<false>(g.lim[1], g.block_size, p.x);
  const long long index = (long long)yc * g.W + xc;
  return (index >= g.cells) ? -1 : index;  // od.cpp:205
}

__global__ void __launch_bounds__(256)
    k_occ_count(const float4* __restrict__ in, int n, OccGrid g, unsigned long long* __restrict__ counts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long c = occ_cell(__ldg(in + i), g);
  if (c >= 0) atomicAdd(&counts[c], 1ull);
}

// MODE: occ_count_mode
template <int MODE>
__global__ void __launch_bounds__(OCC_COUNT_THREADS)
    k_occ_count_wave(const float4* __restrict__ in, size_t in_stride, const int* __restrict__ n_in, OccGrid g, int chunk,
                     int* __restrict__ counts) {
  extern __shared__ unsigned occ_hist[];
  const int f = blockIdx.y;
  const int n = n_in[f];
  const int i0 = blockIdx.x * chunk;
  if (i0 >= n) return;
  const int i1 = min(n, i0 + chunk);
  const float4* src = in + (size_t)f * in_stride;
  int* cnt = counts + (size_t)f * (size_t)g.cells;
  if (MODE == OCC_COUNT_GLOBAL) {
    for (int i = i0 + (int)threadIdx.x; i < i1; i += OCC_COUNT_THREADS) {
      const long long c = occ_cell(__ldg(src + i), g);
      if (c >= 0) atomicAdd(&cnt[c], 1);
    }
    return;
  }
  const int cells = (int)g.cells;
  const int words = (MODE == OCC_COUNT_SMEM16) ? (cells + 1) >> 1 : cells;
  for (int w = threadIdx.x; w < words; w += OCC_COUNT_THREADS) occ_hist[w] = 0u;
  __syncthreads();
  for (int i = i0 + (int)threadIdx.x; i < i1; i += OCC_COUNT_THREADS) {
    const long long c = occ_cell(__ldg(src + i), g);
    if (c < 0) continue;
    if (MODE == OCC_COUNT_SMEM16)
      atomicAdd(&occ_hist[c >> 1], 1u << (16 * (int)(c & 1)));
    else
      atomicAdd(&occ_hist[c], 1u);
  }
  __syncthreads();
  for (int w = threadIdx.x; w < words; w += OCC_COUNT_THREADS) {
    const unsigned v = occ_hist[w];
    if (v == 0u) continue;
    if (MODE == OCC_COUNT_SMEM16) {
      if (v & 0xffffu) atomicAdd(&cnt[2 * w], (int)(v & 0xffffu));
      if (v >> 16) atomicAdd(&cnt[2 * w + 1], (int)(v >> 16));
    } else {
      atomicAdd(&cnt[w], (int)v);
    }
  }
}

// one block per (row, frame): integer row average (od.cpp:226-234, the sum in 64 bits), then the threshold
// (od.cpp:241-266).  warnings (the batched call): the block of row 0 clears the frame's shadow bit, so that a wave
// whose back half runs again sets it afresh.
template <class T>
__global__ void __launch_bounds__(256)
    k_occ_finish(const T* __restrict__ counts, int W, long long frame_cells, float dev_percent,
                 long long* __restrict__ row_avg, signed char* __restrict__ grid, uint32_t* __restrict__ warnings) {
  const int r = blockIdx.x, f = blockIdx.y;
  const T* crow = counts + (size_t)f * (size_t)frame_cells + (size_t)r * W;
  signed char* grow = grid + (size_t)f * (size_t)frame_cells + (size_t)r * W;
  __shared__ unsigned long long part[8];
  __shared__ long long avg_sh;
  unsigned long long s = 0;
  for (int c = threadIdx.x; c < W; c += blockDim.x) s += (unsigned long long)crow[c];
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < 8; ++w) t += part[w];
    avg_sh = (long long)t / (long long)W;
    if (row_avg) row_avg[r] = avg_sh;
    if (warnings && r == 0) warnings[f] &= ~(uint32_t)PCOP_WARN_SHADOW_DEGENERATE;
  }
  __syncthreads();
  const float thr = fmul((float)avg_sh, fsub(1.0f, dev_percent));
  for (int c = threadIdx.x; c < W; c += blockDim.x) grow[c] = ((float)(long long)crow[c] < thr) ? 100 : 0;
}

__device__ __forceinline__ float4 xform(const Mat34& t, const float4 p) {
  float4 o = p;
  o.x = fadd(fadd(fadd(fmul(t.m[0], p.x), fmul(t.m[1], p.y)), fmul(t.m[2], p.z)), t.m[3]);
  o.y = fadd(fadd(fadd(fmul(t.m[4], p.x), fmul(t.m[5], p.y)), fmul(t.m[6], p.z)), t.m[7]);
  o.z = fadd(fadd(fadd(fmul(t.m[8], p.x), fmul(t.m[9], p.y)), fmul(t.m[10], p.z)), t.m[11]);
  return o;
}

// static_cast<int>(double) as cvttsd2si
__device__ __forceinline__ int cvt_d2i(double v) {
  if (v != v || v >= 2147483648.0 || v <= -2147483649.0) return (int)0x80000000;
  return __double2int_rz(v);
}

// running extreme of a strict-compare loop: the first occurrence of the smallest (LESS) / largest value; values that
// compare false against everything (NaN) never win.  pos = INT_MAX: nothing seen yet.
struct Ext {
  float v;
  int pos;
};
template <bool LESS>
__device__ __forceinline__ void ext_add(Ext& e, float v, int pos) {
  if (!(v == v)) return;
  if (e.pos == 0x7fffffff || (LESS ? (v < e.v) : (v > e.v))) {
    e.v = v;
    e.pos = pos;
  }
}
template <bool LESS>
__device__ __forceinline__ void ext_merge(Ext& e, float v, int pos) {
  if (pos == 0x7fffffff) return;
  if (e.pos == 0x7fffffff || (LESS ? (v < e.v) : (v > e.v)) || (v == e.v && pos < e.pos)) {
    e.v = v;
    e.pos = pos;
  }
}
template <bool LESS>
__device__ void ext_block_reduce(Ext& e, Ext* sh /* [SH_THREADS / 32] */) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const float v = __shfl_xor_sync(FULL, e.v, o);
    const int p = __shfl_xor_sync(FULL, e.pos, o);
    ext_merge<LESS>(e, v, p);
  }
  __syncthreads();  // (sh may still be read from the previous reduction)
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = e;
  __syncthreads();
  e = sh[0];
  for (int w = 1; w < SH_THREADS / 32; ++w) ext_merge<LESS>(e, sh[w].v, sh[w].pos);
}

// traceShadow (od.cpp:467-538); false: the line is too long to draw
__device__ bool trace_shadow(float v1x, float v1y, float v2x, float v2y, signed char* __restrict__ grid, int W, long long size,
                             signed char opacity) {
  int x0 = cvt_f2i(v1x), x1 = cvt_f2i(v2x), y0 = cvt_f2i(v1y), y1 = cvt_f2i(v2y);
  const bool steep = llabs((long long)y1 - y0) > llabs((long long)x1 - x0);
  if (steep) {
    int t = x0; x0 = y0; y0 = t;
    t = x1; x1 = y1; y1 = t;
  }
  if (x0 > x1) {
    int t = x0; x0 = x1; x1 = t;
    t = y0; y0 = y1; y1 = t;
  }
  if ((long long)x1 - x0 + 1 > SHADOW_MAX_LINE) return false;
  const float dx = (float)(x1 - x0);
  const float dy = (float)(int)((unsigned)y1 - (unsigned)y0);
  float gradient = fdiv(dy, dx);
  if (dx == 0.0f) gradient = 1.0f;
  float iy = (float)y0;
  for (int x = x0; x <= x1; ++x) {
    const int fl = cvt_f2i(floorf(iy));
    const long long gy = steep ? x : fl, gx = steep ? fl : x;
    long long idx = gy * W + gx;
    if (idx < size && idx > -1) grid[idx] = opacity;
    idx += 1;
    if (idx < size && idx > -1) grid[idx] = opacity;
    iy = fadd(iy, gradient);
  }
  return true;
}

struct ShadowShared {
  Ext red[SH_THREADS / 32];
  int start_x, start_y, end_x, end_y;
  long long n_lines;
  int skipped;
};

__global__ void __launch_bounds__(SH_THREADS) k_occ_shadow(OccShadowArgs a) {
  const int f = blockIdx.y;
  const int n_clusters = a.n_clusters[f];
  const int* __restrict__ offsets = a.offsets + (size_t)f * a.offsets_stride;
  const int* __restrict__ indices = a.indices + (size_t)f * a.indices_stride;
  const float4* __restrict__ cloud = a.cloud + (size_t)f * a.cloud_stride;
  const Mat34& world_to_sensor = a.mats[2 * f];
  const Mat34& sensor_to_world = a.mats[2 * f + 1];
  signed char* __restrict__ grid = a.grid + (size_t)f * (size_t)a.size;
  __shared__ ShadowShared sm;
  for (int c = blockIdx.x; c < n_clusters; c += gridDim.x) {  // (uniform over the block: the barriers below are safe)
    const int o0 = offsets[c], o1 = offsets[c + 1];
    int* rec = a.records ? a.records + 6 * (size_t)c : nullptr;
    if (o1 - o0 < 2) {  // od.cpp:574
      if (rec && threadIdx.x < 6) rec[threadIdx.x] = 0;
      continue;
    }
    // od.cpp:587-609: extrema of the members in the sensor frame
    Ext vmin{0.f, 0x7fffffff}, vmax{0.f, 0x7fffffff}, hmin{0.f, 0x7fffffff}, hmax{0.f, 0x7fffffff};
    for (int j = o0 + (int)threadIdx.x; j < o1; j += SH_THREADS) {
      const float4 q = xform(world_to_sensor, __ldg(cloud + indices[j]));
      ext_add<true>(vmin, q.x, j);
      ext_add<false>(vmax, q.x, j);
      ext_add<true>(hmin, q.y, j);
      ext_add<false>(hmax, q.y, j);
    }
    ext_block_reduce<true>(vmin, sm.red);
    ext_block_reduce<false>(vmax, sm.red);
    ext_block_reduce<true>(hmin, sm.red);
    ext_block_reduce<false>(hmax, sm.red);
    if (threadIdx.x == 0) {
      // the loop starts from member 0: a NaN there is never replaced (every compare against it is false)
      const float4 q0 = xform(world_to_sensor, __ldg(cloud + indices[o0]));
      const bool x0nan = !(q0.x == q0.x), y0nan = !(q0.y == q0.y);
      const float4 vmin_pt = x0nan ? q0 : xform(world_to_sensor, __ldg(cloud + indices[vmin.pos]));
      const float vertical_max = x0nan ? q0.x : vmax.v;
      const float horizontal_min = y0nan ? q0.y : hmin.v, horizontal_max = y0nan ? q0.y : hmax.v;
      const float width = fabsf(fsub(horizontal_max, horizontal_min));  // od.cpp:616
      // calculate_shadow_cast (od.cpp:540-582)
      const float sa = vmin_pt.z;
      const float sb = fabsf(vmin_pt.x);
      const float sc = (float)__dsqrt_rn((double)fadd(fmul(sa, sa), fmul(sb, sb)));
      const float se = (float)dadd(dsub(fabs((double)vertical_max), fabs((double)vmin_pt.x)), 0.04);
      const float D = (float)det_asin((double)fdiv(sa, sc));
      const float d = (float)dadd(dmul(det_tan((double)D), (double)se), 0.25);
      const float v_len = (float)__dsqrt_rn(
          (double)fadd(fadd(fmul(vmin_pt.x, vmin_pt.x), fmul(vmin_pt.y, vmin_pt.y)), fmul(vmin_pt.z, vmin_pt.z)));
      float4 end = vmin_pt;
      end.x = fadd(fmul(fdiv(vmin_pt.x, v_len), d), vmin_pt.x);
      end.y = fadd(fmul(fdiv(vmin_pt.y, v_len), d), vmin_pt.y);
      end.z = fadd(fmul(fdiv(vmin_pt.z, v_len), d), vmin_pt.z);
      const float4 world_end = xform(sensor_to_world, end);
      int end_x = occ_up<true>(a.y_min, a.block_size, world_end.y);     // od.cpp:569: (x, y) := (point.y, point.x)
      const int end_y = occ_down<true>(a.x_max, a.block_size, world_end.x);
      const float4 world_start = xform(sensor_to_world, vmin_pt);      // od.cpp:634-637
      int start_x = occ_up<true>(a.y_min, a.block_size, world_start.y);
      const int start_y = occ_down<true>(a.x_max, a.block_size, world_start.x);
      // od.cpp:642-643: first += ceil((width / block_size) / 2)   (int += double)
      const float wb = fdiv(width, a.block_size);
      const double shift = ceil((double)fdiv(wb, 2.0f));
      start_x = cvt_d2i(dadd((double)start_x, shift));
      end_x = cvt_d2i(dadd((double)end_x, shift));
      // od.cpp:645: for (int i = 0; i < ceil(width / block_size) + 3; i++)
      const double lim = dadd(ceil((double)wb), 3.0);
      long long n_lines = 0;
      if (lim == lim && lim > 0.0) n_lines = (lim > 1.0e9) ? 1000000000ll : (long long)ceil(lim);
      int skipped = 0;
      if (n_lines > SHADOW_MAX_LINE) {
        skipped = 1;
        n_lines = 0;
      }
      sm.start_x = start_x;
      sm.start_y = start_y;
      sm.end_x = end_x;
      sm.end_y = end_y;
      sm.n_lines = n_lines;
      sm.skipped = skipped;
    }
    __syncthreads();
    const signed char opacity = (signed char)a.opacity;
    bool bad = false;
    for (long long i = threadIdx.x; i < sm.n_lines; i += SH_THREADS) {  // od.cpp:645-661
      const int sx = (int)((unsigned)sm.start_x - (unsigned)i), ex = (int)((unsigned)sm.end_x - (unsigned)i);
      if (!trace_shadow((float)sx, (float)sm.start_y, (float)ex, (float)sm.end_y, grid, a.W, a.size, opacity)) bad = true;
    }
    const int any_bad = __syncthreads_or(bad ? 1 : 0);
    if (threadIdx.x == 0) {
      const int skipped = (sm.skipped || any_bad) ? 1 : 0;
      if (skipped) atomicOr(a.warnings + f, (uint32_t)PCOP_WARN_SHADOW_DEGENERATE);
      if (rec) {
        rec[0] = sm.start_x;
        rec[1] = sm.start_y;
        rec[2] = sm.end_x;
        rec[3] = sm.end_y;
        rec[4] = (int)sm.n_lines;
        rec[5] = skipped;
      }
    }
  }
}

// od.cpp:823-833: every remaining point with a non-NaN x marks its cell (bounds-checked like od.cpp:205)
__global__ void __launch_bounds__(256)
    k_occ_mark(const float4* __restrict__ cloud, size_t cloud_stride, const int* __restrict__ n_pts, float y_min,
               float x_max, float bs, int W, long long size, signed char* __restrict__ grid) {
  const int f = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pts[f]) return;
  const float4 p = __ldg(cloud + (size_t)f * cloud_stride + i);
  if (p.x != p.x) return;
  const int xc = occ_up<true>(y_min, bs, p.y);
  const int yc = occ_down<true>(x_max, bs, p.x);
  const long long idx = (long long)yc * W + xc;
  if (idx < size) grid[(size_t)f * (size_t)size + idx] = 100;
}

}  // namespace

int occ_count_mode(long long cells) {
  if (cells * 4 <= OCC_SMEM_BYTES) return OCC_COUNT_SMEM32;
  if (cells * 2 <= OCC_SMEM_BYTES) return OCC_COUNT_SMEM16;
  return OCC_COUNT_GLOBAL;
}

void run_occ_count(const Ctx& c, const float4* in, int n, const OccGrid& g, unsigned long long* counts) {
  if (n <= 0) return;
  KL(c, "k_occ_count", k_occ_count<<<cdiv(n, 256), 256, 0, c.stream>>>(in, n, g, counts));
  count_launch(c);
}

cudaError_t run_occ_count_wave(const Ctx& c, const float4* in, size_t in_stride, const int* n_in, const OccGrid& g,
                               int* counts) {
  const int mode = occ_count_mode(g.cells);
  cudaError_t e = cudaSuccess;
  if (mode == OCC_COUNT_SMEM32) {
    const int smem = (int)g.cells * 4;
    e = cudaFuncSetAttribute(k_occ_count_wave<OCC_COUNT_SMEM32>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    KL(c, "k_occ_count_wave_s32", k_occ_count_wave<OCC_COUNT_SMEM32><<<dim3(cdiv(c.grid_cap, OCC_CHUNK), c.B), OCC_COUNT_THREADS, smem, c.stream>>>(
                                      in, in_stride, n_in, g, OCC_CHUNK, counts));
  } else if (mode == OCC_COUNT_SMEM16) {
    const int smem = (((int)g.cells + 1) >> 1) * 4;
    e = cudaFuncSetAttribute(k_occ_count_wave<OCC_COUNT_SMEM16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    KL(c, "k_occ_count_wave_s16", k_occ_count_wave<OCC_COUNT_SMEM16><<<dim3(cdiv(c.grid_cap, OCC_CHUNK16), c.B), OCC_COUNT_THREADS, smem, c.stream>>>(
                                      in, in_stride, n_in, g, OCC_CHUNK16, counts));
  } else {
    KL(c, "k_occ_count_wave_g", k_occ_count_wave<OCC_COUNT_GLOBAL><<<dim3(cdiv(c.grid_cap, OCC_CHUNK), c.B), OCC_COUNT_THREADS, 0, c.stream>>>(
                                    in, in_stride, n_in, g, OCC_CHUNK, counts));
  }
  count_launch(c);
  return cudaGetLastError();
}

void run_occ_finish(const Ctx& c, const unsigned long long* counts, const OccGrid& g, long long* row_avg, signed char* grid) {
  KL(c, "k_occ_finish", k_occ_finish<unsigned long long><<<dim3(g.H, 1), 256, 0, c.stream>>>(counts, g.W, g.cells, g.dev_percent,
                                                                                          row_avg, grid, nullptr));
  count_launch(c);
}

void run_occ_finish_wave(const Ctx& c, const int* counts, const OccGrid& g, signed char* grids, uint32_t* warnings) {
  KL(c, "k_occ_threshold_wave", k_occ_finish<int><<<dim3(g.H, c.B), 256, 0, c.stream>>>(counts, g.W, g.cells, g.dev_percent,
                                                                                     nullptr, grids, warnings));
  count_launch(c);
}

void run_occ_shadows(const Ctx& c, const OccShadowArgs& a, int blocks_per_frame, int max_points) {
  if (blocks_per_frame > 0) {
    KL(c, "k_occ_shadow", k_occ_shadow<<<dim3(blocks_per_frame, c.B), SH_THREADS, 0, c.stream>>>(a));
    count_launch(c);
  }
  if (max_points > 0) {
    KL(c, "k_occ_mark", k_occ_mark<<<dim3(cdiv(max_points, 256), c.B), 256, 0, c.stream>>>(
                            a.cloud, a.cloud_stride, a.n_points, a.y_min, a.x_max, a.block_size, a.W, a.size, a.grid));
    count_launch(c);
  }
}

}  // namespace pcop
