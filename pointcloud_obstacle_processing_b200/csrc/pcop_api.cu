// C ABI of the library (include/pcop.h): handle, memory, wave scheduling, result packing.
//
// A call processes its frames in waves.  Within a wave every stage is one set of launches over all
// frames (blockIdx.y = frame) and nothing returns to the host between the input upload and the wave's
// counts: the RANSAC loop of od.cpp:379 runs inside one cluster kernel per frame (stage_plane.cu).
// Waves are dealt round-robin to the lanes (a lane = one stream + one set of wave buffers); ONE host
// thread enqueues a wave on every lane, then waits for the oldest wave's counts (an event), enqueues
// its payload copy with the exact size and refills the lane, so a wave's result copy and the host's
// bookkeeping overlap the other lanes' kernels.  Requested outputs of all frames of a wave are packed
// on the device into one contiguous buffer and come back in a single device->host copy.
// Every buffer is allocated by pcop_create; the pinned result buffer only grows (a second call of the
// same shape allocates nothing).
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>

#include "internal.cuh"
#include "primitives.cuh"

using namespace pcop;

namespace {

enum {  // rows of the per-frame count table (device: d_counts[row*maxB + f])
  CNT_IN = 0,
  CNT_CROP,
  CNT_VOX,
  CNT_SOR,
  CNT_REM,
  CNT_CLUS,
  CNT_CLPTS,
  CNT_TMP,
  CNT_NINL,   // inliers of the last segment() call
  CNT_CLUS1,  // C + 1 (CSR offsets length)
  CNT_CELLS,  // occupied clique cells (ECE scratch)
  CNT_ROUTE,  // point count as seen by the generic clustering path (ECE scratch)
  CNT_GROUPS, // groups of the partition voxel path (scratch; the host sizes the next wave's reduce grid by it)
  CNT_ROWS
};

enum {  // packed output arrays
  PK_CROP_KEPT = 0,
  PK_VOX_KEYS,
  PK_VOX_PTS,
  PK_SOR_KEPT,
  PK_INLIERS,
  PK_REM_PTS,
  PK_REM_SRC,
  PK_OFFSETS,
  PK_INDICES,
  PK_OBSTACLES,
  PK_N
};
const int kPkElem[PK_N] = {4, 4, 16, 4, 4, 16, 4, 4, 4, 16};
const int kPkCount[PK_N] = {CNT_CROP, CNT_VOX, CNT_VOX, CNT_SOR, CNT_NINL, CNT_REM, CNT_REM, CNT_CLUS1, CNT_CLPTS, CNT_CLUS};
const uint32_t kPkMask[PK_N] = {PCOP_OUT_CROP,      PCOP_OUT_VOXEL,     PCOP_OUT_VOXEL,    PCOP_OUT_SOR,
                                PCOP_OUT_PLANE,     PCOP_OUT_REMAINING, PCOP_OUT_REMAINING, PCOP_OUT_CLUSTERS,
                                PCOP_OUT_CLUSTERS,  PCOP_OUT_OBSTACLES};

struct PlaneRecord {
  int n_passes;
  int n_inliers_last;
  float4 coeff;
  int pass_points[PCOP_MAX_PLANE_PASSES_RECORDED];
  int pass_inliers[PCOP_MAX_PLANE_PASSES_RECORDED];
  float4 pass_coeff[PCOP_MAX_PLANE_PASSES_RECORDED];
};

struct PackMeta {  // device -> host in one copy
  unsigned long long base[PK_N];  // byte offset of each array inside the pack buffer
  unsigned long long total_bytes;
  int total[PK_N];  // elements
  int overflow;     // the wave's arrays do not fit the pack buffer (nothing was packed)
};

struct Pc2Frame {  // decode descriptor of one PointCloud2 message (device memory, read by k_pc2_ingest)
  const unsigned char* data;  // payload on the device
  int n, point_step, off_x, off_y, off_z;
  int is_dense, apply_transform, aligned;
  Mat34 t;
};

thread_local std::string g_global_error;

constexpr int PCOP_MIN_LANE_WAVE = 8;  // a call is split over the lanes only when every lane gets at least this many frames

}  // namespace

struct pcop_handle {
  pcop_params params;
  int device = 0;
  int cap = 0;
  int maxB = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  std::vector<void*> dev_allocs;
  std::vector<void*> host_allocs;

  // device
  float4 *d_in = nullptr, *d_crop = nullptr, *d_vox = nullptr, *d_sor = nullptr, *d_pbuf[2] = {nullptr, nullptr},
         *d_rem = nullptr, *d_sorted = nullptr, *d_obst = nullptr;
  int *d_crop_kept = nullptr, *d_run_start = nullptr, *d_sor_kept = nullptr, *d_psrc[2] = {nullptr, nullptr},
      *d_rem_src = nullptr, *d_inliers = nullptr, *d_parent = nullptr, *d_csize = nullptr, *d_roots = nullptr,
      *d_rank = nullptr, *d_indices = nullptr, *d_offsets = nullptr, *d_cell_start = nullptr;
  uint32_t* d_cell_key = nullptr;
  uint32_t* d_vox_keys = nullptr;
  float* d_sor_dist = nullptr;
  SortBufs sort{};
  unsigned* d_desc = nullptr;
  int* d_counts = nullptr;        // [CNT_ROWS][maxB]
  uint32_t* d_warnings = nullptr; // [maxB]
  MinMax* d_minmax = nullptr;
  VoxelFrame* d_vf = nullptr;
  EceFrame* d_ef = nullptr;
  PlaneFrame* d_pf = nullptr;
  PlaneRecord* d_prec = nullptr;
  double* d_partial = nullptr;  // [maxB][chunks][10]
  double* d_thr = nullptr;
  int* d_n_active = nullptr;
  int* d_rng = nullptr;
  int* d_pack_off = nullptr;  // [PK_N][maxB]
  PackMeta* d_meta = nullptr;
  unsigned char* d_pack = nullptr;  // packed results of the wave in flight (PCOP_OUT_DEVICE: of all waves of the call)
  unsigned long long* d_pack_cursor = nullptr;  // PCOP_OUT_DEVICE: bytes of d_pack used by the call so far
  cudaStream_t cstream = nullptr;   // result copies (device -> pinned host) run here, beside the next wave's kernels
  cudaEvent_t ev_copied = nullptr;  // the last payload copy out of d_pack
  cudaEvent_t ev_meta = nullptr;    // the wave's counts / pack sizes are in pinned memory
  int wave_seq = 0;                 // waves of the running call seen by this lane
  int call_lane_waves = 1;          // waves of the running call dealt to this lane
  bool pending = false;             // a wave is enqueued and not yet collected
  int pend_w0 = 0, pend_B = 0;
  double d2h_bytes = 0.0;
  float4* d_acc = nullptr;  // accumulated (world-frame) cloud, od.cpp:697
  unsigned char* d_occ = nullptr;  // occupancy grid scratch: int64 counts, int64 row averages, int8 cells
  size_t occ_cap = 0;
  unsigned char* d_shadow = nullptr;  // pcop_occupancy_shadows scratch: grid cells, CSR copy, records, warning word
  size_t shadow_cap = 0;
  // pcop_process_batch_occupancy, per lane (allocated by the first such call; counts / grids grow with W x H and with
  // the largest wave the lane has run)
  int* d_occ_counts = nullptr;       // [wave frames][cells] int32
  signed char* d_occ_grids = nullptr;  // [wave frames][cells]
  size_t occ_scratch_cells = 0;      // frames x cells the two arrays hold
  Mat34* d_occ_mats = nullptr;       // [maxB][2] world_to_sensor, sensor_to_world
  Mat34* h_occ_mats = nullptr;       // pinned staging of the same
  cudaEvent_t ev_grids_copied = nullptr;  // the last copy out of d_occ_grids
  // the running call's grid product (occ = nullptr: a pcop_process_batch call)
  struct OccCall {
    OccGrid g;
    const float* world_to_sensor16;
    const float* sensor_to_world16;
    int8_t* grids;
    bool grids_on_device;
  };
  const OccCall* occ = nullptr;
  unsigned char* d_raw = nullptr;  // staging of raw PointCloud2 payloads from host memory: one message, or the host
  size_t raw_cap = 0;              // messages of one wave at 256-byte aligned offsets (grown on demand)
  Pc2Frame* d_pc2 = nullptr;       // [maxB] decode descriptors of k_pc2_ingest
  Pc2Frame* h_pc2 = nullptr;       // [maxB] pinned staging of the same (the batched PointCloud2 wave)
  int acc_count = 0;
  size_t pack_cap = 0;
  uint32_t alloc_outputs = 0;

  // pinned host
  int* h_n_active = nullptr;
  int* h_counts = nullptr;  // [CNT_ROWS][maxB]
  uint32_t* h_warnings = nullptr;
  PlaneRecord* h_prec = nullptr;
  PackMeta* h_meta = nullptr;
  int* h_n_in = nullptr;  // staging for the per-frame input sizes
  unsigned long long* h_stats = nullptr;
  unsigned long long sort_pass_keys = 0;
  // pinned result buffers: two per lane, used by alternate calls, so the pointers a call returns stay valid while the
  // NEXT call runs (a consumer may still be reading them, e.g. the multi-GPU result gather)
  unsigned char* h_pack_buf[2] = {nullptr, nullptr};
  size_t h_pack_buf_cap[2] = {0, 0};
  int h_pack_sel = 0;
  unsigned char* h_pack = nullptr;  // = h_pack_buf[h_pack_sel]
  size_t h_pack_cap = 0;
  size_t h_pack_used = 0;  // of the running call

  // timing
  cudaEvent_t ev_call[2] = {nullptr, nullptr};
  cudaEvent_t ev_stage[PCOP_N_STAGES][2] = {};
  bool stage_used[PCOP_N_STAGES] = {};
  float stage_us[PCOP_N_STAGES] = {};
  float last_elapsed_us = 0.f;
  int64_t launches = 0;
  double alg_bytes = 0.0;
  KernelTimers kt;

  // lanes: the handle itself is lane 0; a batched call deals its waves round-robin to the lanes (one stream and one
  // set of wave buffers each), so one lane's result copy and the host's bookkeeping overlap the other lanes' kernels
  int wave_frames = 0;             // frames per wave a batched call aims at (<= maxB; PCOP_WAVE_FRAMES at create)
  bool trace = false;              // PCOP_TRACE at create: per-wave device timeline of every call on stderr
  struct TraceRec {
    int w0, B;
    size_t bytes;
    cudaEvent_t meta, c0, c1;  // counts on the host / payload copy start / end
  };
  std::vector<TraceRec> trace_recs;
  size_t trace_used = 0;
  int ece_small_max = 0;           // ECE_SMALL_MAX or PCOP_ECE_SMALL_MAX (read at create)
  int plane_resident = 1;          // 0: PCOP_PLANE_RESIDENT=0 at create (host-looped plane kernels)
  bool expect_big_remaining = false;  // the last collected wave had a remaining cloud above ece_small_max
  bool expect_large_plane = false;    // ... a plane-stage input above the small tier of the resident plane kernel
  int plane_hostloop_waves = 0;       // waves left that take the host-looped plane kernels (a frame was above the resident limit)
  int vox_lsd_waves = 0;              // waves left that take the LSD voxel path (the partition path declined a bucket)
  bool wave_plane_resident = false;   // the wave in flight ran the resident plane path
  bool wave_plane_speculated = false; // the wave in flight ran the small tier only
  const float4* plane_in = nullptr;   // plane-stage input of the wave in flight (for a repeat of the stage)
  size_t plane_stride = 0;
  const int* plane_n = nullptr;
  bool wave_cluster_speculated = false;  // the wave in flight ran the fused clustering kernel only
  int pend_max_n = 1;
  VoxFusedPlan vplan{};            // fused crop + voxel fast path (ok = 0: not applicable to these parameters)
  uint32_t* d_vf_flags = nullptr;  // [maxB]
  unsigned long long* d_vf_pair[2] = {nullptr, nullptr};
  uint32_t* h_vf_flags = nullptr;
  int vox_mode = 0;                // 0 generic crop + voxel kernels, 1 fused LSD path, 2 fused partition path (at create)
  int vox_redo = -1;               // >= 0 while a wave is repeated: the mode to take instead of vox_mode
  bool vox_full_groups = false;    // ... with the worst-case reduce grid of the partition path
  bool wave_used_fused = false;
  uint32_t* d_vp_hist = nullptr;
  uint32_t* d_vp_bstart = nullptr;
  uint32_t* d_vp_nstart = nullptr;
  unsigned short* d_vp_ne = nullptr;
  uint2* d_vp_grec = nullptr;
  unsigned* d_vp_desc = nullptr;
  int vp_gstride = 0;              // worst-case groups per frame + 1
  int vp_group_hint = 0;           // groups per frame the next wave's reduce grid covers (adapts to the frames seen)
  std::vector<pcop_handle*> extra_lanes;
  std::vector<size_t> fixups;  // result-pointer slots of the running call (byte offsets into the caller's array)
  cudaEvent_t ev_lane_done = nullptr;

  int* cnt(int row) { return d_counts + (size_t)row * maxB; }
};

namespace pcop {
int fail_cuda(pcop_handle* h, cudaError_t e, const char* expr, const char* file, int line) {
  char buf[512];
  snprintf(buf, sizeof(buf), "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, expr);
  if (h) h->err = buf;
  g_global_error = buf;
  return PCOP_ERR_CUDA;
}
}  // namespace pcop

namespace {

int fail(pcop_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  g_global_error = msg;
  return code;
}

// boost::mt19937 (== std::mt19937 algorithm) restated; rnd() = uniform_int<>(0, INT_MAX) = raw >> 1
void fill_rng_table(uint32_t seed, int* out, int count) {
  uint32_t mt[624];
  mt[0] = seed;
  for (int i = 1; i < 624; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
  int pos = 624;
  for (int k = 0; k < count; ++k) {
    if (pos >= 624) {
      for (int i = 0; i < 624; ++i) {
        const uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7fffffffu);
        mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
      }
      pos = 0;
    }
    uint32_t y = mt[pos++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    out[k] = (int)(y >> 1);
  }
}

// crop + VoxelGrid paths: the fused partition path when the plan allows it, else the fused LSD path, else the generic
// kernels.  PCOP_VOXEL_FUSED=0 forces the generic kernels, =lsd the LSD path (the tests cover all three).
VoxFusedPlan make_plan(const pcop_params& p, size_t max_points, int* mode) {
  VoxFusedPlan pl = make_vox_fused_plan(p);
  vox_part_plan(pl, max_points);
  const char* s = getenv("PCOP_VOXEL_FUSED");
  if (s && s[0] == '0') pl.ok = 0;
  if (s && (s[0] == 'l' || s[0] == 'L')) pl.part_ok = 0;
  if (!pl.ok) pl.part_ok = 0;
  *mode = pl.part_ok ? 2 : (pl.ok ? 1 : 0);
  return pl;
}

int validate_params(pcop_handle* h, const pcop_params& p) {
  if (p.enable_voxel && !(p.downsample_size > 0.0f)) return fail(h, PCOP_ERR_BAD_PARAM, "downsample_size must be > 0");
  if (p.enable_sor && (p.statistical_outlier_meanK < 1 || p.statistical_outlier_meanK > 63))
    return fail(h, PCOP_ERR_BAD_PARAM, "statistical_outlier_meanK must be in [1, 63]");
  if (p.enable_plane && (p.plane_max_iterations < 0 || p.plane_max_iterations + 1 > PCOP_MAX_HYPOTHESES))
    return fail(h, PCOP_ERR_BAD_PARAM, "plane_max_iterations must be in [0, 63]");
  if (p.enable_plane && !(p.plane_probability > 0.0 && p.plane_probability < 1.0))
    return fail(h, PCOP_ERR_BAD_PARAM, "plane_probability must be in (0, 1)");
  if (p.enable_cluster && !(p.euc_cluster_tolerance > 0.0f))
    return fail(h, PCOP_ERR_BAD_PARAM, "euc_cluster_tolerance must be > 0");
  return PCOP_OK;
}

uint32_t effective_outputs(const pcop_params& p) {
  uint32_t m = p.outputs & (uint32_t)(PCOP_OUT_ALL | PCOP_OUT_DEVICE);
  if (p.publish_point_clouds) m |= PCOP_OUT_ALL;  // od.cpp:945: intermediates wanted
  if (!p.enable_crop) m &= ~(uint32_t)PCOP_OUT_CROP;
  if (!p.enable_voxel) m &= ~(uint32_t)PCOP_OUT_VOXEL;
  if (!p.enable_sor) m &= ~(uint32_t)PCOP_OUT_SOR;
  if (!p.enable_plane) m &= ~(uint32_t)PCOP_OUT_PLANE;
  if (!p.enable_cluster) m &= ~(uint32_t)(PCOP_OUT_CLUSTERS | PCOP_OUT_OBSTACLES);
  return m;
}

size_t pack_capacity_bytes(uint32_t mask, int B, int cap) {
  mask &= (uint32_t)PCOP_OUT_ALL;
  size_t bytes = 0;
  for (int k = 0; k < PK_N; ++k)
    if (mask & kPkMask[k]) bytes += ((size_t)B * (cap + 1)) * kPkElem[k] + 256;
  return (bytes + 256 + 255) & ~(size_t)255;
}

template <class T>
int dalloc(pcop_handle* h, T** p, size_t n) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(T));
  if (e != cudaSuccess) return fail_cuda(h, e, "cudaMalloc", __FILE__, __LINE__);
  h->dev_allocs.push_back(q);
  *p = (T*)q;
  return PCOP_OK;
}
template <class T>
int halloc(pcop_handle* h, T** p, size_t n) {
  void* q = nullptr;
  cudaError_t e = cudaHostAlloc(&q, std::max<size_t>(n, 1) * sizeof(T), cudaHostAllocMapped);
  if (e != cudaSuccess) return fail_cuda(h, e, "cudaHostAlloc", __FILE__, __LINE__);
  h->host_allocs.push_back(q);
  *p = (T*)q;
  return PCOP_OK;
}
#define TRY(x)                      \
  do {                              \
    int _s = (x);                   \
    if (_s != PCOP_OK) return _s;   \
  } while (0)

int ensure_pack_capacity(pcop_handle* h, uint32_t mask) {
  const size_t need = pack_capacity_bytes(mask, h->maxB, h->cap);
  if (need <= h->pack_cap) return PCOP_OK;
  if (h->cstream) cudaStreamSynchronize(h->cstream);
  if (h->d_pack) cudaFree(h->d_pack);  // not tracked in dev_allocs
  h->d_pack = nullptr;
  h->pack_cap = 0;
  cudaError_t e = cudaMalloc((void**)&h->d_pack, need);
  if (e != cudaSuccess) return fail_cuda(h, e, "cudaMalloc(pack)", __FILE__, __LINE__);
  h->pack_cap = need;
  return PCOP_OK;
}

int ensure_host_pack(pcop_handle* h, size_t need) {
  if (need <= h->h_pack_cap) return PCOP_OK;
  size_t ncap = std::max<size_t>(need, h->h_pack_cap * 2);
  ncap = std::max<size_t>(ncap, 1 << 20);
  unsigned char* q = nullptr;
  cudaError_t e = cudaHostAlloc((void**)&q, ncap, cudaHostAllocMapped);
  if (e != cudaSuccess) return fail_cuda(h, e, "cudaHostAlloc(pack)", __FILE__, __LINE__);
  if (h->cstream) cudaStreamSynchronize(h->cstream);  // copies into the old buffer must have landed
  if (h->h_pack) {
    memcpy(q, h->h_pack, h->h_pack_cap);
    cudaFreeHost(h->h_pack);
  }
  h->h_pack = q;
  h->h_pack_cap = ncap;
  h->h_pack_buf[h->h_pack_sel] = q;
  h->h_pack_buf_cap[h->h_pack_sel] = ncap;
  return PCOP_OK;
}

// the raw PointCloud2 staging of lane h holds at least `bytes` (grown by a quarter more, never shrunk)
int ensure_raw(pcop_handle* h, size_t bytes) {
  if (bytes <= h->raw_cap) return PCOP_OK;
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (h->d_raw) cudaFree(h->d_raw);  // (not tracked in dev_allocs)
  h->d_raw = nullptr;
  h->raw_cap = 0;
  PCOP_CUDA_TRY(cudaMalloc((void**)&h->d_raw, bytes + bytes / 4 + 256));
  h->raw_cap = bytes + bytes / 4 + 256;
  return PCOP_OK;
}

// ---- small kernels owned by the API layer -----------------------------------------
__global__ void k_copy_counts(const int* __restrict__ src, int* __restrict__ dst, int B) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < B) dst[f] = src[f];
}

__global__ void k_zero_u32(uint32_t* p, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0u;
}

// pcl::transformPointCloud(cloud_in, cloud_out, Eigen::Matrix4f) (via pcl_ros::transformPointCloud, od.cpp:696):
// out.x = m00*x + m01*y + m02*z + m03 in float, left to right, no FMA; non-dense clouds copy non-finite points
__global__ void __launch_bounds__(256)
    k_transform(const float4* __restrict__ in, int n, Mat34 t, int is_dense, float4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = __ldg(in + i);
  float4 o = p;
  const bool finite = fabsf(p.x) <= 3.402823466e+38f && fabsf(p.y) <= 3.402823466e+38f && fabsf(p.z) <= 3.402823466e+38f;
  if (is_dense || finite) {
    o.x = fadd(fadd(fadd(fmul(t.m[0], p.x), fmul(t.m[1], p.y)), fmul(t.m[2], p.z)), t.m[3]);
    o.y = fadd(fadd(fadd(fmul(t.m[4], p.x), fmul(t.m[5], p.y)), fmul(t.m[6], p.z)), t.m[7]);
    o.z = fadd(fadd(fadd(fmul(t.m[8], p.x), fmul(t.m[9], p.y)), fmul(t.m[10], p.z)), t.m[11]);
  }
  out[i] = o;
}

// sensor_msgs/PointCloud2 payload -> pcl::PointXYZ (od.cpp:688-689) [+ world transform, od.cpp:696] in one pass:
// record i = data + i*point_step; FLOAT32 x, y, z at the given offsets (any alignment); padding float = 1.0f
__device__ __forceinline__ float pc2_load_f32(const unsigned char* p) {
  if ((reinterpret_cast<uintptr_t>(p) & 3u) == 0u) return __ldg(reinterpret_cast<const float*>(p));
  const uint32_t b = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
  return __uint_as_float(b);
}
__device__ __forceinline__ float pc2_lane(const float4& v, int k) {  // (compares, not an indexed register array)
  return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w));
}
// One decode per message (pcop_accumulate_pointcloud2 / pcop_pointcloud2_to_xyz: one frame; the batched PointCloud2
// wave: one frame per message).  blockIdx.y = frame, records along x.  Every per-frame quantity comes from the
// descriptor table in device memory.  aligned = 1 (point_step % 16 == 0, 16-byte aligned base, x / y / z inside one
// aligned 16-byte word of the record): one 16-byte load per record instead of three 4-byte (or twelve 1-byte) loads.
__global__ void __launch_bounds__(256)
    k_pc2_ingest(const Pc2Frame* __restrict__ frames, float4* __restrict__ out, size_t out_stride) {
  const int f = blockIdx.y;
  const int n = frames[f].n;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Pc2Frame& d = frames[f];
  const unsigned char* rec = d.data + (size_t)i * (size_t)d.point_step;
  float x, y, z;
  if (d.aligned) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(rec + (d.off_x & ~15)));
    x = pc2_lane(v, (d.off_x & 15) >> 2);
    y = pc2_lane(v, (d.off_y & 15) >> 2);
    z = pc2_lane(v, (d.off_z & 15) >> 2);
  } else {
    x = pc2_load_f32(rec + d.off_x);
    y = pc2_load_f32(rec + d.off_y);
    z = pc2_load_f32(rec + d.off_z);
  }
  float4 o = make_float4(x, y, z, 1.0f);
  const bool finite = fabsf(x) <= 3.402823466e+38f && fabsf(y) <= 3.402823466e+38f && fabsf(z) <= 3.402823466e+38f;
  if (d.apply_transform && (d.is_dense || finite)) {
    const Mat34& t = d.t;
    o.x = fadd(fadd(fadd(fmul(t.m[0], x), fmul(t.m[1], y)), fmul(t.m[2], z)), t.m[3]);
    o.y = fadd(fadd(fadd(fmul(t.m[4], x), fmul(t.m[5], y)), fmul(t.m[6], z)), t.m[7]);
    o.z = fadd(fadd(fadd(fmul(t.m[8], x), fmul(t.m[9], y)), fmul(t.m[10], z)), t.m[11]);
  }
  out[(size_t)f * out_stride + i] = o;
}

// the descriptor of one message whose payload sits at `src` on the device (validated by the caller)
Pc2Frame make_pc2_frame(const unsigned char* src, int n, int point_step, int ox, int oy, int oz, const float* t16,
                        int is_dense) {
  Pc2Frame d{};
  d.data = src;
  d.n = n;
  d.point_step = point_step;
  d.off_x = ox;
  d.off_y = oy;
  d.off_z = oz;
  d.is_dense = is_dense ? 1 : 0;
  d.apply_transform = t16 ? 1 : 0;
  const float ident[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
  memcpy(d.t.m, t16 ? t16 : ident, sizeof(d.t.m));
  const bool word4 = (ox & 3) == 0 && (oy & 3) == 0 && (oz & 3) == 0;
  const bool one_word = (ox >> 4) == (oy >> 4) && (ox >> 4) == (oz >> 4);
  d.aligned = (point_step % 16 == 0 && (reinterpret_cast<uintptr_t>(src) & 15u) == 0u && word4 && one_word) ? 1 : 0;
  return d;
}

bool pc2_layout_ok(int point_step, int ox, int oy, int oz) {
  return point_step >= 4 && ox >= 0 && oy >= 0 && oz >= 0 && ox <= point_step - 4 && oy <= point_step - 4 &&
         oz <= point_step - 4;
}

// pcl::PointXYZ -> sensor_msgs/PointCloud2 payload (pcl::toROSMsg, od.cpp:290-294): the (16, 0, 4, 8) layout is the
// record itself; any other layout gets the three FLOAT32 fields at their offsets (any alignment), other bytes zero
__device__ __forceinline__ void pc2_store_f32(unsigned char* p, float v) {
  const uint32_t b = __float_as_uint(v);
  if ((reinterpret_cast<uintptr_t>(p) & 3u) == 0u) {
    *reinterpret_cast<uint32_t*>(p) = b;
  } else {
    p[0] = (unsigned char)b;
    p[1] = (unsigned char)(b >> 8);
    p[2] = (unsigned char)(b >> 16);
    p[3] = (unsigned char)(b >> 24);
  }
}
__global__ void __launch_bounds__(256)
    k_pc2_egress(const float4* __restrict__ in, int n, int point_step, int off_x, int off_y, int off_z,
                 unsigned char* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = __ldg(in + i);
  unsigned char* rec = out + (size_t)i * (size_t)point_step;
  if (point_step == 16 && off_x == 0 && off_y == 4 && off_z == 8 && (reinterpret_cast<uintptr_t>(out) & 15u) == 0u) {
    *reinterpret_cast<float4*>(rec) = p;  // toROSMsg: the whole record, padding included
    return;
  }
  for (int b = 0; b < point_step; ++b) rec[b] = 0;
  pc2_store_f32(rec + off_x, p.x);
  pc2_store_f32(rec + off_y, p.y);
  pc2_store_f32(rec + off_z, p.z);
  if (point_step == 16 && off_x == 0 && off_y == 4 && off_z == 8) pc2_store_f32(rec + 12, p.w);
}

// cloud copy for a disabled plane stage: remaining = input, src = identity
__global__ void __launch_bounds__(CT_THREADS)
    k_copy_cloud(const float4* __restrict__ in, size_t in_stride, const int* __restrict__ n_in, float4* __restrict__ out,
                 int* __restrict__ out_src, int cap) {
  const int f = blockIdx.y, tile = blockIdx.x;
  const int n = n_in[f];
  if (tile * CT_TILE >= n) return;
#pragma unroll
  for (int k = 0; k < CT_ITEMS; ++k) {
    const int i = ct_index(tile, k);
    if (i < n) {
      out[(size_t)f * cap + i] = __ldg(in + (size_t)f * in_stride + i);
      out_src[(size_t)f * cap + i] = i;
    }
  }
}

__device__ void plane_record_one(const PlaneFrame* __restrict__ pf, PlaneRecord* __restrict__ rec, int* __restrict__ n_inl,
                                 int* __restrict__ n_clus, int* __restrict__ n_clus1, int plane_enabled, int f) {
  PlaneRecord r;
  r.n_passes = 0;
  r.n_inliers_last = 0;
  r.coeff = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int k = 0; k < PCOP_MAX_PLANE_PASSES_RECORDED; ++k) {
    r.pass_points[k] = 0;
    r.pass_inliers[k] = 0;
    r.pass_coeff[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (plane_enabled) {
    const PlaneFrame& P = pf[f];
    r.n_passes = P.n_passes;
    r.n_inliers_last = P.n_inliers_last;
    r.coeff = P.coeff_ref;
    for (int k = 0; k < PCOP_MAX_PLANE_PASSES_RECORDED; ++k) {
      r.pass_points[k] = P.pass_points[k];
      r.pass_inliers[k] = P.pass_inliers[k];
      r.pass_coeff[k] = P.pass_coeff[k];
    }
  }
  rec[f] = r;
  n_inl[f] = r.n_inliers_last;
  n_clus1[f] = n_clus[f] + 1;
}

__global__ void k_plane_record(const PlaneFrame* __restrict__ pf, PlaneRecord* __restrict__ rec, int* __restrict__ n_inl,
                               int* __restrict__ n_clus, int* __restrict__ n_clus1, int plane_enabled, int B) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < B) plane_record_one(pf, rec, n_inl, n_clus, n_clus1, plane_enabled, f);
}

// exclusive scans over the frames of every requested output's count row + array base offsets
// (first the per-frame plane record + the derived count rows CNT_NINL / CNT_CLUS1, which the scans below read)
// (PCOP_OUT_DEVICE: the arrays of all waves of a call stay in the pack buffer, so the wave's base is a device-side
// cursor that this kernel advances; a wave that does not fit sets meta->overflow and is not packed)
__global__ void k_pack_scan(int* __restrict__ counts, int maxB, int B, uint32_t mask, int* __restrict__ pack_off,
                            PackMeta* __restrict__ meta, const PlaneFrame* __restrict__ pf, PlaneRecord* __restrict__ rec,
                            int plane_enabled, unsigned long long* __restrict__ cursor, unsigned long long capacity) {
  __shared__ int total[PK_N];
  for (int f = threadIdx.x; f < B; f += blockDim.x)
    plane_record_one(pf, rec, counts + (size_t)CNT_NINL * maxB, counts + (size_t)CNT_CLUS * maxB,
                     counts + (size_t)CNT_CLUS1 * maxB, plane_enabled, f);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kPkCountD[PK_N] = {CNT_CROP, CNT_VOX, CNT_VOX, CNT_SOR, CNT_NINL, CNT_REM, CNT_REM, CNT_CLUS1, CNT_CLPTS, CNT_CLUS};
  const uint32_t kPkMaskD[PK_N] = {PCOP_OUT_CROP,     PCOP_OUT_VOXEL,     PCOP_OUT_VOXEL,     PCOP_OUT_SOR,
                                   PCOP_OUT_PLANE,    PCOP_OUT_REMAINING, PCOP_OUT_REMAINING, PCOP_OUT_CLUSTERS,
                                   PCOP_OUT_CLUSTERS, PCOP_OUT_OBSTACLES};
  const int kPkElemD[PK_N] = {4, 4, 16, 4, 4, 16, 4, 4, 4, 16};
  for (int k = warp; k < PK_N; k += blockDim.x / 32) {
    int run = 0;
    if (mask & kPkMaskD[k]) {
      const int* row = counts + (size_t)kPkCountD[k] * maxB;
      for (int base = 0; base < B; base += 32) {
        const int f = base + lane;
        const int v = (f < B) ? row[f] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int up = __shfl_up_sync(FULL, incl, o);
          if (lane >= o) incl += up;
        }
        if (f < B) pack_off[(size_t)k * maxB + f] = run + incl - v;
        run += __shfl_sync(FULL, incl, 31);
      }
    }
    if (lane == 0) total[k] = run;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned long long start = cursor ? *cursor : 0ull;
    unsigned long long off = start;
    for (int k = 0; k < PK_N; ++k) {
      meta->base[k] = off;
      meta->total[k] = total[k];
      off += ((unsigned long long)total[k] * kPkElemD[k] + 255ull) & ~255ull;
    }
    meta->total_bytes = off - start;
    meta->overflow = (off > capacity) ? 1 : 0;
    if (cursor && off <= capacity) *cursor = off;
  }
}

// The wave's counts, warnings, plane records, pack sizes and voxel-path flags go to the host as plain stores into
// pinned (device-mapped) memory: as DMA copies they queue behind another lane's 17 MB payload copy on the same copy
// engine (measured: 0.15-0.35 ms per wave, which also knocks the lanes out of step).
struct MetaOut {
  const uint32_t* src[5];
  uint32_t* dst[5];
  int words[5];
  int frames;  // k_pack: the blocks of this many frames share the work (0: none)
};
__device__ __forceinline__ void meta_out_segment(const uint32_t* __restrict__ s, uint32_t* __restrict__ d, int words, int first,
                                                 int stride) {
  for (int i = first; i < words; i += stride) d[i] = s[i];
}
// (the segment index is compared against constants: indexing the parameter struct with a run-time value would make
// every thread copy it to local memory first)
__device__ __forceinline__ void meta_out(const MetaOut& m, int k, int first, int stride) {
#pragma unroll
  for (int j = 0; j < 5; ++j)
    if (j == k && m.src[j]) meta_out_segment(m.src[j], m.dst[j], m.words[j], first, stride);
}
__global__ void __launch_bounds__(256) k_meta_out(MetaOut m) {
  meta_out(m, blockIdx.y, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}
struct PackSrc {
  const uint32_t* src[PK_N];  // nullptr: not requested
  unsigned long long frame_stride_words[PK_N];
  int count_row[PK_N];
  int words_per_elem[PK_N];
};

// all requested output arrays of all frames of the wave in one launch: blockIdx.z = array, blockIdx.y = frame;
// everything is moved as 32-bit words (the 16-byte arrays as uint4)
__global__ void __launch_bounds__(256)
    k_pack(PackSrc ps, const int* __restrict__ counts, int maxB, const int* __restrict__ pack_off,
           const PackMeta* __restrict__ meta, unsigned char* __restrict__ pack, MetaOut mo) {
  const int which = blockIdx.z, f = blockIdx.y;
  if (f < mo.frames && which < 5)  // (metadata, see MetaOut: spread over the blocks of the first frames)
    meta_out(mo, which, (f * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x, mo.frames * gridDim.x * blockDim.x);
  const uint32_t* base = ps.src[which];
  if (!base || meta->overflow) return;
  const int wpe = ps.words_per_elem[which];
  const int n = counts[(size_t)ps.count_row[which] * maxB + f];
  const uint32_t* s = base + (size_t)f * ps.frame_stride_words[which];
  uint32_t* dst = reinterpret_cast<uint32_t*>(pack + meta->base[which]) + (size_t)pack_off[(size_t)which * maxB + f] * wpe;
  if (wpe == 4) {  // 16-byte elements; bases are 256-byte aligned and offsets are whole elements
    const uint4* s4 = reinterpret_cast<const uint4*>(s);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) d4[i] = s4[i];
  } else {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = s[i];
  }
}

struct StageTimer {
  pcop_handle* h;
  int stage;
  StageTimer(pcop_handle* hh, int s) : h(hh), stage(s) {
    cudaEventRecord(h->ev_stage[s][0], h->stream);
    h->stage_used[s] = true;
  }
  ~StageTimer() { cudaEventRecord(h->ev_stage[stage][1], h->stream); }
};

void resolve_kernel_timers(pcop_handle* h) {
  KernelTimers& k = h->kt;
  for (int sl = 0; sl < k.used; ++sl) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, k.ev[2 * sl], k.ev[2 * sl + 1]) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    int id = -1;
    for (int i = 0; i < k.n_names; ++i)
      if (k.names[i] == k.slot_name[sl] || strcmp(k.names[i], k.slot_name[sl]) == 0) {
        id = i;
        break;
      }
    if (id < 0 && k.n_names < KernelTimers::MAX_NAMES) {
      id = k.n_names++;
      k.names[id] = k.slot_name[sl];
      k.total_us[id] = 0.0;
      k.launches[id] = 0;
    }
    if (id >= 0) {
      k.total_us[id] += (double)ms * 1000.0;
      k.launches[id] += 1;
    }
  }
  k.used = 0;
}

Ctx make_ctx(pcop_handle* h, int B, int grid_cap = -1) {
  return Ctx{h->stream, B, h->cap, &h->launches, &h->kt, (grid_cap > 0 && grid_cap < h->cap) ? grid_cap : h->cap, nullptr};
}

PlaneConst make_plane_const(const pcop_params& p) {
  PlaneConst pc;
  pc.thr = p.plane_segment_dist_thres;
  pc.eps_angle = (double)p.plane_segment_angle;  // od.cpp:371: the int is handed to setEpsAngle as radians
  pc.cos_eps = std::cos(pc.eps_angle);
  for (int a = 0; a < 3; ++a) pc.axis[a] = (double)p.plane_axis[a];
  pc.keep_fraction = p.plane_keep_fraction;
  pc.max_iterations = p.plane_max_iterations;
  pc.probability = p.plane_probability;
  pc.log_probability = 0.0;
  pc.optimize = p.optimize_coefficients ? 1 : 0;
  return pc;
}

PlaneArgs make_plane_args(pcop_handle* h, const float4* in, size_t stride, const int* n_in) {
  PlaneArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.buf[0] = h->d_pbuf[0];
  a.buf[1] = h->d_pbuf[1];
  a.src[0] = h->d_psrc[0];
  a.src[1] = h->d_psrc[1];
  a.inlier_idx = h->d_inliers;
  a.pf = h->d_pf;
  a.partial = h->d_partial;
  a.desc = h->d_desc;
  a.n_tmp = h->cnt(CNT_TMP);
  a.n_active = h->d_n_active;
  a.h_n_active = h->h_n_active;
  a.rng = h->d_rng;
  a.resident = h->plane_resident;
  a.pc = make_plane_const(h->params);
  a.warnings = h->d_warnings;
  a.out = h->d_rem;
  a.out_src = h->d_rem_src;
  a.n_out = h->cnt(CNT_REM);
  return a;
}

ClusterArgs make_cluster_args(pcop_handle* h, const float4* in, size_t stride, const int* n_in) {
  ClusterArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.tol = h->params.euc_cluster_tolerance;
  a.min_size = h->params.euc_min_cluster_size;
  a.max_size = h->params.euc_max_cluster_size;
  a.small_max = h->ece_small_max;
  a.minmax = h->d_minmax;
  a.ef = h->d_ef;
  a.sort = h->sort;
  a.sorted_pts = h->d_sorted;
  a.parent = h->d_parent;
  a.csize = h->d_csize;
  a.roots = h->d_roots;
  a.rank_of = h->d_rank;
  a.cell_start = h->d_cell_start;
  a.cell_key = h->d_cell_key;
  a.n_cells = h->cnt(CNT_CELLS);
  a.n_route = h->cnt(CNT_ROUTE);
  a.desc = h->d_desc;
  a.offsets = h->d_offsets;
  a.indices = h->d_indices;
  a.n_clusters = h->cnt(CNT_CLUS);
  a.n_cluster_pts = h->cnt(CNT_CLPTS);
  a.obstacles = h->d_obst;
  a.partial = h->d_partial;
  a.partial_stride = cdiv(h->cap, TS_CHUNK) * 10;
  return a;
}

CropArgs make_crop_args(pcop_handle* h, const float4* in, size_t stride, const int* n_in) {
  CropArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.out = h->d_crop;
  a.kept_idx = h->d_crop_kept;
  a.n_out = h->cnt(CNT_CROP);
  a.minmax = h->d_minmax;
  a.desc = h->d_desc;
  const pcop_params& p = h->params;
  a.lim[0] = p.x_min;
  a.lim[1] = p.x_max;
  a.lim[2] = p.y_min;
  a.lim[3] = p.y_max;
  a.lim[4] = p.z_min;
  a.lim[5] = p.z_max;
  return a;
}

VoxelArgs make_voxel_args(pcop_handle* h, const float4* in, size_t stride, const int* n_in) {
  VoxelArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.minmax = h->d_minmax;
  a.leaf = h->params.downsample_size;
  a.vf = h->d_vf;
  a.sort = h->sort;
  a.desc = h->d_desc;
  a.run_start = h->d_run_start;
  a.out = h->d_vox;
  a.out_keys = h->d_vox_keys;
  a.n_out = h->cnt(CNT_VOX);
  a.warnings = h->d_warnings;
  return a;
}

SorArgs make_sor_args(pcop_handle* h, const float4* in, size_t stride, const int* n_in) {
  SorArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.meanK = h->params.statistical_outlier_meanK;
  a.mul = (double)h->params.statistical_outlier_stdDevThres;
  // search-grid cell: a speed knob only (the k-NN result is exact for any cell size)
  a.cell = (h->params.enable_voxel && h->params.downsample_size > 0.0f) ? 3.0f * h->params.downsample_size : 0.05f;
  a.minmax = h->d_minmax;
  a.gf = h->d_ef;
  a.sort = h->sort;
  a.sorted_pts = h->d_sorted;
  a.dist = h->d_sor_dist;
  a.partial = h->d_partial;
  a.thr = h->d_thr;
  a.desc = h->d_desc;
  a.out = h->d_sor;
  a.kept_idx = h->d_sor_kept;
  a.n_out = h->cnt(CNT_SOR);
  a.warnings = h->d_warnings;
  return a;
}

bool is_device_pointer(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// The plane loop of one wave on the stage input recorded in the handle.  large_tier: see run_plane.
int run_wave_plane(pcop_handle* h, int B, int max_n, bool large_tier) {
  const pcop_params& p = h->params;
  Ctx c = make_ctx(h, B, max_n);  // (no frame holds more points than the largest input frame)
  StageTimer t(h, PCOP_STAGE_PLANE);
  h->wave_plane_speculated = false;
  if (p.enable_plane) {
    PlaneArgs a = make_plane_args(h, h->plane_in, h->plane_stride, h->plane_n);
    a.n_in_copy = p.enable_sor ? nullptr : h->cnt(CNT_SOR);
    a.large_tier = large_tier ? 1 : 0;
    if (h->plane_hostloop_waves > 0) a.resident = 0;
    h->wave_plane_resident = a.resident != 0;
    if (!(effective_outputs(p) & PCOP_OUT_PLANE)) a.inlier_idx = nullptr;  // the inlier list is only written on request
    cudaError_t e = run_plane(c, a);
    if (e != cudaSuccess) return fail_cuda(h, e, "run_plane", __FILE__, __LINE__);
    h->wave_plane_speculated = a.resident && !large_tier && max_n > plane_small_tier_max();
  } else {
    KL(c, "k_copy_counts", k_copy_counts<<<cdiv(B, 256), 256, 0, h->stream>>>(h->plane_n, h->cnt(CNT_REM), B));
    KL(c, "k_copy_cloud", k_copy_cloud<<<dim3(cdiv(c.grid_cap, CT_TILE), B), CT_THREADS, 0, h->stream>>>(
                              h->plane_in, h->plane_stride, h->plane_n, h->d_rem, h->d_rem_src, h->cap));
    count_launch(c, 2);
  }
  return PCOP_OK;
}

// All stages of one wave up to the plane loop.  `in`/`stride` already on the device; counts row CNT_IN already set.
int run_wave_stages(pcop_handle* h, int B, const float4* in, size_t stride, int max_n) {
  const pcop_params& p = h->params;
  Ctx c = make_ctx(h, B, max_n);  // no stage ever holds more points per frame than the largest input frame
  const int tiles = cdiv(h->cap, CT_TILE);
  const int vmode = (h->vox_redo >= 0) ? h->vox_redo : ((h->vox_mode == 2 && h->vox_lsd_waves > 0) ? 1 : h->vox_mode);
  const bool fused_path = vmode != 0;
  if (!fused_path || (effective_outputs(p) & PCOP_OUT_CROP)) {  // (the fused voxel path zeroes the warnings itself)
    KL(c, "k_zero_u32", k_zero_u32<<<cdiv(B, 256), 256, 0, h->stream>>>(h->d_warnings, B));
    count_launch(c);
  }

  const float4* cur = in;
  size_t cur_stride = stride;
  const int* cur_n = h->cnt(CNT_IN);
  bool have_minmax = false;

  const bool fused = fused_path;
  h->wave_used_fused = fused;
  if (fused && vmode == 2) {
    {
      StageTimer t(h, PCOP_STAGE_CROP);
      if (effective_outputs(p) & PCOP_OUT_CROP) run_crop(c, make_crop_args(h, cur, cur_stride, cur_n));
    }
    StageTimer t(h, PCOP_STAGE_VOXEL);
    VoxelPartArgs a{};
    a.in = cur;
    a.in_stride = cur_stride;
    a.n_in = cur_n;
    a.plan = h->vplan;
    a.leaf = p.downsample_size;
    a.minmax = h->d_minmax;
    a.vf = h->d_vf;
    a.ghist = h->d_vp_hist;
    a.chunk_start = h->d_vp_bstart;
    a.ne_bucket = h->d_vp_ne;
    a.ne_start = h->d_vp_nstart;
    a.grec = h->d_vp_grec;
    a.n_groups = h->cnt(CNT_GROUPS);
    a.part = h->d_sorted;  // (the search-grid point list of SOR / clustering is not live yet)
    a.desc = h->d_vp_desc;
    a.group_stride = h->vp_gstride;
    a.group_launch = h->vox_full_groups ? h->vp_gstride - 1 : std::min(h->vp_group_hint, vox_part_group_bound(h->vplan, max_n));
    a.flags = h->d_vf_flags;
    a.warnings = (effective_outputs(p) & PCOP_OUT_CROP) ? nullptr : h->d_warnings;  // zeroed by k_vp_init
    a.n_crop = h->cnt(CNT_CROP);
    a.out = h->d_vox;
    a.out_keys = h->d_vox_keys;
    a.n_out = h->cnt(CNT_VOX);
    a.want_keys = (effective_outputs(p) & PCOP_OUT_VOXEL) ? 1 : 0;
    run_voxel_part(c, a);
    cur = h->d_vox;
    cur_stride = h->cap;
    cur_n = h->cnt(CNT_VOX);
  } else if (fused) {
    // crop + VoxelGrid in one pass over the input (stage_voxel_fused.cu); the cropped cloud itself is only
    // materialised when it is a requested output
    {
      StageTimer t(h, PCOP_STAGE_CROP);
      if (effective_outputs(p) & PCOP_OUT_CROP) run_crop(c, make_crop_args(h, cur, cur_stride, cur_n));
    }
    StageTimer t(h, PCOP_STAGE_VOXEL);
    VoxelFusedArgs a{};
    a.in = cur;
    a.in_stride = cur_stride;
    a.n_in = cur_n;
    a.plan = h->vplan;
    a.leaf = p.downsample_size;
    a.minmax = h->d_minmax;
    a.vf = h->d_vf;
    a.sort = h->sort;
    a.pair[0] = h->d_vf_pair[0];
    a.pair[1] = h->d_vf_pair[1];
    a.desc = h->d_desc;
    a.flags = h->d_vf_flags;
    a.warnings = (effective_outputs(p) & PCOP_OUT_CROP) ? nullptr : h->d_warnings;  // zeroed by k_vf_init
    a.n_crop = h->cnt(CNT_CROP);
    a.out = h->d_vox;
    a.out_keys = h->d_vox_keys;
    a.n_out = h->cnt(CNT_VOX);
    a.want_keys = (effective_outputs(p) & PCOP_OUT_VOXEL) ? 1 : 0;
    run_voxel_fused(c, a);
    cur = h->d_vox;
    cur_stride = h->cap;
    cur_n = h->cnt(CNT_VOX);
  } else {
    {
      StageTimer t(h, PCOP_STAGE_CROP);
      if (p.enable_crop) {
        run_crop(c, make_crop_args(h, cur, cur_stride, cur_n));
        cur = h->d_crop;
        cur_stride = h->cap;
        cur_n = h->cnt(CNT_CROP);
        have_minmax = true;
      } else {
        KL(c, "k_copy_counts", k_copy_counts<<<cdiv(B, 256), 256, 0, h->stream>>>(cur_n, h->cnt(CNT_CROP), B));
        count_launch(c);
      }
    }
    {
      StageTimer t(h, PCOP_STAGE_VOXEL);
      if (p.enable_voxel) {
        if (!have_minmax) run_minmax(c, cur, cur_stride, cur_n, h->d_minmax);
        run_voxel(c, make_voxel_args(h, cur, cur_stride, cur_n));
        cur = h->d_vox;
        cur_stride = h->cap;
        cur_n = h->cnt(CNT_VOX);
      } else {
        KL(c, "k_copy_counts", k_copy_counts<<<cdiv(B, 256), 256, 0, h->stream>>>(cur_n, h->cnt(CNT_VOX), B));
        count_launch(c);
      }
    }
  }
  {
    StageTimer t(h, PCOP_STAGE_SOR);
    if (p.enable_sor) {
      run_sor(c, make_sor_args(h, cur, cur_stride, cur_n));
      cur = h->d_sor;
      cur_stride = h->cap;
      cur_n = h->cnt(CNT_SOR);
    } else if (!p.enable_plane) {  // (with the plane stage on, its init kernel copies the count row)
      KL(c, "k_copy_counts", k_copy_counts<<<cdiv(B, 256), 256, 0, h->stream>>>(cur_n, h->cnt(CNT_SOR), B));
      count_launch(c);
    }
  }
  h->plane_in = cur;
  h->plane_stride = cur_stride;
  h->plane_n = cur_n;
  TRY(run_wave_plane(h, B, max_n, h->expect_large_plane));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail_cuda(h, e, "stage launches", __FILE__, __LINE__);
  return PCOP_OK;
}

// Clustering + centroid / radius of one wave.  The host does not know the remaining-cloud sizes yet; with_generic =
// false launches only the fused small-cloud kernel (finish_wave repeats the stage with the generic kernels if a frame
// turned out larger, see run_cluster).
int run_wave_cluster(pcop_handle* h, int B, int max_n, bool with_generic) {
  const pcop_params& p = h->params;
  Ctx c = make_ctx(h, B, max_n);
  ClusterArgs ca = make_cluster_args(h, h->d_rem, h->cap, h->cnt(CNT_REM));
  bool generic_centroid = false;
  {
    StageTimer t(h, PCOP_STAGE_CLUSTER);
    if (p.enable_cluster) {
      generic_centroid = run_cluster(c, ca, with_generic);  // the fused small-cloud kernel writes the obstacles itself
    } else {
      cudaMemsetAsync(h->cnt(CNT_CLUS), 0, sizeof(int) * B, h->stream);
      cudaMemsetAsync(h->cnt(CNT_CLPTS), 0, sizeof(int) * B, h->stream);
    }
  }
  {
    StageTimer t(h, PCOP_STAGE_CENTROID);
    if (p.enable_cluster && generic_centroid) run_centroid_radius(c, ca);
  }
  h->wave_cluster_speculated = p.enable_cluster && !generic_centroid && max_n > h->ece_small_max;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail_cuda(h, e, "stage launches", __FILE__, __LINE__);
  return PCOP_OK;
}

// the messages of a pcop_process_batch_pointcloud2 call
struct Pc2Call {
  const pcop_pointcloud2_frame* frames;
  const float* transform16;       // [batch][16] or nullptr
  std::vector<char> on_device;    // per message: the payload is a device pointer (used in place)
};

struct WaveInput {
  const float* xyzw;
  size_t frame_stride_points;
  const int32_t* n;
  bool on_device;
  const Pc2Call* pc2;  // non-null: the frames are PointCloud2 messages, decoded into d_in by the wave (xyzw unused)
};

size_t pc2_payload_bytes(const pcop_pointcloud2_frame& m) { return (size_t)m.n_points * (size_t)m.point_step; }

// PointCloud2 wave, input half: the descriptors go up through the pinned staging (the lane's previous wave no longer
// reads it), every host payload into the lane's raw staging at a 256-byte aligned offset, device payloads are read in
// place; one k_pc2_ingest launch decodes (and transforms) every message into d_in.  A repeat of the wave (voxel
// decline) decodes again from the same staging -- the plane stage has overwritten d_in, the staging is intact.
int enqueue_wave_decode(pcop_handle* h, const Pc2Call& pc, int w0, int B, int max_n) {
  if (h->vox_redo < 0) {
    size_t off = 0;
    for (int f = 0; f < B; ++f) {
      const pcop_pointcloud2_frame& m = pc.frames[w0 + f];
      const size_t bytes = pc2_payload_bytes(m);
      const unsigned char* src = m.data;
      if (bytes > 0 && !pc.on_device[w0 + f]) {
        PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_raw + off, m.data, bytes, cudaMemcpyHostToDevice, h->stream));
        src = h->d_raw + off;
        off += (bytes + 255) & ~(size_t)255;
      }
      h->h_pc2[f] = make_pc2_frame(src, m.n_points, m.point_step, m.off_x, m.off_y, m.off_z,
                                   pc.transform16 ? pc.transform16 + (size_t)(w0 + f) * 16 : nullptr, m.is_dense);
    }
    PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_pc2, h->h_pc2, sizeof(Pc2Frame) * B, cudaMemcpyHostToDevice, h->stream));
  }
  Ctx c = make_ctx(h, B, max_n);
  KL(c, "k_pc2_ingest", k_pc2_ingest<<<dim3(cdiv(max_n, 256), B), 256, 0, h->stream>>>(h->d_pc2, h->d_in, (size_t)h->cap));
  count_launch(c);
  return PCOP_OK;
}

// Second half of a wave: clustering, result packing, and the copy of the wave's counts / plane records / pack sizes
// into pinned memory, followed by ev_meta.
int enqueue_wave_pack(pcop_handle* h, int B, int max_n, uint32_t mask) {
  // pack the requested outputs of all frames of the wave
  Ctx c = make_ctx(h, B, max_n);
  StageTimer t(h, PCOP_STAGE_D2H);
  const bool dev_results = (mask & PCOP_OUT_DEVICE) != 0;  // the arrays stay in d_pack (bump-allocated over the call)
  if (!dev_results && h->wave_seq >= 1) PCOP_CUDA_TRY(cudaStreamWaitEvent(h->stream, h->ev_copied, 0));  // d_pack is free again
  KL(c, "k_pack_scan", k_pack_scan<<<1, 320, 0, h->stream>>>(h->d_counts, h->maxB, B, mask, h->d_pack_off, h->d_meta, h->d_pf, h->d_prec,
                                             h->params.enable_plane ? 1 : 0, dev_results ? h->d_pack_cursor : nullptr,
                                             (unsigned long long)h->pack_cap));
  count_launch(c);
  const void* srcs[PK_N] = {h->d_crop_kept, h->d_vox_keys, h->d_vox,     h->d_sor_kept, h->d_inliers,
                            h->d_rem,       h->d_rem_src,  h->d_offsets, h->d_indices,  h->d_obst};
  const size_t strides[PK_N] = {(size_t)h->cap, (size_t)h->cap, (size_t)h->cap,     (size_t)h->cap, (size_t)h->cap,
                                (size_t)h->cap, (size_t)h->cap, (size_t)h->cap + 1, (size_t)h->cap, (size_t)h->cap};
  {
    PackSrc ps{};
    bool any = false;
    for (int k = 0; k < PK_N; ++k) {
      ps.src[k] = (mask & kPkMask[k]) ? (const uint32_t*)srcs[k] : nullptr;
      ps.frame_stride_words[k] = (unsigned long long)strides[k] * (kPkElem[k] / 4);
      ps.count_row[k] = kPkCount[k];
      ps.words_per_elem[k] = kPkElem[k] / 4;
      any = any || ps.src[k];
    }
    MetaOut m{};
    int nseg = 0;
    auto seg = [&](const void* src, void* dst, size_t bytes) {
      m.src[nseg] = (const uint32_t*)src;
      m.dst[nseg] = (uint32_t*)dst;
      m.words[nseg] = (int)(bytes / 4);
      ++nseg;
    };
    seg(h->d_counts, h->h_counts, sizeof(int) * CNT_ROWS * h->maxB);
    seg(h->d_warnings, h->h_warnings, sizeof(uint32_t) * B);
    seg(h->d_prec, h->h_prec, sizeof(PlaneRecord) * B);
    seg(h->d_meta, h->h_meta, sizeof(PackMeta));
    if (h->wave_used_fused) seg(h->d_vf_flags, h->h_vf_flags, sizeof(uint32_t) * B);
    static_assert(PK_N >= 5, "one pack block per metadata segment");
    if (any) {  // the (frame < 4, array k < 5) blocks of the pack kernel also carry metadata segment k out
      // (parts per (frame, array): 16 for the batched waves; a call of a few large frames gets enough to fill the GPU)
      const int gx = std::max(1, std::min(cdiv(c.grid_cap, 256 * 4), std::max(16, 592 / B)));
      m.frames = std::min(B, 4);
      KL(c, "k_pack", k_pack<<<dim3(gx, B, PK_N), 256, 0, h->stream>>>(ps, h->d_counts, h->maxB, h->d_pack_off, h->d_meta, h->d_pack, m));
      count_launch(c);
    } else {
      KL(c, "k_meta_out", k_meta_out<<<dim3(4, nseg), 256, 0, h->stream>>>(m));
      count_launch(c);
    }
  }
  if (h->trace) {
    if (h->trace_used == h->trace_recs.size()) {
      pcop_handle::TraceRec r{};
      cudaEventCreate(&r.meta);
      cudaEventCreate(&r.c0);
      cudaEventCreate(&r.c1);
      h->trace_recs.push_back(r);
    }
    cudaEventRecord(h->trace_recs[h->trace_used].meta, h->stream);
  }
  PCOP_CUDA_TRY(cudaEventRecord(h->ev_meta, h->stream));
  return PCOP_OK;
}

// Grid product, first half: the wave's poses (from the pinned staging, which the lane's previous wave no longer
// reads) and the per-cell counts of every frame.  Runs before the plane stage, whose second ping-pong cloud is d_in.
int enqueue_wave_counts(pcop_handle* h, int w0, int B, const float4* in, size_t stride, int max_n) {
  const pcop_handle::OccCall& oc = *h->occ;
  for (int f = 0; f < B; ++f) {
    memcpy(h->h_occ_mats[2 * f].m, oc.world_to_sensor16 + (size_t)(w0 + f) * 16, sizeof(Mat34));
    memcpy(h->h_occ_mats[2 * f + 1].m, oc.sensor_to_world16 + (size_t)(w0 + f) * 16, sizeof(Mat34));
  }
  PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_occ_mats, h->h_occ_mats, sizeof(Mat34) * 2 * B, cudaMemcpyHostToDevice, h->stream));
  PCOP_CUDA_TRY(cudaMemsetAsync(h->d_occ_counts, 0, sizeof(int) * (size_t)B * (size_t)oc.g.cells, h->stream));
  Ctx c = make_ctx(h, B, max_n);
  const cudaError_t e = run_occ_count_wave(c, in, stride, h->cnt(CNT_IN), oc.g, h->d_occ_counts);
  if (e != cudaSuccess) return fail_cuda(h, e, "run_occ_count_wave (shared-memory opt-in or launch)", __FILE__, __LINE__);
  return PCOP_OK;
}

// Grid product, second half (after clustering): threshold, shadows, obstacle marks.  Every repeat of the wave's back
// half rebuilds the grids from the counts, so the last repeat leaves exactly what one pass over the final clusters
// leaves.
int enqueue_wave_grids(pcop_handle* h, int B, int max_n) {
  const pcop_handle::OccCall& oc = *h->occ;
  Ctx c = make_ctx(h, B, max_n);
  PCOP_CUDA_TRY(cudaStreamWaitEvent(h->stream, h->ev_grids_copied, 0));  // the previous wave's grids have left d_occ_grids
  run_occ_finish_wave(c, h->d_occ_counts, oc.g, h->d_occ_grids, h->d_warnings);
  OccShadowArgs a{};
  a.cloud = h->d_rem;
  a.cloud_stride = h->cap;
  a.n_points = h->cnt(CNT_REM);
  a.offsets = h->d_offsets;
  a.offsets_stride = (size_t)h->cap + 1;
  a.indices = h->d_indices;
  a.indices_stride = h->cap;
  a.n_clusters = h->cnt(CNT_CLUS);
  a.mats = h->d_occ_mats;
  a.y_min = oc.g.lim[2];
  a.x_max = oc.g.lim[1];
  a.block_size = oc.g.block_size;
  a.W = oc.g.W;
  a.size = oc.g.cells;
  a.opacity = h->params.grid_opacity;
  a.grid = h->d_occ_grids;
  a.warnings = h->d_warnings;
  // (the host does not know the cluster counts: a few blocks per frame, each taking every k-th cluster)
  run_occ_shadows(c, a, std::max(4, std::min(64, cdiv(2048, B))), max_n);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail_cuda(h, e, "grid launches", __FILE__, __LINE__);
  return PCOP_OK;
}

int enqueue_wave_back(pcop_handle* h, int B, int max_n, uint32_t mask, bool cluster_with_generic) {
  TRY(run_wave_cluster(h, B, max_n, cluster_with_generic));
  if (h->occ) TRY(enqueue_wave_grids(h, B, max_n));
  return enqueue_wave_pack(h, B, max_n, mask);
}

// Enqueues one wave on lane h: input upload, all stages and enqueue_wave_back.  Returns without waiting for any of it.
int enqueue_wave(pcop_handle* h, const WaveInput& wi, int w0, int B, uint32_t mask) {
  for (int s = 0; s < PCOP_N_STAGES; ++s) h->stage_used[s] = false;
  const float4* in;
  size_t stride;
  const int32_t* n = wi.n;
  int max_n = 1;
  for (int f = 0; f < B; ++f) max_n = std::max(max_n, (int)n[w0 + f]);
  {
    StageTimer t(h, PCOP_STAGE_H2D);
    memcpy(h->h_n_in, n + w0, sizeof(int) * B);  // (the lane's previous wave has been collected: the staging is free)
    PCOP_CUDA_TRY(cudaMemcpyAsync(h->cnt(CNT_IN), h->h_n_in, sizeof(int) * B, cudaMemcpyHostToDevice, h->stream));
    if (wi.pc2) {  // from the decode on, the wave is a host-input wave
      TRY(enqueue_wave_decode(h, *wi.pc2, w0, B, max_n));
      in = h->d_in;
      stride = h->cap;
    } else if (wi.on_device) {
      in = reinterpret_cast<const float4*>(wi.xyzw) + (size_t)w0 * wi.frame_stride_points;
      stride = wi.frame_stride_points;
    } else {
      const float* src = wi.xyzw + (size_t)w0 * wi.frame_stride_points * 4;
      bool uniform = true;
      for (int f = 1; f < B; ++f) uniform = uniform && (n[w0 + f] == n[w0]);
      if (B > 0 && uniform && n[w0] > 0) {
        PCOP_CUDA_TRY(cudaMemcpy2DAsync(h->d_in, (size_t)h->cap * 16, src, wi.frame_stride_points * 16, (size_t)n[w0] * 16,
                                        B, cudaMemcpyHostToDevice, h->stream));
      } else {
        for (int f = 0; f < B; ++f)
          if (n[w0 + f] > 0)
            PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_in + (size_t)f * h->cap, src + (size_t)f * wi.frame_stride_points * 4,
                                          (size_t)n[w0 + f] * 16, cudaMemcpyHostToDevice, h->stream));
      }
      in = h->d_in;
      stride = h->cap;
    }
  }
  if (h->occ) TRY(enqueue_wave_counts(h, w0, B, in, stride, max_n));
  TRY(run_wave_stages(h, B, in, stride, max_n));
  h->pending = true;
  h->pend_w0 = w0;
  h->pend_B = B;
  h->pend_max_n = max_n;
  return enqueue_wave_back(h, B, max_n, mask, h->expect_big_remaining);
}


// Waits for the lane's wave in flight, starts its payload copy and fills out[w0 .. w0 + B).  (Result pointers into
// the pinned buffer are stored as offsets and fixed up when the call ends: the buffer may still grow.)
int finish_wave(pcop_handle* h, const WaveInput& wi, uint32_t mask, pcop_frame_result* out_all) {
  if (!h->pending) return PCOP_OK;
  const int w0 = h->pend_w0, B = h->pend_B;
  PCOP_CUDA_TRY(cudaEventSynchronize(h->ev_meta));
  if (h->wave_used_fused) {
    uint32_t fl = 0u;
    for (int f = 0; f < B; ++f) fl |= h->h_vf_flags[f];
    if (h->vox_mode == 2 && h->vox_redo < 0) {  // size the next wave's reduce grid: 1.25 x the largest frame seen, >= 64
      int mg = 0;
      for (int f = 0; f < B; ++f) mg = std::max(mg, h->h_counts[(size_t)CNT_GROUPS * h->maxB + f]);
      h->vp_group_hint = std::min(h->vp_gstride - 1, std::max(64, mg + mg / 4 + 8));
    }
    if (h->vox_lsd_waves > 0) --h->vox_lsd_waves;
    if (fl & 2u) h->vox_lsd_waves = 64;  // dense buckets tend to come back: the next waves go straight to the LSD path
    if (fl) {
      // the fused voxel path declined a frame of this wave: a survivor with a NaN y or z (generic kernels), a bucket
      // above the partition path's limit (LSD path), or more groups than the reduce grid covered (worst-case grid)
      h->vox_redo = (fl & 1u) ? 0 : ((fl & 2u) ? 1 : 2);
      h->vox_full_groups = true;
      const int st = enqueue_wave(h, wi, w0, B, mask);
      h->vox_redo = -1;
      h->vox_full_groups = false;
      TRY(st);
      PCOP_CUDA_TRY(cudaEventSynchronize(h->ev_meta));
    }
  }
  if (h->params.enable_plane && h->plane_resident) {
    bool large = false, huge = false;  // (CNT_SOR = the plane stage's input size)
    for (int f = 0; f < B; ++f) {
      const int s = h->h_counts[(size_t)CNT_SOR * h->maxB + f];
      large = large || s > plane_small_tier_max();
      huge = huge || s > plane_resident_max();
    }
    if (h->plane_hostloop_waves > 0) --h->plane_hostloop_waves;
    if (huge) h->plane_hostloop_waves = 64;  // such frames tend to come back: host-looped kernels for the next waves
    if (h->wave_plane_resident && (huge || (large && h->wave_plane_speculated))) {
      // a frame too large for the tiers that ran: repeat the wave from the plane stage on
      TRY(run_wave_plane(h, B, h->pend_max_n, true));
      TRY(enqueue_wave_back(h, B, h->pend_max_n, mask, h->expect_big_remaining));
      PCOP_CUDA_TRY(cudaEventSynchronize(h->ev_meta));
    }
    h->expect_large_plane = large;
  }
  if (h->params.enable_cluster) {
    bool big = false;
    for (int f = 0; f < B; ++f) big = big || h->h_counts[(size_t)CNT_REM * h->maxB + f] > h->ece_small_max;
    if (big && h->wave_cluster_speculated) {  // a remaining cloud too large for the fused kernel: generic clustering
      TRY(enqueue_wave_back(h, B, h->pend_max_n, mask, true));
      PCOP_CUDA_TRY(cudaEventSynchronize(h->ev_meta));
    }
    h->expect_big_remaining = big;
  }
  h->pending = false;
  pcop_frame_result* out = out_all + w0;
  const bool dev_results = (mask & PCOP_OUT_DEVICE) != 0;
  const PackMeta meta = *h->h_meta;
  if (meta.overflow)
    return fail(h, PCOP_ERR_CAPACITY, "PCOP_OUT_DEVICE: the result arrays of this call do not fit the device pack buffer");
  const size_t base_off = (h->h_pack_used + 255) & ~(size_t)255;
  if (h->trace) cudaEventRecord(h->trace_recs[h->trace_used].c0, h->cstream);
  if (!dev_results) {
    // (when the buffer has to grow, grow it for all the waves this lane will see in the call: a pinned allocation
    // costs ~0.4 ms per MB, and every regrowth copies what is already there)
    if (base_off + meta.total_bytes + 256 > h->h_pack_cap)
      TRY(ensure_host_pack(h, base_off + (size_t)((double)(meta.total_bytes + 256) * 1.1 * std::max(1, h->call_lane_waves - h->wave_seq))));
    // payload copy on the copy stream (the pack kernels have finished: ev_meta follows them), in pieces: one large
    // device-to-host copy holds up the kernels of the other lanes for as long as it runs (measured: 6.4 ms per
    // 1024-frame call with one 17 MB copy per wave, 5.7 ms with 0.5-1 MB pieces, 5.9 / 6.2 ms with 2 / 4 MB pieces,
    // 6.3 ms with 256 KB pieces -- the host thread becomes the limit -- and 5.3 ms with no copy at all)
    const size_t piece = (size_t)1 << 20;
    for (size_t o = 0; o < meta.total_bytes; o += piece)
      PCOP_CUDA_TRY(cudaMemcpyAsync(h->h_pack + base_off + o, h->d_pack + o, std::min<size_t>(piece, meta.total_bytes - o),
                                    cudaMemcpyDeviceToHost, h->cstream));
    PCOP_CUDA_TRY(cudaEventRecord(h->ev_copied, h->cstream));
    h->h_pack_used = base_off + meta.total_bytes;
  }
  if (h->occ) {  // the wave's grids, after its last repeat, on the copy stream beside the payload
    const size_t bytes = (size_t)B * (size_t)h->occ->g.cells;
    int8_t* dst = h->occ->grids + (size_t)w0 * (size_t)h->occ->g.cells;
    const unsigned char* src = reinterpret_cast<const unsigned char*>(h->d_occ_grids);
    if (h->occ->grids_on_device) {
      PCOP_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, h->cstream));
    } else {
      const size_t piece = (size_t)1 << 20;  // (pieces: as the payload above)
      for (size_t o = 0; o < bytes; o += piece)
        PCOP_CUDA_TRY(cudaMemcpyAsync(dst + o, src + o, std::min<size_t>(piece, bytes - o), cudaMemcpyDeviceToHost, h->cstream));
      h->d2h_bytes += (double)bytes;
    }
    PCOP_CUDA_TRY(cudaEventRecord(h->ev_grids_copied, h->cstream));
  }
  if (h->trace) {
    pcop_handle::TraceRec& tr = h->trace_recs[h->trace_used++];
    cudaEventRecord(tr.c1, h->cstream);
    tr.w0 = w0;
    tr.B = B;
    tr.bytes = dev_results ? 0 : (size_t)meta.total_bytes;
  }
  h->d2h_bytes += (dev_results ? 0.0 : (double)meta.total_bytes) +
                  (double)(sizeof(int) * CNT_ROWS * h->maxB + sizeof(uint32_t) * B + sizeof(PlaneRecord) * B + sizeof(PackMeta));
  ++h->wave_seq;

  size_t run[PK_N] = {0};
  auto H = [&](int row, int f) { return h->h_counts[(size_t)row * h->maxB + f]; };
  for (int f = 0; f < B; ++f) {
    pcop_frame_result& r = out[f];
    memset(&r, 0, sizeof(r));
    r.status = PCOP_OK;
    r.warnings = h->h_warnings[f];
    r.n_input = H(CNT_IN, f);
    r.n_crop = H(CNT_CROP, f);
    r.n_voxel = H(CNT_VOX, f);
    r.n_sor = H(CNT_SOR, f);
    r.n_remaining = H(CNT_REM, f);
    r.n_clusters = H(CNT_CLUS, f);
    r.n_cluster_points = H(CNT_CLPTS, f);
    const PlaneRecord& pr = h->h_prec[f];
    r.n_plane_passes = pr.n_passes;
    r.n_plane_inliers = pr.n_inliers_last;
    memcpy(r.plane_coeff, &pr.coeff, 16);
    memcpy(r.plane_pass_points, pr.pass_points, sizeof(pr.pass_points));
    memcpy(r.plane_pass_inliers, pr.pass_inliers, sizeof(pr.pass_inliers));
    memcpy(r.plane_pass_coeff, pr.pass_coeff, sizeof(pr.pass_coeff));
    const void** slots[PK_N] = {(const void**)&r.crop_kept_idx,    (const void**)&r.voxel_keys,
                                (const void**)&r.voxel_centroids,  (const void**)&r.sor_kept_idx,
                                (const void**)&r.plane_inlier_idx, (const void**)&r.remaining_cloud,
                                (const void**)&r.remaining_src_idx, (const void**)&r.cluster_offsets,
                                (const void**)&r.cluster_indices,  (const void**)&r.obstacles};
    for (int k = 0; k < PK_N; ++k) {
      if (!(mask & kPkMask[k])) continue;
      if (dev_results) {  // device pointer into the pack buffer (it does not move)
        *slots[k] = h->d_pack + (size_t)meta.base[k] + run[k] * kPkElem[k];
      } else {
        // store the byte offset now; turned into a pointer once the host buffer can no longer move
        const size_t off = base_off + (size_t)meta.base[k] + run[k] * kPkElem[k];
        *slots[k] = (const void*)(uintptr_t)(off + 1);  // +1 so that offset 0 is distinguishable from NULL
        h->fixups.push_back((size_t)((const unsigned char*)slots[k] - (const unsigned char*)out_all));
      }
      run[k] += (size_t)H(kPkCount[k], f);
    }
    // algorithmic bytes (SURVEY 8d)
    double b = 0.0;
    const pcop_params& p = h->params;
    if (wi.pc2) b += (double)(wi.pc2->frames[w0 + f].point_step + 16) * r.n_input;  // the decode: payload in, PointXYZ out
    if (p.enable_crop) b += 16.0 * r.n_input + 20.0 * r.n_crop;
    if (p.enable_voxel) b += 16.0 * r.n_crop + 20.0 * r.n_voxel;
    if (p.enable_sor) b += 16.0 * r.n_voxel + 20.0 * r.n_sor;
    if (p.enable_plane) {
      int pk = r.n_sor;
      const int np = std::min(r.n_plane_passes, (int)PCOP_MAX_PLANE_PASSES_RECORDED);
      for (int k = 0; k < np; ++k) {
        const int ik = r.plane_pass_inliers[k];
        b += 16.0 * pk + 16.0 * (pk - ik) + 4.0 * ik + 16.0;
        pk -= ik;
      }
    }
    if (p.enable_cluster) {
      b += 16.0 * r.n_remaining + 4.0 * r.n_cluster_points + 4.0 * (r.n_clusters + 1);
      b += 16.0 * r.n_remaining + 4.0 * r.n_cluster_points + 16.0 * r.n_clusters;
    }
    h->alg_bytes += b;
  }
  for (int s = 0; s < PCOP_N_STAGES; ++s) {
    if (!h->stage_used[s]) continue;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev_stage[s][0], h->ev_stage[s][1]) == cudaSuccess) h->stage_us[s] += ms * 1000.f;
    else cudaGetLastError();
  }
  resolve_kernel_timers(h);
  return PCOP_OK;
}

// add lane `l`'s per-kernel timing table into h's and clear it
void merge_kernel_timers(pcop_handle* h, pcop_handle* l) {
  KernelTimers& d = h->kt;
  KernelTimers& s = l->kt;
  for (int i = 0; i < s.n_names; ++i) {
    int id = -1;
    for (int j = 0; j < d.n_names; ++j)
      if (d.names[j] == s.names[i] || strcmp(d.names[j], s.names[i]) == 0) {
        id = j;
        break;
      }
    if (id < 0 && d.n_names < KernelTimers::MAX_NAMES) {
      id = d.n_names++;
      d.names[id] = s.names[i];
      d.total_us[id] = 0.0;
      d.launches[id] = 0;
    }
    if (id >= 0) {
      d.total_us[id] += s.total_us[i];
      d.launches[id] += s.launches[i];
    }
  }
  s.n_names = 0;
}

static std::chrono::steady_clock::time_point g_trace_t0;
static double trace_host_us() {
  return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - g_trace_t0).count();
}

// occupancy grid scratch of one lane for waves of `frames` frames of `cells` cells (grown, never shrunk)
int ensure_occ_scratch(pcop_handle* h, size_t frames, size_t cells) {
  if (!h->d_occ_mats) {
    TRY(dalloc(h, &h->d_occ_mats, 2 * (size_t)h->maxB));
    TRY(halloc(h, &h->h_occ_mats, 2 * (size_t)h->maxB));
  }
  const size_t need = frames * cells;
  if (need <= h->occ_scratch_cells) return PCOP_OK;
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->cstream));
  if (h->d_occ_counts) cudaFree(h->d_occ_counts);  // (not tracked in dev_allocs)
  if (h->d_occ_grids) cudaFree(h->d_occ_grids);
  h->d_occ_counts = nullptr;
  h->d_occ_grids = nullptr;
  h->occ_scratch_cells = 0;
  PCOP_CUDA_TRY(cudaMalloc((void**)&h->d_occ_counts, sizeof(int) * need));
  PCOP_CUDA_TRY(cudaMalloc((void**)&h->d_occ_grids, need));
  h->occ_scratch_cells = need;
  return PCOP_OK;
}

// occ: the grid product of every frame as well (pcop_process_batch_occupancy), nullptr: pcop_process_batch
// pc2: the frames are PointCloud2 messages (pcop_process_batch_pointcloud2; xyzw unused, n = their record counts)
int process_impl(pcop_handle* h, const float* xyzw, size_t frame_stride_points, const int32_t* n, int32_t batch,
                 pcop_frame_result* out, const pcop_handle::OccCall* occ = nullptr, const Pc2Call* pc2 = nullptr) {
  if (!h) return fail(nullptr, PCOP_ERR_BAD_PARAM, "null handle");
  if ((!xyzw && !pc2) || !n || !out || batch < 0) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  for (int f = 0; f < batch; ++f) {
    if (n[f] < 0) return fail(h, PCOP_ERR_BAD_PARAM, "negative point count");
    if (n[f] > h->cap) return fail(h, PCOP_ERR_CAPACITY, "frame has more points than max_points");
    if ((size_t)n[f] > frame_stride_points && batch > 1) return fail(h, PCOP_ERR_BAD_PARAM, "frame_stride_points < n");
  }
  const uint32_t mask = effective_outputs(h->params);
  const WaveInput wi{xyzw, frame_stride_points, n, pc2 ? false : is_device_pointer(xyzw), pc2};
  // lanes used by this call: per-kernel timing needs each kernel alone on the GPU, so it serialises the lanes
  std::vector<pcop_handle*> lanes(1, h);
  if (!h->kt.enabled)
    for (pcop_handle* l : h->extra_lanes) lanes.push_back(l);
  // waves: about wave_frames frames each (never more than a lane holds), at least one per lane when the call is large
  // enough, the last one half as large as the others (its result copy is the only one nothing overlaps).  Measured on
  // B200 (1024 HDL-64 frames, 3 lanes, results to the host): waves of 256 / 192 / 128 / 96 frames 6.73 / 6.88 / 6.25 /
  // 6.36 ms per call; a tail of one quarter-size wave per lane 6.39 ms (a wave has a latency floor of ~0.7 ms
  // whatever its size, so small tail waves cost more than their copies save).
  std::vector<std::pair<int, int>> waves;  // (first frame, frames)
  {
    const int L = (int)lanes.size();
    int nw = std::max(1, cdiv(batch, std::max(1, std::min(h->wave_frames, h->maxB))));
    if (nw < L) nw = std::max(1, std::min(L, batch / PCOP_MIN_LANE_WAVE));
    const int full = (nw > 1) ? std::min(h->maxB, cdiv(2 * batch, 2 * nw - 1)) : std::min(h->maxB, batch);
    for (int w0 = 0; w0 < batch;) {
      const int B = std::min(full, batch - w0);
      waves.push_back({w0, B});
      w0 += B;
    }
  }
  size_t raw_need = 0;  // PointCloud2 messages: host payload bytes of the largest wave, as staged (256-byte aligned)
  if (pc2)
    for (const auto& w : waves) {
      size_t bytes = 0;
      for (int f = w.first; f < w.first + w.second; ++f)
        if (!pc2->on_device[f]) bytes += (pc2_payload_bytes(pc2->frames[f]) + 255) & ~(size_t)255;
      raw_need = std::max(raw_need, bytes);
    }
  h->occ = nullptr;  // (lanes the call does not use must not see a previous call's grid request)
  for (pcop_handle* l : h->extra_lanes) l->occ = nullptr;
  for (pcop_handle* l : lanes) {
    l->occ = occ;
    if (occ && !waves.empty()) TRY(ensure_occ_scratch(l, (size_t)waves[0].second, (size_t)occ->g.cells));  // (the first wave is the largest)
    if (raw_need) TRY(ensure_raw(l, raw_need));
    l->params = h->params;
    l->vplan = h->vplan;
    l->vox_mode = h->vox_mode;
    l->launches = 0;
    l->alg_bytes = 0.0;
    l->d2h_bytes = 0.0;
    l->kt.used = 0;
    l->sort_pass_keys = 0;
    l->h_pack_used = 0;
    l->h_pack_sel ^= 1;
    l->h_pack = l->h_pack_buf[l->h_pack_sel];
    l->h_pack_cap = l->h_pack_buf_cap[l->h_pack_sel];
    l->fixups.clear();
    l->wave_seq = 0;
    l->call_lane_waves = cdiv((int)waves.size(), (int)lanes.size());
    l->trace_used = 0;
    l->pending = false;
    for (int s = 0; s < PCOP_N_STAGES; ++s) l->stage_us[s] = 0.f;
    TRY(ensure_pack_capacity(l, mask));
  }
  PCOP_CUDA_TRY(cudaEventRecord(h->ev_call[0], h->stream));
  if (h->trace) g_trace_t0 = std::chrono::steady_clock::now();
  for (size_t l = 0; l < lanes.size(); ++l) {
    if (l > 0) PCOP_CUDA_TRY(cudaStreamWaitEvent(lanes[l]->stream, h->ev_call[0], 0));
    PCOP_CUDA_TRY(cudaMemsetAsync(lanes[l]->sort.stats, 0, sizeof(unsigned long long), lanes[l]->stream));
    if (mask & PCOP_OUT_DEVICE)
      PCOP_CUDA_TRY(cudaMemsetAsync(lanes[l]->d_pack_cursor, 0, sizeof(unsigned long long), lanes[l]->stream));
  }
  int status = PCOP_OK;
  for (size_t w = 0; w < waves.size() && status == PCOP_OK; ++w) {
    pcop_handle* l = lanes[w % lanes.size()];
    const double th0 = h->trace ? trace_host_us() : 0.0;
    status = finish_wave(l, wi, mask, out);  // (the lane's previous wave, if any)
    const double th1 = h->trace ? trace_host_us() : 0.0;
    if (status == PCOP_OK) status = enqueue_wave(l, wi, waves[w].first, waves[w].second, mask);
    if (h->trace)
      fprintf(stderr, "[pcop trace]   host: wave %4d+%-4d lane %zu: finish of the lane's previous wave %7.0f .. %7.0f us, enqueue .. %7.0f us\n",
              waves[w].first, waves[w].second, w % lanes.size(), th0, th1, trace_host_us());
    if (status != PCOP_OK && l != h) h->err = l->err;
  }
  // collect what is still in flight, oldest first
  for (size_t k = 0; k < lanes.size(); ++k) {
    pcop_handle* l = lanes[(waves.size() + k) % lanes.size()];
    const int st = finish_wave(l, wi, mask, out);
    if (st != PCOP_OK && status == PCOP_OK) {
      status = st;
      if (l != h) h->err = l->err;
    }
  }
  for (pcop_handle* l : lanes) {  // the call is done when every lane's last result copy has landed
    cudaMemcpyAsync(l->h_stats, l->sort.stats, sizeof(unsigned long long), cudaMemcpyDeviceToHost, l->stream);
    cudaEventRecord(l->ev_lane_done, l->cstream);
    cudaStreamWaitEvent(l->stream, l->ev_lane_done, 0);
    cudaEventRecord(l->ev_lane_done, l->stream);
    if (l != h) cudaStreamWaitEvent(h->stream, l->ev_lane_done, 0);
  }
  PCOP_CUDA_TRY(cudaEventRecord(h->ev_call[1], h->stream));
  PCOP_CUDA_TRY(cudaEventSynchronize(h->ev_call[1]));
  if (status != PCOP_OK) return status;
  float ms = 0.f;
  PCOP_CUDA_TRY(cudaEventElapsedTime(&ms, h->ev_call[0], h->ev_call[1]));
  h->last_elapsed_us = ms * 1000.f;
  if (h->trace) {
    fprintf(stderr, "[pcop trace] call of %d frames: %.0f us on the device\n", batch, ms * 1000.f);
    for (size_t li = 0; li < lanes.size(); ++li) {
      for (size_t k = 0; k < lanes[li]->trace_used; ++k) {
        const pcop_handle::TraceRec& tr = lanes[li]->trace_recs[k];
        float a = 0.f, b = 0.f, c = 0.f;
        cudaEventElapsedTime(&a, h->ev_call[0], tr.meta);
        cudaEventElapsedTime(&b, h->ev_call[0], tr.c0);
        cudaEventElapsedTime(&c, h->ev_call[0], tr.c1);
        fprintf(stderr, "[pcop trace]   lane %zu wave %4d+%-4d counts at %7.0f us, payload copy %7.0f .. %7.0f us (%.1f MB, %.1f GB/s)\n", li,
                tr.w0, tr.B, a * 1000.f, b * 1000.f, c * 1000.f, tr.bytes / 1e6, tr.bytes / 1e3 / std::max(1e-3f, (c - b) * 1000.f));
      }
      lanes[li]->trace_used = 0;
    }
    cudaGetLastError();
  }
  for (pcop_handle* l : lanes) {
    l->sort_pass_keys = *l->h_stats;
    // the host pack buffers are final now: turn the stored offsets into pointers
    for (size_t fx : l->fixups) {
      const void** slot = (const void**)((unsigned char*)out + fx);
      const size_t off = (size_t)(uintptr_t)(*slot) - 1;
      *slot = l->h_pack + off;
    }
    if (l == h) continue;  // per-call accounting is reported on the handle (sums over the lanes)
    h->launches += l->launches;
    h->alg_bytes += l->alg_bytes;
    h->d2h_bytes += l->d2h_bytes;
    h->sort_pass_keys += l->sort_pass_keys;
    for (int s = 0; s < PCOP_N_STAGES; ++s) h->stage_us[s] += l->stage_us[s];
    merge_kernel_timers(h, l);
  }
  return PCOP_OK;
}

// upload a single cloud into d_in as frame 0 and set a count row
int upload_single(pcop_handle* h, const float* xyzw, int32_t n, int count_row) {
  if (n < 0) return fail(h, PCOP_ERR_BAD_PARAM, "negative point count");
  if (n > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  h->h_n_in[0] = n;
  PCOP_CUDA_TRY(cudaMemcpyAsync(h->cnt(count_row), h->h_n_in, sizeof(int), cudaMemcpyHostToDevice, h->stream));
  if (n > 0) PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_in, xyzw, (size_t)n * 16, cudaMemcpyDefault, h->stream));
  k_zero_u32<<<1, 32, 0, h->stream>>>(h->d_warnings, 1);
  return PCOP_OK;
}

int download(pcop_handle* h, void* dst, const void* src, size_t bytes) {
  if (!dst || bytes == 0) return PCOP_OK;
  PCOP_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->stream));
  return PCOP_OK;
}

int fetch_count(pcop_handle* h, int row, int32_t* out) {
  PCOP_CUDA_TRY(cudaMemcpyAsync(h->h_counts, h->cnt(row), sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  *out = h->h_counts[0];
  return PCOP_OK;
}

int fetch_warnings(pcop_handle* h, uint32_t* w) {
  PCOP_CUDA_TRY(cudaMemcpyAsync(h->h_warnings, h->d_warnings, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (w) *w = h->h_warnings[0];
  return PCOP_OK;
}

}  // namespace

// =====================================================================================
extern "C" {

int pcop_abi_version(void) { return PCOP_ABI_VERSION; }
const char* pcop_global_error(void) { return g_global_error.c_str(); }
const char* pcop_last_error(const pcop_handle* h) { return h ? h->err.c_str() : g_global_error.c_str(); }

void pcop_params_init_code_defaults(pcop_params* p) {
  memset(p, 0, sizeof(*p));
  // od.cpp:948-953
  p->x_min = -1.0f; p->x_max = 1.0f; p->y_min = -0.5f; p->y_max = 0.6f; p->z_min = 0.0f; p->z_max = -0.5f;
  p->downsample_size = 0.015f;                   // od.cpp:964
  p->statistical_outlier_meanK = 15;             // od.cpp:966
  p->statistical_outlier_stdDevThres = 1.0f;     // od.cpp:967
  p->plane_segment_dist_thres = 0.040f;          // od.cpp:969
  p->plane_segment_angle = 20;                   // od.cpp:970
  p->euc_cluster_tolerance = 0.4f;               // od.cpp:972
  p->euc_min_cluster_size = 5;                   // od.cpp:973
  p->euc_max_cluster_size = 20000;               // od.cpp:974
  p->plane_axis[0] = 0.0f; p->plane_axis[1] = 0.0f; p->plane_axis[2] = 1.0f;  // od.cpp:769
  p->plane_keep_fraction = 0.3;                  // od.cpp:379
  p->plane_max_iterations = 50;                  // pcl::SACSegmentation default
  p->plane_probability = 0.99;                   // pcl::SACSegmentation default
  p->ransac_seed = 12345u;                       // pcl::SampleConsensusModel rng seed
  p->optimize_coefficients = 1;                  // od.cpp:365
  p->enable_crop = p->enable_voxel = p->enable_sor = p->enable_plane = p->enable_cluster = 1;
  p->publish_point_clouds = 1;                   // od.cpp:945
  p->outputs = PCOP_OUT_DEFAULT;
  p->accumulate_count = 2;                       // od.cpp:940
  p->block_size = 0.15f;                         // od.cpp:955
  p->dev_percent = 0.5f;                         // od.cpp:956
  p->grid_opacity = 0;                           // od.cpp:946
  p->downsample_input_data = 1;                  // od.cpp:943
  p->passthrough_filter_enable = 1;              // od.cpp:944
  p->convex_hull_alpha = 180.0f;                 // od.cpp:975
}

void pcop_params_init_params_yaml(pcop_params* p) {
  pcop_params_init_code_defaults(p);
  // minibot_cr18/params.yaml:2-31
  p->x_min = 0.0f; p->x_max = 4.5f; p->y_min = 0.0f; p->y_max = 3.78f; p->z_min = -0.5f; p->z_max = 0.25f;
  p->accumulate_count = 200;
  p->block_size = 0.0375f;
  p->dev_percent = 0.9f;
  p->grid_opacity = 0;
  p->downsample_size = 0.015f;
  p->statistical_outlier_meanK = 15;
  p->statistical_outlier_stdDevThres = 4.0f;
  p->plane_segment_dist_thres = 0.040f;
  p->plane_segment_angle = 20;
  p->euc_cluster_tolerance = 0.4f;
  p->euc_min_cluster_size = 5;
  p->euc_max_cluster_size = 20000;
  p->convex_hull_alpha = 180.0f;
  p->publish_point_clouds = 1;
}

static int create_lane(const pcop_params* params, int device, size_t max_points, int max_batch, pcop_handle** out) {
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(nullptr, PCOP_ERR_CUDA, "pcop_create: no CUDA device (this library has no CPU fallback)");
  }
  if (device < 0 || device >= ndev) return fail(nullptr, PCOP_ERR_BAD_PARAM, "pcop_create: bad device index");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail_cuda(nullptr, e, "props", __FILE__, __LINE__);
  if (prop.major != 10)
    return fail(nullptr, PCOP_ERR_CUDA, "pcop_create: device is not sm_100-class (kernels are built for sm_100a only)");
  pcop_handle* h = new pcop_handle();
  h->params = *params;
  h->vplan = make_plan(*params, max_points, &h->vox_mode);
  h->device = device;
  h->cap = (int)max_points;
  h->maxB = max_batch;
  int st = validate_params(h, *params);
  if (st != PCOP_OK) {
    g_global_error = h->err;
    delete h;
    return st;
  }
  auto bail = [&](int code) {
    g_global_error = h->err;
    pcop_destroy(h);
    return code;
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(fail_cuda(h, e, "cudaSetDevice", __FILE__, __LINE__));
  if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess)
    return bail(fail_cuda(h, e, "cudaStreamCreate", __FILE__, __LINE__));
  const size_t BC = (size_t)h->maxB * h->cap;
  const int B = h->maxB;
  const int chunks = cdiv(h->cap, TS_CHUNK);
  const int tiles = cdiv(h->cap, CT_TILE);
#define A(x)                         \
  do {                               \
    int _s = (x);                    \
    if (_s != PCOP_OK) return bail(_s); \
  } while (0)
  A(dalloc(h, &h->d_in, BC));
  A(dalloc(h, &h->d_acc, (size_t)h->cap));
  A(dalloc(h, &h->d_crop, BC));
  A(dalloc(h, &h->d_vox, BC));
  A(dalloc(h, &h->d_sor, BC));
  // plane ping-pong clouds (only frames that need a second pass touch them): the cropped cloud and the input staging
  // are dead by then (the fused voxel path gathers from the caller's / staged input before the plane stage starts)
  h->d_pbuf[0] = h->d_crop;
  h->d_pbuf[1] = h->d_in;
  A(dalloc(h, &h->d_rem, BC));
  A(dalloc(h, &h->d_sorted, BC));
  A(dalloc(h, &h->d_obst, BC));
  A(dalloc(h, &h->d_crop_kept, BC));
  A(dalloc(h, &h->d_run_start, BC));
  A(dalloc(h, &h->d_sor_kept, BC));
  A(dalloc(h, &h->d_psrc[0], BC));
  A(dalloc(h, &h->d_psrc[1], BC));
  A(dalloc(h, &h->d_rem_src, BC));
  A(dalloc(h, &h->d_inliers, BC));
  A(dalloc(h, &h->d_parent, BC));
  A(dalloc(h, &h->d_csize, BC));
  A(dalloc(h, &h->d_roots, BC));
  A(dalloc(h, &h->d_rank, BC));
  A(dalloc(h, &h->d_indices, BC));
  A(dalloc(h, &h->d_cell_start, BC));
  A(dalloc(h, &h->d_cell_key, BC));
  A(dalloc(h, &h->d_offsets, BC + B));
  A(dalloc(h, &h->d_vox_keys, BC));
  A(dalloc(h, &h->d_sor_dist, BC));
  A(dalloc(h, &h->sort.key[0], BC));
  A(dalloc(h, &h->sort.key[1], BC));
  A(dalloc(h, &h->sort.val[0], BC));
  A(dalloc(h, &h->sort.val[1], BC));
  A(dalloc(h, &h->sort.hist, std::max((size_t)B * RS_MAX_PASSES * RS_BINS, vox_fused_hist_elems(B))));
  {
    unsigned char* d = nullptr;
    A(dalloc(h, &d, std::max(sort_desc_bytes(B, h->cap), vox_fused_desc_bytes(B, h->cap))));
    h->sort.desc = (uint32_t*)d;
  }
  A(dalloc(h, &h->d_vf_flags, B));
  if (h->vplan.part_ok) {
    h->vp_gstride = vox_part_group_bound(h->vplan, h->cap) + 1;
    h->vp_group_hint = h->vp_gstride - 1;
    A(dalloc(h, &h->d_vp_hist, vox_part_hist_elems(B)));
    A(dalloc(h, &h->d_vp_bstart, vox_part_chunk_start_elems(B)));
    A(dalloc(h, &h->d_vp_nstart, vox_part_start_elems(B)));
    A(dalloc(h, &h->d_vp_ne, vox_part_bucket_elems(B)));
    A(dalloc(h, &h->d_vp_grec, (size_t)B * h->vp_gstride));
    A(dalloc(h, &h->d_vp_desc, (size_t)B * h->vp_gstride));
  }
  // (key, index) pairs of the fused voxel path: they overlay the search-grid point list of SOR / clustering
  h->d_vf_pair[0] = reinterpret_cast<unsigned long long*>(h->d_sorted);
  h->d_vf_pair[1] = reinterpret_cast<unsigned long long*>(h->d_sorted) + BC;
  A(halloc(h, &h->h_vf_flags, B));
  A(dalloc(h, &h->sort.maxkey, B));
  A(dalloc(h, &h->sort.npass, B));
  A(dalloc(h, &h->sort.stats, 1));
  A(halloc(h, &h->h_stats, 1));
  A(dalloc(h, &h->d_desc, (size_t)B * tiles));
  A(dalloc(h, &h->d_counts, (size_t)CNT_ROWS * B));
  A(dalloc(h, &h->d_warnings, B));
  A(dalloc(h, &h->d_minmax, B));
  A(dalloc(h, &h->d_vf, B));
  A(dalloc(h, &h->d_ef, B));
  A(dalloc(h, &h->d_pf, B));
  A(dalloc(h, &h->d_prec, B));
  A(dalloc(h, &h->d_partial, (size_t)B * chunks * 10));
  A(dalloc(h, &h->d_thr, B));
  A(dalloc(h, &h->d_n_active, 64));
  A(dalloc(h, &h->d_rng, RNG_TABLE));
  A(dalloc(h, &h->d_pack_off, (size_t)PK_N * B));
  A(dalloc(h, &h->d_meta, 1));
  A(dalloc(h, &h->d_pack_cursor, 1));
  A(dalloc(h, &h->d_pc2, B));
  A(halloc(h, &h->h_pc2, B));
  A(halloc(h, &h->h_n_active, 16));
  A(halloc(h, &h->h_counts, (size_t)CNT_ROWS * B));
  A(halloc(h, &h->h_warnings, B));
  A(halloc(h, &h->h_prec, B));
  A(halloc(h, &h->h_meta, 1));
  A(halloc(h, &h->h_n_in, (size_t)B + 16));
#undef A
  if ((e = cudaMemset(h->d_counts, 0, sizeof(int) * CNT_ROWS * B)) != cudaSuccess)
    return bail(fail_cuda(h, e, "memset", __FILE__, __LINE__));
  if ((e = cudaMemset(h->d_pf, 0, sizeof(PlaneFrame) * B)) != cudaSuccess)
    return bail(fail_cuda(h, e, "memset", __FILE__, __LINE__));
  {
    std::vector<int> tbl(RNG_TABLE);
    fill_rng_table(params->ransac_seed, tbl.data(), RNG_TABLE);
    if ((e = cudaMemcpy(h->d_rng, tbl.data(), sizeof(int) * RNG_TABLE, cudaMemcpyHostToDevice)) != cudaSuccess)
      return bail(fail_cuda(h, e, "rng upload", __FILE__, __LINE__));
  }
  for (int i = 0; i < 2; ++i)
    if ((e = cudaEventCreate(&h->ev_call[i])) != cudaSuccess) return bail(fail_cuda(h, e, "event", __FILE__, __LINE__));
  for (int s = 0; s < PCOP_N_STAGES; ++s)
    for (int i = 0; i < 2; ++i)
      if ((e = cudaEventCreate(&h->ev_stage[s][i])) != cudaSuccess)
        return bail(fail_cuda(h, e, "event", __FILE__, __LINE__));
  if ((e = cudaEventCreateWithFlags(&h->ev_lane_done, cudaEventDisableTiming)) != cudaSuccess)
    return bail(fail_cuda(h, e, "event", __FILE__, __LINE__));
  if ((e = cudaStreamCreateWithFlags(&h->cstream, cudaStreamNonBlocking)) != cudaSuccess)
    return bail(fail_cuda(h, e, "cudaStreamCreate", __FILE__, __LINE__));
  if ((e = cudaEventCreateWithFlags(&h->ev_copied, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_meta, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_grids_copied, cudaEventDisableTiming)) != cudaSuccess)
    return bail(fail_cuda(h, e, "event", __FILE__, __LINE__));
  st = ensure_pack_capacity(h, effective_outputs(h->params));
  if (st != PCOP_OK) return bail(st);
  *out = h;
  return PCOP_OK;
}

int pcop_create(const pcop_params* params, int device, size_t max_points, int max_batch, pcop_handle** out) {
  // (frame-major launches put the tile index in gridDim.y, and look-back descriptors carry 30-bit prefixes)
  if (!params || !out || max_points == 0 || max_points > (size_t)65535 * BT_TILE || max_batch < 1)
    return fail(nullptr, PCOP_ERR_BAD_PARAM, "pcop_create: bad argument (max_points must be in [1, 268431360])");
  *out = nullptr;
  // Lanes (PCOP_LANES, default 3 once max_batch allows waves of 64 frames): every lane owns the buffers of one wave;
  // a batched call keeps one wave in flight per lane.  Wave size (PCOP_WAVE_FRAMES, default max_batch / 8, at least
  // 64): large enough to fill the GPU, small enough that the last wave's result copy -- the only one nothing
  // overlaps -- is short.  Both knobs are read here, once; nothing on the frame path looks at the environment.
  int wave_frames = std::min(max_batch, std::max(64, max_batch / 8));
  if (const char* s = getenv("PCOP_WAVE_FRAMES")) wave_frames = (int)std::min<long>(std::max<long>(strtol(s, nullptr, 10), 1), max_batch);
  int n_lanes = std::max(1, std::min(3, max_batch / wave_frames));
  if (const char* s = getenv("PCOP_LANES")) n_lanes = (int)std::min<long>(std::max<long>(strtol(s, nullptr, 10), 1), 8);
  n_lanes = std::max(1, std::min(n_lanes, max_batch / PCOP_MIN_LANE_WAVE));
  const int lane_batch = n_lanes == 1 ? max_batch : std::min(max_batch, wave_frames + wave_frames / 4);
  pcop_handle* h = nullptr;
  int st = create_lane(params, device, max_points, lane_batch, &h);
  if (st != PCOP_OK) return st;
  for (int l = 1; l < n_lanes; ++l) {
    pcop_handle* x = nullptr;
    st = create_lane(params, device, max_points, lane_batch, &x);
    if (st != PCOP_OK) {
      pcop_destroy(h);
      return st;
    }
    h->extra_lanes.push_back(x);
  }
  h->wave_frames = std::min(wave_frames, lane_batch);
  h->trace = getenv("PCOP_TRACE") != nullptr;
  for (pcop_handle* l : h->extra_lanes) l->trace = h->trace;
  h->ece_small_max = ece_small_limit();
  if (const char* s = getenv("PCOP_PLANE_RESIDENT")) h->plane_resident = (s[0] == '0') ? 0 : 1;  // (the tests cover both paths)
  for (pcop_handle* l : h->extra_lanes) {
    l->ece_small_max = h->ece_small_max;
    l->plane_resident = h->plane_resident;
  }
  *out = h;
  return PCOP_OK;
}

void pcop_destroy(pcop_handle* h) {
  if (!h) return;
  for (pcop_handle* l : h->extra_lanes) pcop_destroy(l);
  h->extra_lanes.clear();
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->cstream) cudaStreamSynchronize(h->cstream);
  for (void* p : h->dev_allocs) cudaFree(p);
  for (void* p : h->host_allocs) cudaFreeHost(p);
  if (h->d_pack) cudaFree(h->d_pack);
  if (h->d_raw) cudaFree(h->d_raw);
  if (h->d_occ) cudaFree(h->d_occ);
  if (h->d_shadow) cudaFree(h->d_shadow);
  if (h->d_occ_counts) cudaFree(h->d_occ_counts);
  if (h->d_occ_grids) cudaFree(h->d_occ_grids);
  for (int i = 0; i < 2; ++i)
    if (h->h_pack_buf[i]) cudaFreeHost(h->h_pack_buf[i]);
  if (h->kt.ev) {
    for (int i = 0; i < 2 * KernelTimers::MAX_SLOTS; ++i) cudaEventDestroy(h->kt.ev[i]);
    delete[] h->kt.ev;
  }
  for (int i = 0; i < 2; ++i)
    if (h->ev_call[i]) cudaEventDestroy(h->ev_call[i]);
  if (h->ev_lane_done) cudaEventDestroy(h->ev_lane_done);
  if (h->ev_copied) cudaEventDestroy(h->ev_copied);
  if (h->ev_meta) cudaEventDestroy(h->ev_meta);
  if (h->ev_grids_copied) cudaEventDestroy(h->ev_grids_copied);
  if (h->cstream) cudaStreamDestroy(h->cstream);
  for (int s = 0; s < PCOP_N_STAGES; ++s)
    for (int i = 0; i < 2; ++i)
      if (h->ev_stage[s][i]) cudaEventDestroy(h->ev_stage[s][i]);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

int pcop_set_params(pcop_handle* h, const pcop_params* params) {
  if (!h || !params) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  int st = validate_params(h, *params);
  if (st != PCOP_OK) return st;
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (params->ransac_seed != h->params.ransac_seed) {
    std::vector<int> tbl(RNG_TABLE);
    fill_rng_table(params->ransac_seed, tbl.data(), RNG_TABLE);
    PCOP_CUDA_TRY(cudaMemcpy(h->d_rng, tbl.data(), sizeof(int) * RNG_TABLE, cudaMemcpyHostToDevice));
  }
  h->params = *params;
  h->vplan = make_plan(*params, (size_t)h->cap, &h->vox_mode);
  h->vox_lsd_waves = 0;
  h->plane_hostloop_waves = 0;
  for (pcop_handle* l : h->extra_lanes) {
    const int ls = pcop_set_params(l, params);
    if (ls != PCOP_OK) {
      h->err = l->err;
      return ls;
    }
  }
  return ensure_pack_capacity(h, effective_outputs(h->params));
}

int pcop_process(pcop_handle* h, const float* xyzw, int32_t n, pcop_frame_result* out) {
  return process_impl(h, xyzw, (size_t)(n > 0 ? n : 1), &n, 1, out);
}

int pcop_process_batch(pcop_handle* h, const float* xyzw, size_t frame_stride_points, const int32_t* n, int32_t batch,
                       pcop_frame_result* out) {
  return process_impl(h, xyzw, frame_stride_points, n, batch, out);
}

static int occ_grid_of(pcop_handle* h, OccGrid* g);

// the grid request of a batched call: the handle's grid (PCOP_ERR_CAPACITY above PCOP_OCC_BATCH_MAX_CELLS) + poses
static int occ_call_of(pcop_handle* h, const char* who, const float* world_to_sensor16, const float* sensor_to_world16,
                       int8_t* grids, pcop_handle::OccCall* oc) {
  TRY(occ_grid_of(h, &oc->g));
  if (oc->g.cells > PCOP_OCC_BATCH_MAX_CELLS)
    return fail(h, PCOP_ERR_CAPACITY,
                std::string(who) + ": grid of " + std::to_string(oc->g.W) + " x " + std::to_string(oc->g.H) +
                    " cells exceeds PCOP_OCC_BATCH_MAX_CELLS (use pcop_occupancy_grid + pcop_occupancy_shadows)");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  oc->world_to_sensor16 = world_to_sensor16;
  oc->sensor_to_world16 = sensor_to_world16;
  oc->grids = grids;
  oc->grids_on_device = is_device_pointer(grids);
  return PCOP_OK;
}

int pcop_process_batch_occupancy(pcop_handle* h, const float* xyzw, size_t frame_stride_points, const int32_t* n,
                                 int32_t batch, const float* world_to_sensor16, const float* sensor_to_world16,
                                 int8_t* grids, pcop_frame_result* out) {
  if (!h) return fail(nullptr, PCOP_ERR_BAD_PARAM, "null handle");
  if (!world_to_sensor16 || !sensor_to_world16 || !grids || !out || batch < 0 || (!xyzw && batch != 1))
    return fail(h, PCOP_ERR_BAD_PARAM, "pcop_process_batch_occupancy: null argument (xyzw = NULL takes batch = 1)");
  pcop_handle::OccCall oc{};
  TRY(occ_call_of(h, "pcop_process_batch_occupancy", world_to_sensor16, sensor_to_world16, grids, &oc));
  int st;
  if (!xyzw) {  // the accumulated cloud, consumed by this run (od.cpp:701), as pcop_process_accumulated
    const int32_t acc_n = h->acc_count;
    st = process_impl(h, reinterpret_cast<const float*>(h->d_acc), (size_t)(acc_n > 0 ? acc_n : 1), &acc_n, 1, out, &oc);
    h->acc_count = 0;
  } else {
    st = process_impl(h, xyzw, frame_stride_points, n, batch, out, &oc);
  }
  h->occ = nullptr;
  for (pcop_handle* l : h->extra_lanes) l->occ = nullptr;
  return st;
}

int pcop_process_batch_pointcloud2(pcop_handle* h, const pcop_pointcloud2_frame* frames, int32_t batch,
                                   const float* transform16, const float* world_to_sensor16,
                                   const float* sensor_to_world16, int8_t* grids, pcop_frame_result* out) {
  if (!h) return fail(nullptr, PCOP_ERR_BAD_PARAM, "null handle");
  if (!out || batch < 0 || (!frames && batch > 0) || (grids && (!world_to_sensor16 || !sensor_to_world16)))
    return fail(h, PCOP_ERR_BAD_PARAM,
                "pcop_process_batch_pointcloud2: null argument (grids need world_to_sensor16 and sensor_to_world16)");
  Pc2Call pc;
  pc.frames = frames;
  pc.transform16 = transform16;
  std::vector<int32_t> n((size_t)batch + 1, 0);
  for (int f = 0; f < batch; ++f) {
    const pcop_pointcloud2_frame& m = frames[f];
    if (m.n_points < 0 || (!m.data && m.n_points > 0))
      return fail(h, PCOP_ERR_BAD_PARAM, "pcop_process_batch_pointcloud2: frame " + std::to_string(f) + ": bad count or NULL data");
    if (!pc2_layout_ok(m.point_step, m.off_x, m.off_y, m.off_z))
      return fail(h, PCOP_ERR_BAD_PARAM,
                  "pcop_process_batch_pointcloud2: frame " + std::to_string(f) + ": PointCloud2 field offsets do not fit point_step");
    if (m.n_points > h->cap)
      return fail(h, PCOP_ERR_CAPACITY, "pcop_process_batch_pointcloud2: frame " + std::to_string(f) + " has more points than max_points");
    n[f] = m.n_points;
  }
  pcop_handle::OccCall oc{};
  if (grids) TRY(occ_call_of(h, "pcop_process_batch_pointcloud2", world_to_sensor16, sensor_to_world16, grids, &oc));
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  pc.on_device.resize((size_t)batch);
  for (int f = 0; f < batch; ++f) pc.on_device[f] = frames[f].n_points > 0 && is_device_pointer(frames[f].data);
  const int st = process_impl(h, nullptr, (size_t)h->cap, n.data(), batch, out, grids ? &oc : nullptr, &pc);
  h->occ = nullptr;
  for (pcop_handle* l : h->extra_lanes) l->occ = nullptr;
  return st;
}

int pcop_enable_kernel_timing(pcop_handle* h, int enable) {
  if (!h) return PCOP_ERR_BAD_PARAM;
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (enable && !h->kt.ev) {
    h->kt.ev = new cudaEvent_t[2 * KernelTimers::MAX_SLOTS];
    for (int i = 0; i < 2 * KernelTimers::MAX_SLOTS; ++i) PCOP_CUDA_TRY(cudaEventCreate(&h->kt.ev[i]));
  }
  h->kt.enabled = enable != 0;
  h->kt.used = 0;
  h->kt.n_names = 0;
  return PCOP_OK;
}

int pcop_kernel_timing_count(const pcop_handle* h) { return h ? h->kt.n_names : 0; }

int pcop_kernel_timing_get(const pcop_handle* h, int i, const char** name, double* total_us, int64_t* launches) {
  if (!h || i < 0 || i >= h->kt.n_names) return PCOP_ERR_BAD_PARAM;
  if (name) *name = h->kt.names[i];
  if (total_us) *total_us = h->kt.total_us[i];
  if (launches) *launches = h->kt.launches[i];
  return PCOP_OK;
}

float pcop_last_elapsed_us(const pcop_handle* h) { return h ? h->last_elapsed_us : 0.f; }
int pcop_stage_times_us(const pcop_handle* h, float us[PCOP_N_STAGES]) {
  if (!h || !us) return PCOP_ERR_BAD_PARAM;
  for (int s = 0; s < PCOP_N_STAGES; ++s) us[s] = h->stage_us[s];
  return PCOP_OK;
}
int64_t pcop_last_launch_count(const pcop_handle* h) { return h ? h->launches : 0; }
double pcop_last_algorithmic_bytes(const pcop_handle* h) { return h ? h->alg_bytes : 0.0; }
int pcop_download(pcop_handle* h, void* dst, const void* src_device, size_t bytes) {
  if (!h || (bytes && (!dst || !src_device))) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (bytes) PCOP_CUDA_TRY(cudaMemcpyAsync(dst, src_device, bytes, cudaMemcpyDefault, h->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

int64_t pcop_last_sort_pass_keys(const pcop_handle* h) { return h ? (int64_t)h->sort_pass_keys : 0; }
double pcop_last_d2h_bytes(const pcop_handle* h) { return h ? h->d2h_bytes : 0.0; }

// ---- accumulator ingest (od.cpp:691-698) -------------------------------------------------
static int transform_into(pcop_handle* h, const float* xyzw, int32_t n, const float* t16, int is_dense, float4* dst) {
  // staged through d_in (frame 0) when the source is host memory
  const float4* src = reinterpret_cast<const float4*>(xyzw);
  if (!is_device_pointer(xyzw)) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_in, xyzw, (size_t)n * 16, cudaMemcpyHostToDevice, h->stream));
    src = h->d_in;
  }
  Mat34 t;
  const float ident[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
  memcpy(t.m, t16 ? t16 : ident, sizeof(t.m));
  Ctx c = make_ctx(h, 1, n);
  KL(c, "k_transform", k_transform<<<cdiv(n, 256), 256, 0, h->stream>>>(src, n, t, is_dense, dst));
  count_launch(c);
  return PCOP_OK;
}

int pcop_accumulate(pcop_handle* h, const float* xyzw, int32_t n, const float* transform16, int32_t is_dense, int32_t* total) {
  if (!h || (!xyzw && n > 0) || n < 0) return fail(h, PCOP_ERR_BAD_PARAM, "pcop_accumulate: bad argument");
  if ((long long)h->acc_count + n > h->cap) return fail(h, PCOP_ERR_CAPACITY, "accumulated cloud exceeds max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (n > 0) {
    TRY(transform_into(h, xyzw, n, transform16, is_dense, h->d_acc + h->acc_count));
    if (!is_device_pointer(xyzw)) PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));  // the caller may reuse its buffer
  }
  h->acc_count += n;
  if (total) *total = h->acc_count;
  return PCOP_OK;
}

int32_t pcop_accumulated_count(const pcop_handle* h) { return h ? h->acc_count : 0; }

int pcop_accumulate_reset(pcop_handle* h) {
  if (!h) return PCOP_ERR_BAD_PARAM;
  h->acc_count = 0;
  return PCOP_OK;
}

int pcop_process_accumulated(pcop_handle* h, pcop_frame_result* out) {
  if (!h || !out) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  const int32_t n = h->acc_count;
  // od.cpp:701: current_frame_count = 0; the accumulator is consumed by this run
  const int st = process_impl(h, reinterpret_cast<const float*>(h->d_acc), (size_t)(n > 0 ? n : 1), &n, 1, out);
  h->acc_count = 0;
  return st;
}

int pcop_transform(pcop_handle* h, const float* xyzw, int32_t n, const float* transform16, int32_t is_dense, float* out_xyzw) {
  if (!h || !xyzw || !out_xyzw || n < 0) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (n > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return PCOP_OK;
  TRY(transform_into(h, xyzw, n, transform16, is_dense, h->d_crop));
  TRY(download(h, out_xyzw, h->d_crop, (size_t)n * 16));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

static int pc2_ingest(pcop_handle* h, const unsigned char* data, int32_t n, int32_t point_step, int32_t ox, int32_t oy,
                      int32_t oz, const float* t16, int is_dense, float4* dst) {
  if (!pc2_layout_ok(point_step, ox, oy, oz)) return fail(h, PCOP_ERR_BAD_PARAM, "PointCloud2 field offsets do not fit point_step");
  const size_t bytes = (size_t)n * (size_t)point_step;
  const unsigned char* src = data;
  if (!is_device_pointer(data)) {
    TRY(ensure_raw(h, bytes));
    PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_raw, data, bytes, cudaMemcpyHostToDevice, h->stream));
    src = h->d_raw;
  }
  // the batched decode with one frame; the descriptor goes up from pageable memory (staged before the call returns)
  const Pc2Frame d = make_pc2_frame(src, n, point_step, ox, oy, oz, t16, is_dense);
  PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_pc2, &d, sizeof(d), cudaMemcpyHostToDevice, h->stream));
  Ctx c = make_ctx(h, 1, n);
  KL(c, "k_pc2_ingest", k_pc2_ingest<<<dim3(cdiv(n, 256), 1), 256, 0, h->stream>>>(h->d_pc2, dst, (size_t)0));
  count_launch(c);
  if (src != data) PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));  // the caller may reuse its buffer
  return PCOP_OK;
}

int pcop_accumulate_pointcloud2(pcop_handle* h, const unsigned char* data, int32_t n_points, int32_t point_step,
                                int32_t off_x, int32_t off_y, int32_t off_z, const float* transform16, int32_t is_dense,
                                int32_t* total) {
  if (!h || (!data && n_points > 0) || n_points < 0) return fail(h, PCOP_ERR_BAD_PARAM, "pcop_accumulate_pointcloud2: bad argument");
  if ((long long)h->acc_count + n_points > h->cap) return fail(h, PCOP_ERR_CAPACITY, "accumulated cloud exceeds max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (n_points > 0) TRY(pc2_ingest(h, data, n_points, point_step, off_x, off_y, off_z, transform16, is_dense, h->d_acc + h->acc_count));
  h->acc_count += n_points;
  if (total) *total = h->acc_count;
  return PCOP_OK;
}

int pcop_pointcloud2_to_xyz(pcop_handle* h, const unsigned char* data, int32_t n_points, int32_t point_step, int32_t off_x,
                            int32_t off_y, int32_t off_z, float* out_xyzw) {
  if (!h || !data || !out_xyzw || n_points < 0) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (n_points > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (n_points == 0) return PCOP_OK;
  TRY(pc2_ingest(h, data, n_points, point_step, off_x, off_y, off_z, nullptr, 1, h->d_crop));
  TRY(download(h, out_xyzw, h->d_crop, (size_t)n_points * 16));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

int pcop_cloud_to_pointcloud2(pcop_handle* h, const float* xyzw, int32_t n, int32_t point_step, int32_t off_x, int32_t off_y,
                              int32_t off_z, unsigned char* out_data) {
  if (!h || n < 0 || (n > 0 && (!xyzw || !out_data))) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (point_step < 12 || off_x < 0 || off_y < 0 || off_z < 0 || off_x + 4 > point_step || off_y + 4 > point_step ||
      off_z + 4 > point_step)
    return fail(h, PCOP_ERR_BAD_PARAM, "PointCloud2 field offsets do not fit point_step");
  if (n > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return PCOP_OK;
  const float4* src = reinterpret_cast<const float4*>(xyzw);
  if (!is_device_pointer(xyzw)) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_in, xyzw, (size_t)n * 16, cudaMemcpyHostToDevice, h->stream));
    src = h->d_in;
  }
  const size_t bytes = (size_t)n * (size_t)point_step;
  unsigned char* dst = out_data;
  const bool out_on_device = is_device_pointer(out_data);
  if (!out_on_device) {  // staged through the raw-payload buffer of the ingest path
    TRY(ensure_raw(h, bytes));
    dst = h->d_raw;
  }
  Ctx c = make_ctx(h, 1, n);
  KL(c, "k_pc2_egress", k_pc2_egress<<<cdiv(n, 256), 256, 0, h->stream>>>(src, n, point_step, off_x, off_y, off_z, dst));
  count_launch(c);
  PCOP_CUDA_TRY(cudaGetLastError());
  if (!out_on_device) TRY(download(h, out_data, dst, bytes));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

int pcop_occupancy_dims(const pcop_handle* h, int32_t* width, int32_t* height) {
  if (!h || !width || !height || !(h->params.block_size > 0.0f)) return PCOP_ERR_BAD_PARAM;
  const pcop_params& p = h->params;  // od.cpp:958-959 (double: the unqualified fabs is ::fabs(double))
  *width = (int32_t)std::ceil((std::fabs((double)p.y_min) + std::fabs((double)p.y_max)) / (double)p.block_size);
  *height = (int32_t)std::ceil((std::fabs((double)p.x_min) + std::fabs((double)p.x_max)) / (double)p.block_size);
  return PCOP_OK;
}

// the grid of the handle's parameters; BAD_PARAM when they give none
static int occ_grid_of(pcop_handle* h, OccGrid* g) {
  int32_t W = 0, H = 0;
  if (pcop_occupancy_dims(h, &W, &H) != PCOP_OK || W <= 0 || H <= 0 || (long long)W * H > (1ll << 26))
    return fail(h, PCOP_ERR_BAD_PARAM, "occupancy grid: block_size / crop limits give no usable grid");
  const pcop_params& p = h->params;
  const float lim[6] = {p.x_min, p.x_max, p.y_min, p.y_max, p.z_min, p.z_max};
  memcpy(g->lim, lim, sizeof(lim));
  g->block_size = p.block_size;
  g->dev_percent = p.dev_percent;
  g->W = W;
  g->H = H;
  g->cells = (long long)W * H;
  return PCOP_OK;
}

int pcop_occupancy_grid(pcop_handle* h, const float* xyzw, int32_t n, int8_t* grid_data, int64_t* counts, int64_t* row_avg) {
  if (!h || !grid_data || n < 0) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  OccGrid g;
  TRY(occ_grid_of(h, &g));
  const int32_t H = g.H;
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  const float4* src;
  if (!xyzw) {  // the accumulated cloud
    src = h->d_acc;
    n = h->acc_count;
  } else {
    if (n > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
    src = reinterpret_cast<const float4*>(xyzw);
    if (!is_device_pointer(xyzw)) {
      if (n > 0) PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_in, xyzw, (size_t)n * 16, cudaMemcpyHostToDevice, h->stream));
      src = h->d_in;
    }
  }
  const size_t cells = (size_t)g.cells;
  const size_t need = cells * 8 + (size_t)H * 8 + cells;
  if (need > h->occ_cap) {
    PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (h->d_occ) cudaFree(h->d_occ);
    h->d_occ = nullptr;
    h->occ_cap = 0;
    PCOP_CUDA_TRY(cudaMalloc((void**)&h->d_occ, need + 256));
    h->occ_cap = need;
  }
  unsigned long long* d_counts = reinterpret_cast<unsigned long long*>(h->d_occ);
  long long* d_avg = reinterpret_cast<long long*>(h->d_occ + cells * 8);
  signed char* d_grid = reinterpret_cast<signed char*>(h->d_occ + cells * 8 + (size_t)H * 8);
  Ctx c = make_ctx(h, 1, n);
  PCOP_CUDA_TRY(cudaMemsetAsync(d_counts, 0, cells * 8, h->stream));
  run_occ_count(c, src, n, g, d_counts);
  run_occ_finish(c, d_counts, g, d_avg, d_grid);
  TRY(download(h, grid_data, d_grid, cells));
  TRY(download(h, counts, d_counts, cells * 8));
  TRY(download(h, row_avg, d_avg, (size_t)H * 8));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

// Shadow casting + obstacle marking (od.cpp:467-672, 817-833) on a grid produced by pcop_occupancy_grid
int pcop_occupancy_shadows(pcop_handle* h, const float* remaining_xyzw, int32_t n_remaining, const int32_t* cluster_offsets,
                           const int32_t* cluster_indices, int32_t n_clusters, const float* world_to_sensor16,
                           const float* sensor_to_world16, int8_t* grid_data, int32_t* shadow_records, uint32_t* warnings) {
  if (!h || !grid_data || n_remaining < 0 || n_clusters < 0 || (n_remaining > 0 && !remaining_xyzw) ||
      (n_clusters > 0 && (!cluster_offsets || !cluster_indices || !world_to_sensor16 || !sensor_to_world16)))
    return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  int32_t W = 0, H = 0;
  if (pcop_occupancy_dims(h, &W, &H) != PCOP_OK || W <= 0 || H <= 0 || (long long)W * H > (1ll << 26))
    return fail(h, PCOP_ERR_BAD_PARAM, "occupancy grid: block_size / crop limits give no usable grid");
  if (n_remaining > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  const size_t cells = (size_t)W * H;
  // the member list's length is the last CSR offset
  int32_t L = 0;
  if (n_clusters > 0) {
    if (is_device_pointer(cluster_offsets)) {
      PCOP_CUDA_TRY(cudaMemcpyAsync(&L, cluster_offsets + n_clusters, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
      PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
    } else {
      L = cluster_offsets[n_clusters];
    }
    if (L < 0 || L > h->cap) return fail(h, PCOP_ERR_BAD_PARAM, "cluster_offsets: last offset out of range");
  }
  // scratch: [grid cells][pad][offsets C+1][indices L][records 6C][warnings 1][P, C][poses 2 x 12 floats]
  const size_t off_ints = (cells + 15) & ~(size_t)15;
  const size_t need = off_ints + ((size_t)n_clusters + 1 + (size_t)L + 6 * (size_t)n_clusters + 3) * sizeof(int32_t) +
                      2 * sizeof(Mat34);
  if (need > h->shadow_cap) {
    PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (h->d_shadow) cudaFree(h->d_shadow);
    h->d_shadow = nullptr;
    h->shadow_cap = 0;
    PCOP_CUDA_TRY(cudaMalloc((void**)&h->d_shadow, need + 256));
    h->shadow_cap = need;
  }
  int32_t* d_off = reinterpret_cast<int32_t*>(h->d_shadow + off_ints);
  int32_t* d_idx = d_off + n_clusters + 1;
  int32_t* d_rec = d_idx + L;
  uint32_t* d_warn = reinterpret_cast<uint32_t*>(d_rec + 6 * (size_t)n_clusters);
  int32_t* d_sizes = reinterpret_cast<int32_t*>(d_warn + 1);
  Mat34* d_mats = reinterpret_cast<Mat34*>(d_sizes + 2);
  pcop::OccShadowArgs a{};
  a.cloud = reinterpret_cast<const float4*>(remaining_xyzw);
  if (n_remaining > 0 && !is_device_pointer(remaining_xyzw)) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_in, remaining_xyzw, (size_t)n_remaining * 16, cudaMemcpyHostToDevice, h->stream));
    a.cloud = h->d_in;
  }
  a.offsets = cluster_offsets;
  a.indices = cluster_indices;
  if (n_clusters > 0 && !is_device_pointer(cluster_offsets)) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(d_off, cluster_offsets, ((size_t)n_clusters + 1) * 4, cudaMemcpyHostToDevice, h->stream));
    a.offsets = d_off;
  }
  if (n_clusters > 0 && L > 0 && !is_device_pointer(cluster_indices)) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(d_idx, cluster_indices, (size_t)L * 4, cudaMemcpyHostToDevice, h->stream));
    a.indices = d_idx;
  }
  struct {
    int32_t sizes[2];
    Mat34 mats[2];
  } up;
  up.sizes[0] = n_remaining;
  up.sizes[1] = n_clusters;
  for (int r = 0; r < 12; ++r) {
    up.mats[0].m[r] = world_to_sensor16 ? world_to_sensor16[r] : ((r % 5 == 0) ? 1.0f : 0.0f);
    up.mats[1].m[r] = sensor_to_world16 ? sensor_to_world16[r] : ((r % 5 == 0) ? 1.0f : 0.0f);
  }
  static_assert(sizeof(up) == 2 * sizeof(int32_t) + 2 * sizeof(Mat34), "packed upload");
  PCOP_CUDA_TRY(cudaMemcpyAsync(d_sizes, &up, sizeof(up), cudaMemcpyHostToDevice, h->stream));  // (pageable: staged before return)
  a.n_points = d_sizes;
  a.n_clusters = d_sizes + 1;
  a.mats = d_mats;
  const pcop_params& p = h->params;
  a.y_min = p.y_min;
  a.x_max = p.x_max;
  a.block_size = p.block_size;
  a.W = W;
  a.size = (long long)cells;
  a.opacity = p.grid_opacity;
  const bool grid_on_device = is_device_pointer(grid_data);
  a.grid = reinterpret_cast<signed char*>(grid_data);
  if (!grid_on_device) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_shadow, grid_data, cells, cudaMemcpyHostToDevice, h->stream));
    a.grid = reinterpret_cast<signed char*>(h->d_shadow);
  }
  a.records = shadow_records ? d_rec : nullptr;
  a.warnings = d_warn;
  PCOP_CUDA_TRY(cudaMemsetAsync(d_warn, 0, sizeof(uint32_t), h->stream));
  Ctx c = make_ctx(h, 1, n_remaining);
  pcop::run_occ_shadows(c, a, n_clusters, n_remaining);
  PCOP_CUDA_TRY(cudaGetLastError());
  if (!grid_on_device) TRY(download(h, grid_data, a.grid, cells));
  if (shadow_records && n_clusters > 0) {
    if (is_device_pointer(shadow_records))
      PCOP_CUDA_TRY(cudaMemcpyAsync(shadow_records, d_rec, 6 * (size_t)n_clusters * 4, cudaMemcpyDeviceToDevice, h->stream));
    else
      TRY(download(h, shadow_records, d_rec, 6 * (size_t)n_clusters * 4));
  }
  uint32_t wv = 0;
  PCOP_CUDA_TRY(cudaMemcpyAsync(&wv, d_warn, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (warnings) *warnings = wv;
  return PCOP_OK;
}

// ---- stage-isolated entry points -------------------------------------------------------
int pcop_crop(pcop_handle* h, const float* xyzw, int32_t n, float* out_xyzw, int32_t* kept_idx, int32_t* m) {
  if (!h || !xyzw || !m) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  TRY(upload_single(h, xyzw, n, CNT_IN));
  Ctx c = make_ctx(h, 1, n);
  run_crop(c, make_crop_args(h, h->d_in, h->cap, h->cnt(CNT_IN)));
  TRY(fetch_count(h, CNT_CROP, m));
  TRY(download(h, out_xyzw, h->d_crop, (size_t)*m * 16));
  TRY(download(h, kept_idx, h->d_crop_kept, (size_t)*m * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

int pcop_voxel(pcop_handle* h, const float* xyzw, int32_t m, float* out_xyzw, uint32_t* out_keys, int32_t* v,
               uint32_t* warnings) {
  if (!h || !xyzw || !v) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (!(h->params.downsample_size > 0.0f)) return fail(h, PCOP_ERR_BAD_PARAM, "downsample_size must be > 0");
  TRY(upload_single(h, xyzw, m, CNT_CROP));
  Ctx c = make_ctx(h, 1, m);
  run_minmax(c, h->d_in, h->cap, h->cnt(CNT_CROP), h->d_minmax);
  run_voxel(c, make_voxel_args(h, h->d_in, h->cap, h->cnt(CNT_CROP)));
  TRY(fetch_count(h, CNT_VOX, v));
  TRY(fetch_warnings(h, warnings));
  TRY(download(h, out_xyzw, h->d_vox, (size_t)*v * 16));
  TRY(download(h, out_keys, h->d_vox_keys, (size_t)*v * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

int pcop_sor(pcop_handle* h, const float* xyzw, int32_t v, float* out_xyzw, int32_t* kept_idx, int32_t* s,
             uint32_t* warnings) {
  if (!h || !xyzw || !s) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (h->params.statistical_outlier_meanK < 1 || h->params.statistical_outlier_meanK > 63)
    return fail(h, PCOP_ERR_BAD_PARAM, "statistical_outlier_meanK must be in [1, 63]");
  TRY(upload_single(h, xyzw, v, CNT_VOX));
  Ctx c = make_ctx(h, 1, v);
  run_sor(c, make_sor_args(h, h->d_in, h->cap, h->cnt(CNT_VOX)));
  TRY(fetch_count(h, CNT_SOR, s));
  TRY(fetch_warnings(h, warnings));
  TRY(download(h, out_xyzw, h->d_sor, (size_t)*s * 16));
  TRY(download(h, kept_idx, h->d_sor_kept, (size_t)*s * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

int pcop_plane(pcop_handle* h, const float* xyzw, int32_t s, float* remaining_xyzw, int32_t* remaining_src_idx,
               int32_t* p, int32_t* n_passes, int32_t* pass_points, int32_t* pass_inliers, float* pass_coeff,
               float* last_coeff, int32_t* inlier_idx, int32_t* n_inliers, uint32_t* warnings) {
  if (!h || !xyzw || !p) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  TRY(upload_single(h, xyzw, s, CNT_SOR));
  Ctx c = make_ctx(h, 1, s);
  PlaneArgs a = make_plane_args(h, h->d_in, h->cap, h->cnt(CNT_SOR));
  a.large_tier = 1;
  if (s > plane_resident_max()) a.resident = 0;  // (the host knows the size here)
  cudaError_t e = run_plane(c, a);
  if (e != cudaSuccess) return fail_cuda(h, e, "run_plane", __FILE__, __LINE__);
  KL(c, "k_plane_record", k_plane_record<<<1, 32, 0, h->stream>>>(h->d_pf, h->d_prec, h->cnt(CNT_NINL), h->cnt(CNT_CLUS), h->cnt(CNT_CLUS1), 1, 1));
  TRY(fetch_count(h, CNT_REM, p));
  TRY(fetch_warnings(h, warnings));
  PCOP_CUDA_TRY(cudaMemcpyAsync(h->h_prec, h->d_prec, sizeof(PlaneRecord), cudaMemcpyDeviceToHost, h->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  const PlaneRecord& r = h->h_prec[0];
  if (n_passes) *n_passes = r.n_passes;
  if (pass_points) memcpy(pass_points, r.pass_points, sizeof(r.pass_points));
  if (pass_inliers) memcpy(pass_inliers, r.pass_inliers, sizeof(r.pass_inliers));
  if (pass_coeff) memcpy(pass_coeff, r.pass_coeff, sizeof(r.pass_coeff));
  if (last_coeff) memcpy(last_coeff, &r.coeff, 16);
  if (n_inliers) *n_inliers = r.n_inliers_last;
  TRY(download(h, remaining_xyzw, h->d_rem, (size_t)*p * 16));
  TRY(download(h, remaining_src_idx, h->d_rem_src, (size_t)*p * 4));
  TRY(download(h, inlier_idx, h->d_inliers, (size_t)r.n_inliers_last * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

int pcop_cluster(pcop_handle* h, const float* xyzw, int32_t p, int32_t* cluster_offsets, int32_t* cluster_indices,
                 int32_t* c_out, int32_t* l_out) {
  if (!h || !xyzw || !c_out || !l_out) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (!(h->params.euc_cluster_tolerance > 0.0f)) return fail(h, PCOP_ERR_BAD_PARAM, "euc_cluster_tolerance must be > 0");
  TRY(upload_single(h, xyzw, p, CNT_REM));
  Ctx c = make_ctx(h, 1, p);
  run_cluster(c, make_cluster_args(h, h->d_in, h->cap, h->cnt(CNT_REM)), /*with_generic=*/true);
  TRY(fetch_count(h, CNT_CLUS, c_out));
  TRY(fetch_count(h, CNT_CLPTS, l_out));
  TRY(download(h, cluster_offsets, h->d_offsets, (size_t)(*c_out + 1) * 4));
  TRY(download(h, cluster_indices, h->d_indices, (size_t)*l_out * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

int pcop_centroid_radius(pcop_handle* h, const float* xyzw, int32_t p, const int32_t* cluster_offsets,
                         const int32_t* cluster_indices, int32_t c_in, float* obstacles) {
  if (!h || !xyzw || !cluster_offsets || !cluster_indices || !obstacles || c_in < 0)
    return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (c_in > h->cap) return fail(h, PCOP_ERR_CAPACITY, "too many clusters");
  TRY(upload_single(h, xyzw, p, CNT_REM));
  const int l = cluster_offsets[c_in];
  if (l < 0 || l > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cluster index list longer than max_points");
  h->h_n_in[1] = c_in;
  PCOP_CUDA_TRY(cudaMemcpyAsync(h->cnt(CNT_CLUS), h->h_n_in + 1, sizeof(int), cudaMemcpyHostToDevice, h->stream));
  PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_offsets, cluster_offsets, (size_t)(c_in + 1) * 4, cudaMemcpyDefault, h->stream));
  if (l > 0) PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_indices, cluster_indices, (size_t)l * 4, cudaMemcpyDefault, h->stream));
  Ctx c = make_ctx(h, 1, p);
  run_centroid_radius(c, make_cluster_args(h, h->d_in, h->cap, h->cnt(CNT_REM)));
  TRY(download(h, obstacles, h->d_obst, (size_t)c_in * 16));
  PCOP_CUDA_TRY(cudaStreamSynchronize(h->stream));
  return PCOP_OK;
}

}  // extern "C"
