// The handle and its lanes (pcop_api.cu, batch.cu).  The handle holds the parameters, knobs, per-call counters and error
// text once; a lane holds what one wave in flight needs and reaches the parameters through its handle.
#pragma once
#include <cmath>
#include <memory>
#include <string>
#include <vector>

#include <cuda.h>  // (types of cuPointerGetAttributes only; see PayloadClassifier)

#include "internal.cuh"

namespace pcop {

enum {  // rows of the per-frame count table (device: d_counts[row*maxB + f])
  CNT_IN = 0,
  CNT_CROP,
  CNT_VOX,
  CNT_SOR,
  CNT_REM,
  CNT_CLUS,
  CNT_CLPTS,
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
  size_t dst;                 // element offset of the message's first decoded point in the output
  int n, point_step, off_x, off_y, off_z;
  int is_dense, apply_transform, aligned;
  int tile0;                  // the message's first record tile (PC2_TILE records each) in the launch
  Mat34 t;
};
constexpr int PC2_THREADS = 256, PC2_ITEMS = 4, PC2_TILE = PC2_THREADS * PC2_ITEMS;  // k_pc2_ingest

// the grid product of a batched call (pcop_process_batch_occupancy, pcop_process_batch_pointcloud2 with grids)
struct OccCall {
  OccGrid g;
  const float* world_to_sensor16;
  const float* sensor_to_world16;
  int8_t* grids;
  bool grids_on_device;
};

// the messages of a pcop_process_batch_pointcloud2_windows call
struct Pc2Call {
  const pcop_pointcloud2_frame* msgs;
  const int32_t* window_first;    // [batch + 1]: frame f = messages window_first[f] .. window_first[f + 1] - 1
  const float* transform16;       // [messages][16] or nullptr
  std::vector<char> on_device;    // per message: the payload is a device pointer (used in place)
};

struct WaveInput {
  const float* xyzw;
  size_t frame_stride_points;
  const int32_t* n;
  bool on_device;
  const Pc2Call* pc2;  // non-null: the frames are PointCloud2 messages, decoded into d_in by the wave (xyzw unused)
  const OccCall* occ;  // non-null: the grid product of every frame as well
};

// What one wave launches where the frame sizes decide the path.  The host does not know those sizes when it enqueues
// the wave, so the first route is a guess from the lane's earlier waves (next_route, batch.cu); settle_wave checks it
// against the wave's counts and repeats the part of the wave a wrong guess left undone.
struct WaveRoute {
  enum Vox { VOX_GENERIC, VOX_LSD, VOX_PARTITION } vox = VOX_GENERIC;  // crop + VoxelGrid: generic, fused LSD / partition
  int vox_groups = 0;  // VOX_PARTITION: reduce groups per frame
  bool plane_large = false;  // the large plane tier runs beside the small one
  bool cluster_generic = false;  // the generic clustering kernels run beside the fused small-cloud kernel
};

constexpr int PCOP_MIN_LANE_WAVE = 8;  // a call is split over the lanes only when every lane gets at least this many frames
struct Lane;

}  // namespace pcop

struct pcop_handle {
  pcop_params params;
  pcop::VoxFusedPlan vplan{};  // fused crop + voxel paths (ok = 0: generic kernels; part_ok = 0: no partition path)
  int device = 0;
  int cap = 0;
  int maxB = 0;                // frames of one lane's wave buffers
  // create-time knobs
  int wave_frames = 0;         // frames per wave a batched call aims at (<= maxB; PCOP_WAVE_FRAMES at create)
  bool trace = false;          // PCOP_TRACE at create: per-wave device timeline of every call on stderr
  int ece_small_max = 0;       // ECE_SMALL_MAX or PCOP_ECE_SMALL_MAX (read at create)
  std::vector<std::unique_ptr<pcop::Lane>> lanes;  // batched calls deal their waves round-robin to the lanes
  std::string err;
  std::vector<void*> dev_allocs;
  std::vector<void*> host_allocs;
  int* d_rng = nullptr;
  float4* d_acc = nullptr;  // accumulated (world-frame) cloud, od.cpp:697
  int acc_count = 0;
  unsigned char* d_occ = nullptr;  // occupancy grid scratch: int64 counts, int64 row averages, int8 cells
  size_t occ_cap = 0;
  unsigned char* d_shadow = nullptr;  // pcop_occupancy_shadows scratch: grid cells, CSR copy, records, warning word
  size_t shadow_cap = 0;

  // per-call accounting (launch counts also accumulate over the single-frame calls until the next pcop_process* call)
  cudaEvent_t ev_call[2] = {nullptr, nullptr};
  float stage_us[PCOP_N_STAGES] = {};
  float last_elapsed_us = 0.f;
  int64_t launches = 0;
  double alg_bytes = 0.0;
  double d2h_bytes = 0.0;
  unsigned long long sort_pass_keys = 0;
  pcop::KernelTimers kt;
};

namespace pcop {

struct Lane {
  pcop_handle* h;  // parameters, knobs, per-call counters and the error text
  cudaStream_t stream = nullptr;
  cudaStream_t cstream = nullptr;   // result copies (device -> pinned host) run here, beside the next wave's kernels
  cudaEvent_t ev_copied = nullptr;  // the last payload copy out of d_pack
  cudaEvent_t ev_meta = nullptr;    // the wave's counts / pack sizes are in pinned memory
  cudaEvent_t ev_lane_done = nullptr;
  cudaEvent_t ev_stage[PCOP_N_STAGES][2] = {};
  bool stage_used[PCOP_N_STAGES] = {};

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
  int* d_pack_off = nullptr;  // [PK_N][maxB]
  PackMeta* d_meta = nullptr;
  unsigned char* d_pack = nullptr;  // packed results of the wave in flight (PCOP_OUT_DEVICE: of all waves of the call)
  size_t pack_cap = 0;
  unsigned long long* d_pack_cursor = nullptr;  // PCOP_OUT_DEVICE: bytes of d_pack used by the call so far
  // pcop_process_batch_occupancy (allocated by the first such call; counts / grids grow with W x H and with the
  // largest wave the lane has run)
  int* d_occ_counts = nullptr;       // [wave frames][cells] int32
  signed char* d_occ_grids = nullptr;  // [wave frames][cells]
  size_t occ_scratch_cells = 0;      // frames x cells the two arrays hold
  Mat34* d_occ_mats = nullptr;       // [maxB][2] world_to_sensor, sensor_to_world
  Mat34* h_occ_mats = nullptr;       // pinned staging of the same
  cudaEvent_t ev_grids_copied = nullptr;  // the last copy out of d_occ_grids
  unsigned char* d_raw = nullptr;  // staging of raw PointCloud2 payloads from host memory: one message, or the host
  size_t raw_cap = 0;              // messages of one wave at 256-byte aligned offsets (grown on demand)
  Pc2Frame* d_pc2 = nullptr;       // decode descriptors of k_pc2_ingest: one per message of a wave
  Pc2Frame* h_pc2 = nullptr;       // pinned staging of the same (the batched PointCloud2 wave)
  size_t pc2_cap = 0;              // descriptors the two hold (grown on demand, never shrunk)
  int pc2_msgs = 0, pc2_tiles = 0; // messages and record tiles of the wave in flight (a repeat decodes them again)

  // pinned host
  int* h_counts = nullptr;  // [CNT_ROWS][maxB]
  uint32_t* h_warnings = nullptr;
  PlaneRecord* h_prec = nullptr;
  PackMeta* h_meta = nullptr;
  int* h_n_in = nullptr;  // staging for the per-frame input sizes
  unsigned long long* h_stats = nullptr;
  // pinned result buffers: two per lane, used by alternate calls, so the pointers a call returns stay valid while the
  // NEXT call runs (a consumer may still be reading them, e.g. the multi-GPU result gather)
  unsigned char* h_pack_buf[2] = {nullptr, nullptr};
  size_t h_pack_buf_cap[2] = {0, 0};
  int h_pack_sel = 0;
  unsigned char* h_pack = nullptr;  // = h_pack_buf[h_pack_sel]
  size_t h_pack_cap = 0;
  size_t h_pack_used = 0;  // of the running call

  int wave_seq = 0;                 // waves of the running call seen by this lane
  int call_lane_waves = 1;          // waves of the running call dealt to this lane
  bool pending = false;             // a wave is enqueued and not yet collected
  int pend_w0 = 0, pend_B = 0;
  int pend_max_n = 1;
  WaveRoute route;                  // of the wave in flight
  std::vector<size_t> fixups;  // result-pointer slots of the running call (byte offsets into the caller's array)
  struct TraceRec {
    int w0, B;
    size_t bytes;
    cudaEvent_t meta, c0, c1;  // counts on the host / payload copy start / end
  };
  std::vector<TraceRec> trace_recs;
  size_t trace_used = 0;

  // history: what the lane's last waves needed decides the next wave's route (next_route, batch.cu)
  bool expect_big_remaining = false;  // the last collected wave had a remaining cloud above ece_small_max
  bool expect_large_plane = false;    // ... a plane-stage input above the small tier of the plane kernel
  int vox_lsd_waves = 0;              // waves left that take the LSD voxel path (the partition path declined a bucket)
  const float4* plane_in = nullptr;   // plane-stage input of the wave in flight (for a repeat of the stage)
  size_t plane_stride = 0;
  const int* plane_n = nullptr;
  uint32_t* d_vf_flags = nullptr;  // [maxB]
  unsigned long long* d_vf_pair[2] = {nullptr, nullptr};
  uint32_t* h_vf_flags = nullptr;
  // partition voxel path (allocated and grown by apply_params while the plan allows the path)
  uint32_t* d_vp_hist = nullptr;
  uint32_t* d_vp_bstart = nullptr;
  uint32_t* d_vp_nstart = nullptr;
  unsigned short* d_vp_ne = nullptr;
  uint2* d_vp_grec = nullptr;
  unsigned* d_vp_desc = nullptr;
  int vp_gcap = 0;                 // groups per frame d_vp_grec / d_vp_desc hold
  int vp_gstride = 0;              // worst-case groups per frame + 1
  int vp_group_hint = 0;           // groups per frame the next wave's reduce grid covers (adapts to the frames seen)

  ~Lane();
  int* cnt(int row) { return d_counts + (size_t)row * h->maxB; }
};

// records the error text in the handle (and the thread's global error slot); returns code
int fail(pcop_handle* h, int code, const std::string& msg);

#define TRY(x)                      \
  do {                              \
    int _s = (x);                   \
    if (_s != PCOP_OK) return _s;   \
  } while (0)

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

inline uint32_t effective_outputs(const pcop_params& p) {
  uint32_t m = p.outputs & (uint32_t)(PCOP_OUT_ALL | PCOP_OUT_DEVICE);
  if (p.publish_point_clouds) m |= PCOP_OUT_ALL;  // od.cpp:945: intermediates wanted
  if (!p.enable_crop) m &= ~(uint32_t)PCOP_OUT_CROP;
  if (!p.enable_voxel) m &= ~(uint32_t)PCOP_OUT_VOXEL;
  if (!p.enable_sor) m &= ~(uint32_t)PCOP_OUT_SOR;
  if (!p.enable_plane) m &= ~(uint32_t)PCOP_OUT_PLANE;
  if (!p.enable_cluster) m &= ~(uint32_t)(PCOP_OUT_CLUSTERS | PCOP_OUT_OBSTACLES);
  return m;
}

inline size_t pack_capacity_bytes(uint32_t mask, int B, int cap) {
  mask &= (uint32_t)PCOP_OUT_ALL;
  size_t bytes = 0;
  for (int k = 0; k < PK_N; ++k)
    if (mask & kPkMask[k]) bytes += ((size_t)B * (cap + 1)) * kPkElem[k] + 256;
  return (bytes + 256 + 255) & ~(size_t)255;
}

inline int ensure_pack_capacity(Lane* l, uint32_t mask) {
  pcop_handle* h = l->h;
  const size_t need = pack_capacity_bytes(mask, h->maxB, h->cap);
  if (need <= l->pack_cap) return PCOP_OK;
  if (l->cstream) cudaStreamSynchronize(l->cstream);
  if (l->d_pack) cudaFree(l->d_pack);  // not tracked in dev_allocs
  l->d_pack = nullptr;
  l->pack_cap = 0;
  cudaError_t e = cudaMalloc((void**)&l->d_pack, need);
  if (e != cudaSuccess) return fail_cuda(h, e, "cudaMalloc(pack)", __FILE__, __LINE__);
  l->pack_cap = need;
  return PCOP_OK;
}

// the raw PointCloud2 staging of lane l holds at least `bytes` (grown by a quarter more, never shrunk)
inline int ensure_raw(Lane* l, size_t bytes) {
  pcop_handle* h = l->h;
  if (bytes <= l->raw_cap) return PCOP_OK;
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  if (l->d_raw) cudaFree(l->d_raw);  // (not tracked in dev_allocs)
  l->d_raw = nullptr;
  l->raw_cap = 0;
  PCOP_CUDA_TRY(cudaMalloc((void**)&l->d_raw, bytes + bytes / 4 + 256));
  l->raw_cap = bytes + bytes / 4 + 256;
  return PCOP_OK;
}

// the PointCloud2 decode descriptors of lane l hold at least `msgs` messages (grown, never shrunk)
inline int ensure_pc2(Lane* l, size_t msgs) {
  pcop_handle* h = l->h;
  if (msgs <= l->pc2_cap) return PCOP_OK;
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  cudaFree(l->d_pc2);  // (not tracked in dev_allocs / host_allocs)
  if (l->h_pc2) cudaFreeHost(l->h_pc2);
  l->d_pc2 = nullptr;
  l->h_pc2 = nullptr;
  l->pc2_cap = 0;
  PCOP_CUDA_TRY(cudaMalloc((void**)&l->d_pc2, sizeof(Pc2Frame) * msgs));
  PCOP_CUDA_TRY(cudaHostAlloc((void**)&l->h_pc2, sizeof(Pc2Frame) * msgs, cudaHostAllocDefault));
  l->pc2_cap = msgs;
  return PCOP_OK;
}

inline bool is_device_pointer(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// is_device_pointer for the many payloads of one call, one driver query per allocation: the query also returns the
// allocation's address range, and a later pointer inside the last range takes that range's answer.  Memory the driver
// does not know (pageable host memory) has no range and is queried per pointer.  (cuPointerGetAttributes comes through
// cudaGetDriverEntryPoint: the library links the runtime only.)  Valid within one call: allocations may change between calls.
struct PayloadClassifier {
  uintptr_t lo = 0, hi = 0;
  bool dev = false;

  using GetAttributes = CUresult (*)(unsigned, CUpointer_attribute*, void**, CUdeviceptr);
  static GetAttributes entry() {
    static const GetAttributes fn = [] {
      void* f = nullptr;
      cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
      if (cudaGetDriverEntryPoint("cuPointerGetAttributes", &f, cudaEnableDefault, &q) != cudaSuccess ||
          q != cudaDriverEntryPointSuccess) {
        cudaGetLastError();
        f = nullptr;
      }
      return reinterpret_cast<GetAttributes>(f);
    }();
    return fn;
  }

  bool operator()(const void* p) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    if (a >= lo && a < hi) return dev;
    const GetAttributes fn = entry();
    unsigned type = 0, managed = 0;
    CUdeviceptr start = 0;
    size_t size = 0;
    CUpointer_attribute at[4] = {CU_POINTER_ATTRIBUTE_MEMORY_TYPE, CU_POINTER_ATTRIBUTE_IS_MANAGED,
                                 CU_POINTER_ATTRIBUTE_RANGE_START_ADDR, CU_POINTER_ATTRIBUTE_RANGE_SIZE};
    void* data[4] = {&type, &managed, &start, &size};
    if (!fn || fn(4, at, data, (CUdeviceptr)a) != CUDA_SUCCESS) return is_device_pointer(p);
    const bool d = type == CU_MEMORYTYPE_DEVICE || type == CU_MEMORYTYPE_UNIFIED || managed != 0;
    if (size > 0 && a >= (uintptr_t)start && a - (uintptr_t)start < size) {
      lo = (uintptr_t)start;
      hi = (uintptr_t)start + size;
      dev = d;
    }
    return d;
  }
};

inline bool pc2_layout_ok(int point_step, int ox, int oy, int oz) {
  return point_step >= 4 && ox >= 0 && oy >= 0 && oz >= 0 && ox <= point_step - 4 && oy <= point_step - 4 &&
         oz <= point_step - 4;
}

inline Ctx make_ctx(Lane* l, int B, int grid_cap = -1) {
  const int cap = l->h->cap;
  return Ctx{l->stream, B, cap, &l->h->launches, &l->h->kt, (grid_cap > 0 && grid_cap < cap) ? grid_cap : cap};
}

inline PlaneConst make_plane_const(const pcop_params& p) {
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

inline PlaneArgs make_plane_args(Lane* l, const float4* in, size_t stride, const int* n_in) {
  pcop_handle* h = l->h;
  PlaneArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.buf[0] = l->d_pbuf[0];
  a.buf[1] = l->d_pbuf[1];
  a.src[0] = l->d_psrc[0];
  a.src[1] = l->d_psrc[1];
  a.inlier_idx = l->d_inliers;
  a.pf = l->d_pf;
  a.partial = l->d_partial;
  a.rng = h->d_rng;
  a.pc = make_plane_const(h->params);
  a.warnings = l->d_warnings;
  a.out = l->d_rem;
  a.out_src = l->d_rem_src;
  a.n_out = l->cnt(CNT_REM);
  return a;
}

inline ClusterArgs make_cluster_args(Lane* l, const float4* in, size_t stride, const int* n_in) {
  pcop_handle* h = l->h;
  ClusterArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.tol = h->params.euc_cluster_tolerance;
  a.min_size = h->params.euc_min_cluster_size;
  a.max_size = h->params.euc_max_cluster_size;
  a.small_max = h->ece_small_max;
  a.minmax = l->d_minmax;
  a.ef = l->d_ef;
  a.sort = l->sort;
  a.sorted_pts = l->d_sorted;
  a.parent = l->d_parent;
  a.csize = l->d_csize;
  a.roots = l->d_roots;
  a.rank_of = l->d_rank;
  a.cell_start = l->d_cell_start;
  a.cell_key = l->d_cell_key;
  a.n_cells = l->cnt(CNT_CELLS);
  a.n_route = l->cnt(CNT_ROUTE);
  a.desc = l->d_desc;
  a.offsets = l->d_offsets;
  a.indices = l->d_indices;
  a.n_clusters = l->cnt(CNT_CLUS);
  a.n_cluster_pts = l->cnt(CNT_CLPTS);
  a.obstacles = l->d_obst;
  a.partial = l->d_partial;
  a.partial_stride = cdiv(h->cap, TS_CHUNK) * 10;
  return a;
}

inline CropArgs make_crop_args(Lane* l, const float4* in, size_t stride, const int* n_in) {
  CropArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.out = l->d_crop;
  a.kept_idx = l->d_crop_kept;
  a.n_out = l->cnt(CNT_CROP);
  a.minmax = l->d_minmax;
  a.desc = l->d_desc;
  const pcop_params& p = l->h->params;
  a.lim[0] = p.x_min;
  a.lim[1] = p.x_max;
  a.lim[2] = p.y_min;
  a.lim[3] = p.y_max;
  a.lim[4] = p.z_min;
  a.lim[5] = p.z_max;
  return a;
}

inline VoxelArgs make_voxel_args(Lane* l, const float4* in, size_t stride, const int* n_in) {
  VoxelArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.minmax = l->d_minmax;
  a.leaf = l->h->params.downsample_size;
  a.vf = l->d_vf;
  a.sort = l->sort;
  a.desc = l->d_desc;
  a.run_start = l->d_run_start;
  a.out = l->d_vox;
  a.out_keys = l->d_vox_keys;
  a.n_out = l->cnt(CNT_VOX);
  a.warnings = l->d_warnings;
  return a;
}

inline SorArgs make_sor_args(Lane* l, const float4* in, size_t stride, const int* n_in) {
  const pcop_params& p = l->h->params;
  SorArgs a{};
  a.in = in;
  a.in_stride = stride;
  a.n_in = n_in;
  a.meanK = p.statistical_outlier_meanK;
  a.mul = (double)p.statistical_outlier_stdDevThres;
  // search-grid cell: a speed knob only (the k-NN result is exact for any cell size)
  a.cell = (p.enable_voxel && p.downsample_size > 0.0f) ? 3.0f * p.downsample_size : 0.05f;
  a.minmax = l->d_minmax;
  a.gf = l->d_ef;
  a.sort = l->sort;
  a.sorted_pts = l->d_sorted;
  a.dist = l->d_sor_dist;
  a.partial = l->d_partial;
  a.thr = l->d_thr;
  a.desc = l->d_desc;
  a.out = l->d_sor;
  a.kept_idx = l->d_sor_kept;
  a.n_out = l->cnt(CNT_SOR);
  a.warnings = l->d_warnings;
  return a;
}

__device__ inline void plane_record_one(const PlaneFrame* __restrict__ pf, PlaneRecord* __restrict__ rec, int* __restrict__ n_inl,
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

// batch.cu: the batched calls (occ, pc2: see WaveInput), and the decode of one PointCloud2 message into dst (lane 0)
int process_impl(pcop_handle* h, const float* xyzw, size_t frame_stride_points, const int32_t* n, int32_t batch,
                 pcop_frame_result* out, const OccCall* occ = nullptr, const Pc2Call* pc2 = nullptr);
int pc2_ingest(pcop_handle* h, const unsigned char* data, int32_t n, int32_t point_step, int32_t ox, int32_t oy,
               int32_t oz, const float* t16, int is_dense, float4* dst);
__global__ void k_zero_u32(uint32_t* p, int n);  // batch.cu; upload_single zeroes one frame's warning word with it

}  // namespace pcop
