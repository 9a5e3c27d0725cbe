// The handle and its lanes (pcop_api.cu, batch.cu).  The handle holds the parameters, knobs, per-call counters and error
// text once; a lane holds what one wave in flight needs and reaches the parameters through its handle.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <memory>
#include <string>
#include <utility>
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
  CNT_HULL,   // H: hull vertices of the frame's clusters (PCOP_OUT_FOOTPRINTS; the last row: without the bit the wave's
              // metadata copy stops before it)
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
  PK_BOXES,
  PK_HULL_OFFSETS,
  PK_HULL_INDICES,
  PK_N
};
struct PackArray {  // one packed output array: row PK_* of kPack
  uint32_t bit;     // the output bit that requests it
  int count_row;    // elements of each frame's part
  int elem_bytes;
  bool csr;         // the lane buffer holds cap + 1 elements per frame (CSR offsets), not cap
  bool fp;          // the result pointer is a field of pcop_frame_footprints, not of pcop_frame_result
  size_t slot;      // offsetof that field
};
constexpr PackArray kPack[] = {
    {PCOP_OUT_CROP, CNT_CROP, 4, false, false, offsetof(pcop_frame_result, crop_kept_idx)},
    {PCOP_OUT_VOXEL, CNT_VOX, 4, false, false, offsetof(pcop_frame_result, voxel_keys)},
    {PCOP_OUT_VOXEL, CNT_VOX, 16, false, false, offsetof(pcop_frame_result, voxel_centroids)},
    {PCOP_OUT_SOR, CNT_SOR, 4, false, false, offsetof(pcop_frame_result, sor_kept_idx)},
    {PCOP_OUT_PLANE, CNT_NINL, 4, false, false, offsetof(pcop_frame_result, plane_inlier_idx)},
    {PCOP_OUT_REMAINING, CNT_REM, 16, false, false, offsetof(pcop_frame_result, remaining_cloud)},
    {PCOP_OUT_REMAINING, CNT_REM, 4, false, false, offsetof(pcop_frame_result, remaining_src_idx)},
    {PCOP_OUT_CLUSTERS, CNT_CLUS1, 4, true, false, offsetof(pcop_frame_result, cluster_offsets)},
    {PCOP_OUT_CLUSTERS, CNT_CLPTS, 4, false, false, offsetof(pcop_frame_result, cluster_indices)},
    {PCOP_OUT_OBSTACLES, CNT_CLUS, 16, false, false, offsetof(pcop_frame_result, obstacles)},
    {PCOP_OUT_FOOTPRINTS, CNT_CLUS, 32, false, true, offsetof(pcop_frame_footprints, boxes)},
    {PCOP_OUT_FOOTPRINTS, CNT_CLUS1, 4, true, true, offsetof(pcop_frame_footprints, hull_offsets)},
    {PCOP_OUT_FOOTPRINTS, CNT_HULL, 4, false, true, offsetof(pcop_frame_footprints, hull_indices)},
};
static_assert(sizeof(kPack) / sizeof(kPack[0]) == PK_N, "one kPack row per PK_* entry");
// (footprint rows last: a wave without PCOP_OUT_FOOTPRINTS packs and copies only the rows and counts before them)
constexpr bool pack_row_ok(const PackArray& a, bool fp) {
  return a.elem_bytes % 4 == 0 && a.fp == fp && (a.bit == PCOP_OUT_FOOTPRINTS) == fp && (a.count_row != CNT_HULL || fp);
}
constexpr bool pack_rows_ok(int k = 0) { return k == PK_N || (pack_row_ok(kPack[k], k >= PK_BOXES) && pack_rows_ok(k + 1)); }
static_assert(pack_rows_ok(), "kPack: elements of whole 32-bit words (k_pack), footprint rows last");

struct PlaneRecord {
  int n_passes;
  int n_inliers_last;
  float4 coeff;
  int pass_points[PCOP_MAX_PLANE_PASSES_RECORDED];
  int pass_inliers[PCOP_MAX_PLANE_PASSES_RECORDED];
  float4 pass_coeff[PCOP_MAX_PLANE_PASSES_RECORDED];
};

// device -> host in one copy.  The footprint arrays' entries come last, so that a wave without PCOP_OUT_FOOTPRINTS
// copies only the part before them (meta_bytes), exactly the record of the arrays of PCOP_OUT_ALL.
struct PackMeta {
  unsigned long long base[PK_BOXES];  // byte offset of each array inside the pack buffer
  unsigned long long total_bytes;
  int total[PK_BOXES];  // elements
  int overflow;         // the wave's arrays do not fit the pack buffer (nothing was packed)
  unsigned long long fp_base[PK_N - PK_BOXES];  // the same for the footprint arrays
  int fp_total[PK_N - PK_BOXES];

  __host__ __device__ unsigned long long& base_of(int k) { return k < PK_BOXES ? base[k] : fp_base[k - PK_BOXES]; }
  __host__ __device__ unsigned long long base_of(int k) const { return k < PK_BOXES ? base[k] : fp_base[k - PK_BOXES]; }
  __host__ __device__ int& total_of(int k) { return k < PK_BOXES ? total[k] : fp_total[k - PK_BOXES]; }
};
static_assert(offsetof(PackMeta, fp_base) == 136, "the record of the PCOP_OUT_ALL arrays keeps its 136 bytes");
inline size_t meta_bytes(uint32_t mask) {
  return (mask & PCOP_OUT_FOOTPRINTS) ? sizeof(PackMeta) : offsetof(PackMeta, fp_base);
}

// decode descriptor of one message (device memory): a PointCloud2 message, read by k_pc2_ingest, or a depth image,
// read by k_depth_ingest (n = width * height pixels; point_step and the field offsets unused)
struct Pc2Frame {
  const unsigned char* data;  // payload on the device
  size_t dst;                 // element offset of the message's first decoded point in the output
  int n, point_step, off_x, off_y, off_z;
  int is_dense, apply_transform, aligned;  // depth image: aligned = 16-byte loads along its rows
  int tile0;                  // the message's first record tile (PC2_TILE records each) in the launch
  Mat34 t;
  // depth image only: Image.width, Image.step, PCOP_DEPTH_*, and the back-projection constants of depth_image_proc
  int width, step, encoding;
  float center_x, center_y, kx, ky;
};
constexpr int PC2_THREADS = 256, PC2_ITEMS = 4, PC2_TILE = PC2_THREADS * PC2_ITEMS;  // k_pc2_ingest, k_depth_ingest

// the grid product of a batched call (pcop_process_batch_occupancy, pcop_process_batch_pointcloud2 with grids)
struct OccCall {
  OccGrid g;
  const float* world_to_sensor16;
  const float* sensor_to_world16;
  int8_t* grids;
  bool grids_on_device;
};

inline int depth_pixel_bytes(int encoding) { return encoding == PCOP_DEPTH_16UC1 ? 2 : 4; }

// the messages of a pcop_process_batch_pointcloud2_windows call, or the images of a pcop_process_batch_depth_windows call
struct Pc2Call {
  const pcop_pointcloud2_frame* msgs;
  const pcop_depth_image* images = nullptr;  // non-null: the messages are depth images (msgs unused)
  const int32_t* window_first;    // [batch + 1]: frame f = messages window_first[f] .. window_first[f + 1] - 1
  const float* transform16;       // [messages][16] or nullptr
  std::vector<char> on_device;    // per message: the payload is a device pointer (used in place)

  int points(int k) const { return images ? images[k].width * images[k].height : msgs[k].n_points; }
  const unsigned char* data(int k) const { return images ? images[k].data : msgs[k].data; }
  size_t payload_bytes(int k) const {  // (an image of 0 pixels uploads nothing, whatever its step)
    if (!images) return (size_t)msgs[k].n_points * (size_t)msgs[k].point_step;
    return points(k) > 0 ? (size_t)images[k].step * (size_t)images[k].height : 0;
  }
  double decode_bytes(int k) const {  // algorithmic bytes of the decode: the payload's records in, PointXYZ out
    const int in = images ? depth_pixel_bytes(images[k].encoding) : msgs[k].point_step;
    return (double)(in + 16) * points(k);
  }
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

// Owns n elements of T in device memory, or (Pinned) in pinned host memory mapped into the device's address space,
// and frees them when it is destroyed.  It reads as a T*: the kernel argument structs and the other views hold plain
// pointers into buffers that a lane or the handle owns.
template <class T, bool Pinned = false>
class Buffer {
 public:
  Buffer() = default;
  Buffer(const Buffer&) = delete;
  Buffer& operator=(const Buffer&) = delete;
  Buffer(Buffer&& o) noexcept : p_(o.p_), n_(o.n_) {
    o.p_ = nullptr;
    o.n_ = 0;
  }
  Buffer& operator=(Buffer&& o) noexcept {
    if (this != &o) {
      reset();
      std::swap(p_, o.p_);
      std::swap(n_, o.n_);
    }
    return *this;
  }
  ~Buffer() { reset(); }

  operator T*() const { return p_; }
  T* get() const { return p_; }  // (for casts, which do not convert)
  size_t size() const { return n_; }  // elements

  void reset() {
    if (p_) {
      if constexpr (Pinned) cudaFreeHost(p_);
      else cudaFree(p_);
    }
    p_ = nullptr;
    n_ = 0;
  }
  // frees what the buffer holds, then allocates n elements (at least one); on failure the buffer is left empty
  cudaError_t allocate(size_t n) {
    reset();
    void* q = nullptr;
    const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
    cudaError_t e;
    if constexpr (Pinned) e = cudaHostAlloc(&q, bytes, cudaHostAllocMapped);
    else e = cudaMalloc(&q, bytes);
    if (e != cudaSuccess) return e;
    p_ = static_cast<T*>(q);
    n_ = n;
    return cudaSuccess;
  }
  // allocate(n), the error recorded in h
  int alloc(pcop_handle* h, size_t n) {
    const cudaError_t e = allocate(n);
    return e == cudaSuccess ? PCOP_OK : fail_cuda(h, e, Pinned ? "cudaHostAlloc" : "cudaMalloc", __FILE__, __LINE__);
  }

 private:
  T* p_ = nullptr;
  size_t n_ = 0;
};
template <class T>
using HostBuffer = Buffer<T, true>;

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
  pcop::Buffer<int> d_rng;
  pcop::Buffer<float4> d_acc;  // accumulated (world-frame) cloud, od.cpp:697
  int acc_count = 0;

  // per-call accounting (launch counts also accumulate over the single-frame calls until the next pcop_process* call)
  cudaEvent_t ev_call[2] = {nullptr, nullptr};
  float stage_us[PCOP_N_STAGES] = {};
  float last_elapsed_us = 0.f;
  int64_t launches = 0;
  double alg_bytes = 0.0;
  double d2h_bytes = 0.0;
  unsigned long long sort_pass_keys = 0;
  pcop::KernelTimers kt;
  // footprints of every frame of the last pcop_process* call (PCOP_OUT_FOOTPRINTS); fp_ok = 0 after a failed call
  std::vector<pcop_frame_footprints> fp;
  bool fp_ok = false;
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

  // device: [maxB * cap] wave arrays and per-frame records, allocated by pcop_create
  Buffer<float4> d_in, d_crop, d_vox, d_sor, d_rem, d_sorted, d_obst;
  Buffer<int> d_crop_kept, d_run_start, d_sor_kept, d_psrc[2], d_rem_src, d_inliers, d_parent, d_csize, d_roots, d_rank,
      d_indices, d_offsets, d_cell_start;
  Buffer<uint32_t> d_cell_key, d_vox_keys;
  Buffer<float> d_sor_dist;
  Buffer<uint32_t> d_sort_key[2], d_sort_val[2], d_sort_hist, d_sort_desc, d_sort_maxkey;
  Buffer<int> d_sort_npass;
  Buffer<unsigned long long> d_sort_stats;
  SortBufs sort{};  // views of the d_sort_* buffers
  Buffer<unsigned> d_desc;
  Buffer<int> d_counts;        // [CNT_ROWS][maxB]
  Buffer<uint32_t> d_warnings; // [maxB]
  Buffer<MinMax> d_minmax;
  Buffer<VoxelFrame> d_vf;
  Buffer<EceFrame> d_ef;
  Buffer<PlaneFrame> d_pf;
  Buffer<PlaneRecord> d_prec;
  Buffer<double> d_partial;  // [maxB][chunks][10]
  Buffer<double> d_thr;
  Buffer<int> d_pack_off;  // [PK_N][maxB]
  Buffer<PackMeta> d_meta;
  Buffer<unsigned long long> d_pack_cursor;  // PCOP_OUT_DEVICE: bytes of d_pack used by the call so far
  // from here on, buffers that grow (grow(), never shrunk) with the parameters or with the calls the lane has run
  Buffer<unsigned char> d_pack;  // packed results of the wave in flight (PCOP_OUT_DEVICE: of all waves of the call)
  // pcop_process_batch_occupancy (allocated by the first such call; counts / grids grow with W x H and with the
  // largest wave the lane has run)
  Buffer<int> d_occ_counts;          // [wave frames][cells] int32
  Buffer<signed char> d_occ_grids;   // [wave frames][cells]
  Buffer<Mat34> d_occ_mats;          // [maxB][2] world_to_sensor, sensor_to_world
  HostBuffer<Mat34> h_occ_mats;      // pinned staging of the same
  cudaEvent_t ev_grids_copied = nullptr;  // the last copy out of d_occ_grids
  Buffer<unsigned char> d_raw;  // staging of raw PointCloud2 payloads from host memory: one message, or the host
                                // messages of one wave at 256-byte aligned offsets (a quarter more slack when it grows)
  Buffer<Pc2Frame> d_pc2;       // decode descriptors of k_pc2_ingest: one per message of a wave
  HostBuffer<Pc2Frame> h_pc2;   // pinned staging of the same (the batched PointCloud2 wave)
  int pc2_msgs = 0, pc2_tiles = 0; // messages and record tiles of the wave in flight (a repeat decodes them again)
  // single-frame occupancy calls (lane 0): pcop_occupancy_grid's int64 counts, int64 row averages and int8 cells;
  // pcop_occupancy_shadows' grid cells, CSR copy, records and warning word
  Buffer<unsigned char> d_occ, d_shadow;
  // PCOP_OUT_FOOTPRINTS (allocated by the first call with the bit, or the first pcop_cluster_footprints): boxes
  // [maxB][cap][8], hull sizes and CSR offsets [maxB][cap + 1], staged and final hull indices [maxB][cap]
  Buffer<float> d_fp_box;
  Buffer<int> d_fp_count, d_fp_stage, d_fp_hoff, d_fp_hidx;

  // pinned host
  HostBuffer<int> h_counts;  // [CNT_ROWS][maxB]
  HostBuffer<uint32_t> h_warnings;
  HostBuffer<PlaneRecord> h_prec;
  HostBuffer<PackMeta> h_meta;
  HostBuffer<int> h_n_in;  // staging for the per-frame input sizes
  HostBuffer<unsigned long long> h_stats;
  // pinned result buffers: two per lane, used by alternate calls, so the pointers a call returns stay valid while the
  // NEXT call runs (a consumer may still be reading them, e.g. the multi-GPU result gather)
  HostBuffer<unsigned char> h_pack_buf[2];
  int h_pack_sel = 0;
  size_t h_pack_used = 0;  // of the running call
  HostBuffer<unsigned char>& h_pack() { return h_pack_buf[h_pack_sel]; }  // the running call's

  int wave_seq = 0;                 // waves of the running call seen by this lane
  int call_lane_waves = 1;          // waves of the running call dealt to this lane
  bool pending = false;             // a wave is enqueued and not yet collected
  int pend_w0 = 0, pend_B = 0;
  int pend_max_n = 1;
  WaveRoute route;                  // of the wave in flight
  std::vector<const void**> fixups;  // result pointers of the running call that hold a pinned-buffer offset (finish_wave)
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
  Buffer<uint32_t> d_vf_flags;  // [maxB]
  unsigned long long* d_vf_pair[2] = {nullptr, nullptr};  // (overlays, see init_lane)
  HostBuffer<uint32_t> h_vf_flags;
  // partition voxel path (allocated and grown by apply_params while the plan allows the path)
  Buffer<uint32_t> d_vp_hist, d_vp_bstart, d_vp_nstart;
  Buffer<unsigned short> d_vp_ne;
  Buffer<uint2> d_vp_grec;         // [maxB][vp_gstride]
  Buffer<unsigned> d_vp_desc;      // [maxB][vp_gstride]
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

// The one way a lane's buffer grows: when b holds fewer than n elements, wait for the lane's kernels and copies (they
// may still use the old allocation), free it and allocate exactly n.  On failure b is left empty.
template <class T, bool Pinned>
int grow(Lane* l, Buffer<T, Pinned>& b, size_t n) {
  if (n <= b.size()) return PCOP_OK;
  pcop_handle* h = l->h;
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->cstream));
  return b.alloc(h, n);
}

inline uint32_t effective_outputs(const pcop_params& p) {
  uint32_t m = p.outputs & (uint32_t)(PCOP_OUT_ALL | PCOP_OUT_FOOTPRINTS | PCOP_OUT_DEVICE);
  if (p.publish_point_clouds) m |= PCOP_OUT_ALL;  // od.cpp:945: intermediates wanted
  if (!p.enable_crop) m &= ~(uint32_t)PCOP_OUT_CROP;
  if (!p.enable_voxel) m &= ~(uint32_t)PCOP_OUT_VOXEL;
  if (!p.enable_sor) m &= ~(uint32_t)PCOP_OUT_SOR;
  if (!p.enable_plane) m &= ~(uint32_t)PCOP_OUT_PLANE;
  if (!p.enable_cluster) m &= ~(uint32_t)(PCOP_OUT_CLUSTERS | PCOP_OUT_OBSTACLES | PCOP_OUT_FOOTPRINTS);
  return m;
}

// rows of the count table a wave copies to the host: CNT_HULL, the last row, only when footprints are requested
inline int count_rows(uint32_t mask) { return (mask & PCOP_OUT_FOOTPRINTS) ? CNT_ROWS : CNT_HULL; }

inline size_t pack_capacity_bytes(uint32_t mask, int B, int cap) {
  size_t bytes = 0;
  for (const PackArray& a : kPack)
    if (mask & a.bit) bytes += ((size_t)B * (cap + 1)) * a.elem_bytes + 256;
  return (bytes + 256 + 255) & ~(size_t)255;
}

// the raw PointCloud2 staging of lane l holds at least `bytes` (when it grows, by a quarter more)
inline int grow_raw(Lane* l, size_t bytes) {
  return bytes <= l->d_raw.size() ? PCOP_OK : grow(l, l->d_raw, bytes + bytes / 4 + 256);
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
  // plane ping-pong clouds (only frames that need a second pass touch them): buffers the chain has no use for by then,
  // and never the stage input, which pass 0 reads while it writes buf[0] and which a repeat of the stage reads again.
  // The cropped cloud and the input staging are dead once the plane stage starts (the fused voxel path gathers from
  // the caller's / staged input before it) unless the stage reads them: then the SOR output (SOR off) and the voxel
  // output (crop, voxel and SOR off) take their place.
  a.buf[0] = (in == l->d_crop) ? l->d_sor : l->d_crop;
  a.buf[1] = (in == l->d_in) ? l->d_vox : l->d_in;
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
int depth_ingest(pcop_handle* h, const pcop_depth_image& im, const float* t16, float4* dst);  // (validated image)
// the footprint buffers of lane l hold a wave (grow(), on the first call that asks for footprints)
int grow_footprints(Lane* l);
// the footprints of lane l's wave in flight from its remaining cloud `in` (frame stride in_stride) and clusters
int enqueue_footprints(Lane* l, const Ctx& c, const float4* in, size_t in_stride);
__global__ void k_zero_u32(uint32_t* p, int n);  // batch.cu; upload_single zeroes one frame's warning word with it

}  // namespace pcop
