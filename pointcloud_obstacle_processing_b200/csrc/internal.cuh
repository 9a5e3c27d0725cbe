// Host-side interfaces between the stage translation units.
#pragma once
#include "common.cuh"

struct pcop_handle;

namespace pcop {

// records the error text in the handle (and the thread's global error slot); returns PCOP_ERR_CUDA
int fail_cuda(pcop_handle* h, cudaError_t e, const char* expr, const char* file, int line);

// Optional per-kernel timing: CUDA event pairs recorded on the launching stream around every
// kernel launch of a call, resolved after the call's final synchronisation (bench.py's live
// roofline measurement).  Disabled => zero overhead beyond one branch per launch.
struct KernelTimers {
  static constexpr int MAX_SLOTS = 8192;
  static constexpr int MAX_NAMES = 64;
  bool enabled = false;
  cudaEvent_t* ev = nullptr;  // [2*MAX_SLOTS], created lazily
  int used = 0;
  const char* slot_name[MAX_SLOTS];
  // accumulated per kernel name
  int n_names = 0;
  const char* names[MAX_NAMES];
  double total_us[MAX_NAMES];
  long long launches[MAX_NAMES];
};

struct Ctx {
  cudaStream_t stream;
  int B;    // frames in the wave
  int cap;  // per-frame capacity (points) = stride of every frame-strided buffer
  int64_t* launches;
  KernelTimers* kt;
  int grid_cap;  // points per frame the launch grids must cover (<= cap; the host lowers it when it knows a bound)
};

inline void count_launch(const Ctx& c, int n = 1) { *c.launches += n; }

struct KScope {
  const Ctx& c;
  int slot;
  KScope(const Ctx& cc, const char* name) : c(cc), slot(-1) {
    KernelTimers* k = c.kt;
    if (k && k->enabled && k->ev && k->used < KernelTimers::MAX_SLOTS) {
      slot = k->used++;
      k->slot_name[slot] = name;
      cudaEventRecord(k->ev[2 * slot], c.stream);
    }
  }
  ~KScope() {
    if (slot >= 0) cudaEventRecord(c.kt->ev[2 * slot + 1], c.stream);
  }
};
#define KL(ctx, name, ...)          \
  do {                              \
    ::pcop::KScope _ks(ctx, name);  \
    __VA_ARGS__;                    \
  } while (0)

// ---- batched stable LSD radix sort of (key32, val32) pairs ---------------------
struct SortBufs {
  uint32_t* key[2];  // [B*cap] ping-pong
  uint32_t* val[2];
  uint32_t* hist;    // [B][RS_MAX_PASSES][RS_BINS]  (becomes exclusive bin bases)
  uint32_t* desc;    // [RS_MAX_PASSES][B][tiles][RS_BINS] look-back descriptors
  uint32_t* maxkey;  // [B]  written (atomicMax) by the kernel that produced the keys
  int* npass;        // [B]  passes actually needed for this frame (>= 1)
  unsigned long long* stats;  // [1] keys moved by all sort passes of the call (accounting only)
};
size_t sort_desc_bytes(int B, int cap);
// Sorts frame f's `count[f]` pairs that sit in key[0]/val[0] (val[0] is ignored and taken as
// 0..count-1 when iota_vals).  Frame f's result is in key[npass[f]&1] / val[npass[f]&1].
void radix_sort_batched(const Ctx& c, const SortBufs& s, const int* count, bool iota_vals);
// zero maxkey before a key-producing kernel
void sort_reset_maxkey(const Ctx& c, const SortBufs& s);

// ---- stages ---------------------------------------------------------------------
struct CropArgs {
  const float4* in;
  size_t in_stride;  // points between frames of `in`
  const int* n_in;   // [B]
  float4* out;       // [B*cap]
  int* kept_idx;     // [B*cap]
  int* n_out;        // [B]
  MinMax* minmax;    // [B] of the kept points
  unsigned* desc;    // [B*tiles] compaction descriptors (zeroed here)
  float lim[6];      // x_min,x_max,y_min,y_max,z_min,z_max
};
void run_crop(const Ctx& c, const CropArgs& a);

// min/max of an arbitrary frame-strided cloud (used when crop is disabled and by the search grids);
// finite_only skips +-inf as well as NaN (the search grids must only span finite points)
void run_minmax(const Ctx& c, const float4* pts, size_t stride, const int* n, MinMax* minmax, bool finite_only = false);

struct VoxelArgs {
  const float4* in;  // [B*stride]
  size_t in_stride;
  const int* n_in;
  const MinMax* minmax;
  float leaf;
  VoxelFrame* vf;      // [B]
  SortBufs sort;
  unsigned* desc;      // compaction descriptors [B*tiles]
  int* run_start;      // [B*cap]
  float4* out;         // [B*cap]
  uint32_t* out_keys;  // [B*cap]
  int* n_out;          // [B]
  uint32_t* warnings;  // [B]
};
void run_voxel(const Ctx& c, const VoxelArgs& a);

// Uniform grid over a frame-strided cloud: cell >= `cell`*(1+2^-8) per axis (<= 1024 cells per axis),
// points radix-sorted by cell key; sorted_pts[j] = {x,y,z, original index}.  parent/csize (optional)
// are initialised for the union-find.  Sorted keys: sort.key[sort.npass[f]&1].
// clique != 0 (ECE): cell edge = cell*0.5728 (< cell/sqrt(3)) so that all points of a cell are within `cell` of each
// other, per-frame fallback to mode 1 when that needs more than 1024 cells on an axis; points with a non-finite
// coordinate get a private key >= 2^30.
void run_grid_sort(const Ctx& c, const float4* in, size_t in_stride, const int* n_in, float cell, MinMax* minmax,
                   EceFrame* ef, const SortBufs& sort, float4* sorted_pts, int* parent, int* csize, int clique = 0);

// ---- fused crop + VoxelGrid fast path (stage_voxel_fused.cu) ----------------------------------------------
struct VoxFusedPlan {
  int ok;          // the crop box bounds the voxel grid tightly enough (and PCL's overflow guard cannot fire)
  float lim[6];    // x_min,x_max,y_min,y_max,z_min,z_max
  float inv;       // 1 / leaf
  int b0[3];       // floor(lo_a * inv)
  uint32_t nx, ny, nz;  // cells of the crop box per axis
  int bits, npass, digit_bits;
  // partition variant (stage_voxel_part.cu): bucket = key >> part_shift, nb buckets per frame
  int part_ok, part_shift, nb, nb_pad;
};
VoxFusedPlan make_vox_fused_plan(const pcop_params& p);
void vox_part_plan(VoxFusedPlan& pl, size_t max_points);  // fills the partition fields of a plan
size_t vox_fused_hist_elems(int B);
size_t vox_fused_desc_bytes(int B, int cap);
struct VoxelFusedArgs {
  const float4* in;  // wave input (uncropped), frame-strided
  size_t in_stride;
  const int* n_in;
  VoxFusedPlan plan;
  float leaf;
  MinMax* minmax;    // [B] min/max of the crop survivors
  VoxelFrame* vf;    // [B]
  SortBufs sort;     // hist: vox_fused_hist_elems, desc: vox_fused_desc_bytes (key/val arrays unused)
  unsigned long long* pair[2];  // [B*cap] ping-pong (key << 32) | original index
  unsigned* desc;    // compaction descriptors
  uint32_t* flags;   // [B] bit 0: the frame needs the generic path (a survivor with a non-finite y or z)
  uint32_t* warnings;  // [B] zeroed by the stage's init kernel when non-null (saves the wave's k_zero_u32 launch)
  int* n_crop;       // [B] out: M
  float4* out;       // [B*cap] voxel centroids
  uint32_t* out_keys;
  int* n_out;        // [B] V
  int want_keys;     // PCL's voxel keys are an output (PCOP_OUT_VOXEL); otherwise they are not computed
};
void run_voxel_fused(const Ctx& c, const VoxelFusedArgs& a);

// ---- fused crop + VoxelGrid, partition variant (stage_voxel_part.cu) ----------------------------------------------
int vox_part_chunks(int max_n, int B);
int vox_part_group_bound(const VoxFusedPlan& pl, int max_n);  // worst-case groups of a frame of max_n points
size_t vox_part_hist_elems(int B);
size_t vox_part_start_elems(int B);
size_t vox_part_chunk_start_elems(int B);
size_t vox_part_bucket_elems(int B);
struct VoxelPartArgs {
  const float4* in;  // wave input (uncropped), frame-strided
  size_t in_stride;
  const int* n_in;
  VoxFusedPlan plan;
  float leaf;
  MinMax* minmax;            // [B] min/max of the crop survivors
  VoxelFrame* vf;            // [B]
  uint32_t* ghist;           // [B][chunks][nb_pad] per-chunk bucket counts -> offsets inside the bucket
  uint32_t* chunk_start;     // [B][chunks][nb_pad] first slot of every (chunk, bucket) range
  unsigned short* ne_bucket; // [B][16384] non-empty buckets in key order
  uint32_t* ne_start;        // [B][16385] their element starts (then M)
  uint2* grec;               // [B][group_stride] {element start, first non-empty ordinal} of every group (+ end marker)
  int* n_groups;             // [B]
  float4* part;              // [B*cap] {x, y, z, original index} partitioned by bucket
  unsigned* desc;            // [B][group_stride] look-back descriptors
  int group_stride;
  int group_launch;          // groups per frame the reduce grid covers (a frame with more raises flag bit 2)
  uint32_t* flags;           // [B] bit 0: NaN y/z survivor (generic path), bit 1: bucket too large (LSD path), bit 2: see above
  uint32_t* warnings;        // [B] zeroed by the stage's init kernel when non-null
  int* n_crop;               // [B] out: M
  float4* out;               // [B*cap] voxel centroids
  uint32_t* out_keys;
  int* n_out;                // [B] V
  int want_keys;
};
void run_voxel_part(const Ctx& c, const VoxelPartArgs& a);

struct SorArgs {
  const float4* in;
  size_t in_stride;
  const int* n_in;
  int meanK;
  double mul;
  float cell;  // grid cell for the k-NN search (speed only)
  MinMax* minmax;
  EceFrame* gf;
  SortBufs sort;
  float4* sorted_pts;  // [B*cap]
  float* dist;         // [B*cap] mean k-NN distance per point (original order)
  double* partial;     // [B][chunks][2]
  double* thr;         // [B]
  unsigned* desc;
  float4* out;
  int* kept_idx;
  int* n_out;
  uint32_t* warnings;
};
void run_sor(const Ctx& c, const SorArgs& a);

struct PlaneArgs {
  const float4* in;  // plane-loop input (S points per frame)
  size_t in_stride;
  const int* n_in;
  int* n_in_copy;  // optional [B]: the init kernel copies n_in there (the count row of a disabled SOR stage)
  float4* buf[2];  // [B*cap] ping-pong clouds
  int* src[2];     // [B*cap] index into `in` of each remaining point
  int* inlier_idx; // [B*cap] last pass' inliers
  PlaneFrame* pf;  // [B]
  double* partial; // [B][chunks][10] chunk partials of the large tier's frames above 131072 points
  const int* rng;  // [RNG_TABLE] rnd() values
  int large_tier;  // also launch the tier for frames above plane_small_tier_max() points
  PlaneConst pc;
  uint32_t* warnings;
  // outputs
  float4* out;   // [B*cap] remaining cloud (planar_cloud_y, od.cpp:765)
  int* out_src;  // [B*cap] index into `in` of each remaining point
  int* n_out;    // [B] remaining count
};
// The whole loop of od.cpp:376-399 for every frame of the wave: one thread-block cluster per frame runs every pass
// (two or three launches, no host synchronisation).  Returns the first failing runtime error.
cudaError_t run_plane(const Ctx& c, const PlaneArgs& a);
// Largest plane-stage input the small tier processes (see run_plane).
int plane_small_tier_max();

struct ClusterArgs {
  const float4* in;  // remaining cloud, frame f at in + f*in_stride
  size_t in_stride;
  const int* n_in;
  float tol;
  int min_size, max_size;
  int small_max;  // largest cloud the fused shared-memory kernel takes (0: generic path only)
  MinMax* minmax;
  EceFrame* ef;
  SortBufs sort;
  float4* sorted_pts;  // [B*cap] xyz + original index in w
  int* parent;         // [B*cap]
  int* csize;          // [B*cap]
  int* roots;          // [B*cap]
  int* rank_of;        // [B*cap]
  int* cell_start;     // [B*cap] first sorted position of each occupied cell
  uint32_t* cell_key;  // [B*cap] key of each occupied cell
  int* n_cells;        // [B]
  int* n_route;        // [B] scratch: per-frame point count as seen by the generic path
  unsigned* desc;
  int* offsets;  // [B*(cap+1)]
  int* indices;  // [B*cap]
  int* n_clusters;
  int* n_cluster_pts;
  float4* obstacles;  // [B*cap]
  double* partial;    // [B][partial_stride] scratch of the centroid pass (sums of the pieces of large clusters)
  int partial_stride;
};
// Largest cloud the fused shared-memory clustering kernel takes (stage_cluster_small.cu).
constexpr int ECE_SMALL_MAX = 8960;
// ECE_SMALL_MAX, or the value of the environment variable PCOP_ECE_SMALL_MAX clamped to [0, ECE_SMALL_MAX]
// (0 forces every frame through the generic path; used by the tests to cover both paths).  Read by pcop_create.
int ece_small_limit();
// returns true when the generic centroid/radius kernel still has to run (see stage_cluster.cu)
bool run_cluster(const Ctx& c, const ClusterArgs& a, bool with_generic);
void run_cluster_small(const Ctx& c, const ClusterArgs& a, int small_max, bool zero_skipped);
void run_centroid_radius(const Ctx& c, const ClusterArgs& a);

// ---- occupancy grid (stage_occupancy.cu; od.cpp:134-157, 175-269, 467-672, 817-833) ------------------------------
struct OccGrid {
  float lim[6];  // crop box x_min,x_max,y_min,y_max,z_min,z_max (od.cpp:197-199)
  float block_size, dev_percent;
  int W, H;
  long long cells;  // W * H
};
// counters of the batched count kernel, chosen from the grid size alone: a shared-memory histogram of 32-bit or of
// 16-bit counters (the latter with chunks of at most 65535 points) while it fits OCC_SMEM_BYTES, else global atomics
enum { OCC_COUNT_SMEM32 = 0, OCC_COUNT_SMEM16 = 1, OCC_COUNT_GLOBAL = 2 };
constexpr int OCC_SMEM_BYTES = 220 * 1024;
int occ_count_mode(long long cells);
// one frame: 64-bit counts (zeroed by the caller), then row averages + cells
void run_occ_count(const Ctx& c, const float4* in, int n, const OccGrid& g, unsigned long long* counts);
void run_occ_finish(const Ctx& c, const unsigned long long* counts, const OccGrid& g, long long* row_avg, signed char* grid);
// every frame of a wave: counts [B][cells] int32 (zeroed by the caller), then grids [B][cells]; the threshold also
// clears PCOP_WARN_SHADOW_DEGENERATE in warnings[f] (the shadow kernel sets it afresh)
// returns the first error of the dynamic shared-memory opt-in or the launch
cudaError_t run_occ_count_wave(const Ctx& c, const float4* in, size_t in_stride, const int* n_in, const OccGrid& g,
                               int* counts);
void run_occ_finish_wave(const Ctx& c, const int* counts, const OccGrid& g, signed char* grids, uint32_t* warnings);

struct Mat34 {
  float m[12];  // rows 0..2 of a row-major 4x4 (pcl::transformPointCloud's coefficient formula)
};
struct OccShadowArgs {  // frame f of c.B: every array below at its frame's stride
  const float4* cloud;  // remaining cloud (planar_cloud_y, od.cpp:765)
  size_t cloud_stride;
  const int* n_points;  // [B] device
  const int* offsets;   // CSR [n_clusters + 1]
  size_t offsets_stride;
  const int* indices;
  size_t indices_stride;
  const int* n_clusters;  // [B] device
  const Mat34* mats;      // [B][2] device: world_to_sensor, sensor_to_world (the TF lookups of od.cpp:592 / 570, 634)
  float y_min, x_max, block_size;
  int W;
  long long size;       // W * H = grid stride
  int opacity;          // grid_opacity
  signed char* grid;    // [B][size] in/out
  int* records;         // [n_clusters][6] or nullptr (one frame only)
  uint32_t* warnings;   // [B], OR-ed
};
// blocks_per_frame: blocks that share a frame's clusters; max_points: bound of every frame's n_points
void run_occ_shadows(const Ctx& c, const OccShadowArgs& a, int blocks_per_frame, int max_points);

}  // namespace pcop
