// C ABI of the library (include/pcop.h): handle creation and parameters, the single-frame and stage-isolated entry
// points.  The batched calls run in the wave scheduler (batch.cu).
// Every buffer is allocated by pcop_create (pcop_set_params may grow the partition voxel path's); the pinned result
// buffer only grows (a second call of the same shape allocates nothing).
#include <cstdio>
#include <cstdlib>

#include "handle.cuh"
#include "primitives.cuh"

using namespace pcop;

static thread_local std::string g_global_error;

namespace pcop {
int fail_cuda(pcop_handle* h, cudaError_t e, const char* expr, const char* file, int line) {
  char buf[512];
  snprintf(buf, sizeof(buf), "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, expr);
  if (h) h->err = buf;
  g_global_error = buf;
  return PCOP_ERR_CUDA;
}

int fail(pcop_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  g_global_error = msg;
  return code;
}
}  // namespace pcop

namespace {

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
VoxFusedPlan make_plan(const pcop_params& p, size_t max_points) {
  VoxFusedPlan pl = make_vox_fused_plan(p);
  vox_part_plan(pl, max_points);
  const char* s = getenv("PCOP_VOXEL_FUSED");
  if (s && s[0] == '0') pl.ok = 0;
  if (s && (s[0] == 'l' || s[0] == 'L')) pl.part_ok = 0;
  if (!pl.ok) pl.part_ok = 0;
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

__global__ void k_plane_record(const PlaneFrame* __restrict__ pf, PlaneRecord* __restrict__ rec, int* __restrict__ n_inl,
                               int* __restrict__ n_clus, int* __restrict__ n_clus1, int plane_enabled, int B) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < B) plane_record_one(pf, rec, n_inl, n_clus, n_clus1, plane_enabled, f);
}

// upload a single cloud into lane 0's d_in as frame 0 and set a count row
int upload_single(pcop_handle* h, const float* xyzw, int32_t n, int count_row) {
  if (n < 0) return fail(h, PCOP_ERR_BAD_PARAM, "negative point count");
  if (n > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  Lane* l = h->lanes[0].get();
  l->h_n_in[0] = n;
  PCOP_CUDA_TRY(cudaMemcpyAsync(l->cnt(count_row), l->h_n_in, sizeof(int), cudaMemcpyHostToDevice, l->stream));
  if (n > 0) PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_in, xyzw, (size_t)n * 16, cudaMemcpyDefault, l->stream));
  k_zero_u32<<<1, 32, 0, l->stream>>>(l->d_warnings, 1);
  return PCOP_OK;
}

// a cloud for a single-frame kernel: device memory is read in place, host memory is copied into lane 0's d_in
int device_cloud(pcop_handle* h, const float* xyzw, int32_t n, const float4** src) {
  Lane* l = h->lanes[0].get();
  *src = reinterpret_cast<const float4*>(xyzw);
  if (n > 0 && !is_device_pointer(xyzw)) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_in, xyzw, (size_t)n * 16, cudaMemcpyHostToDevice, l->stream));
    *src = l->d_in;
  }
  return PCOP_OK;
}

int download(pcop_handle* h, void* dst, const void* src, size_t bytes) {
  if (!dst || bytes == 0) return PCOP_OK;
  PCOP_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->lanes[0]->stream));
  return PCOP_OK;
}

// one 32-bit word of lane 0 (a count row entry or the warning word) into *out, if out is non-null
int fetch_word(pcop_handle* h, const void* src, void* out) {
  Lane* l = h->lanes[0].get();
  PCOP_CUDA_TRY(cudaMemcpyAsync(l->h_counts, src, sizeof(uint32_t), cudaMemcpyDeviceToHost, l->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  if (out) memcpy(out, l->h_counts, sizeof(uint32_t));
  return PCOP_OK;
}

// streams, events and wave buffers of one lane: everything that does not depend on the parameters
int init_lane(Lane* l) {
  pcop_handle* h = l->h;
  PCOP_CUDA_TRY(cudaStreamCreateWithFlags(&l->stream, cudaStreamNonBlocking));
  PCOP_CUDA_TRY(cudaStreamCreateWithFlags(&l->cstream, cudaStreamNonBlocking));
  const size_t BC = (size_t)h->maxB * h->cap;
  const int B = h->maxB;
  const int chunks = cdiv(h->cap, TS_CHUNK);
  const int tiles = cdiv(h->cap, CT_TILE);
  TRY(dalloc(h, &l->d_in, BC));
  TRY(dalloc(h, &l->d_crop, BC));
  TRY(dalloc(h, &l->d_vox, BC));
  TRY(dalloc(h, &l->d_sor, BC));
  // plane ping-pong clouds (only frames that need a second pass touch them): the cropped cloud and the input staging
  // are dead by then (the fused voxel path gathers from the caller's / staged input before the plane stage starts)
  l->d_pbuf[0] = l->d_crop;
  l->d_pbuf[1] = l->d_in;
  TRY(dalloc(h, &l->d_rem, BC));
  TRY(dalloc(h, &l->d_sorted, BC));
  TRY(dalloc(h, &l->d_obst, BC));
  TRY(dalloc(h, &l->d_crop_kept, BC));
  TRY(dalloc(h, &l->d_run_start, BC));
  TRY(dalloc(h, &l->d_sor_kept, BC));
  TRY(dalloc(h, &l->d_psrc[0], BC));
  TRY(dalloc(h, &l->d_psrc[1], BC));
  TRY(dalloc(h, &l->d_rem_src, BC));
  TRY(dalloc(h, &l->d_inliers, BC));
  TRY(dalloc(h, &l->d_parent, BC));
  TRY(dalloc(h, &l->d_csize, BC));
  TRY(dalloc(h, &l->d_roots, BC));
  TRY(dalloc(h, &l->d_rank, BC));
  TRY(dalloc(h, &l->d_indices, BC));
  TRY(dalloc(h, &l->d_cell_start, BC));
  TRY(dalloc(h, &l->d_cell_key, BC));
  TRY(dalloc(h, &l->d_offsets, BC + B));
  TRY(dalloc(h, &l->d_vox_keys, BC));
  TRY(dalloc(h, &l->d_sor_dist, BC));
  TRY(dalloc(h, &l->sort.key[0], BC));
  TRY(dalloc(h, &l->sort.key[1], BC));
  TRY(dalloc(h, &l->sort.val[0], BC));
  TRY(dalloc(h, &l->sort.val[1], BC));
  TRY(dalloc(h, &l->sort.hist, std::max((size_t)B * RS_MAX_PASSES * RS_BINS, vox_fused_hist_elems(B))));
  {
    unsigned char* d = nullptr;
    TRY(dalloc(h, &d, std::max(sort_desc_bytes(B, h->cap), vox_fused_desc_bytes(B, h->cap))));
    l->sort.desc = (uint32_t*)d;
  }
  TRY(dalloc(h, &l->d_vf_flags, B));
  // (key, index) pairs of the fused voxel path: they overlay the search-grid point list of SOR / clustering
  l->d_vf_pair[0] = reinterpret_cast<unsigned long long*>(l->d_sorted);
  l->d_vf_pair[1] = reinterpret_cast<unsigned long long*>(l->d_sorted) + BC;
  TRY(halloc(h, &l->h_vf_flags, B));
  TRY(dalloc(h, &l->sort.maxkey, B));
  TRY(dalloc(h, &l->sort.npass, B));
  TRY(dalloc(h, &l->sort.stats, 1));
  TRY(halloc(h, &l->h_stats, 1));
  TRY(dalloc(h, &l->d_desc, (size_t)B * tiles));
  TRY(dalloc(h, &l->d_counts, (size_t)CNT_ROWS * B));
  TRY(dalloc(h, &l->d_warnings, B));
  TRY(dalloc(h, &l->d_minmax, B));
  TRY(dalloc(h, &l->d_vf, B));
  TRY(dalloc(h, &l->d_ef, B));
  TRY(dalloc(h, &l->d_pf, B));
  TRY(dalloc(h, &l->d_prec, B));
  TRY(dalloc(h, &l->d_partial, (size_t)B * chunks * 10));
  TRY(dalloc(h, &l->d_thr, B));
  TRY(dalloc(h, &l->d_pack_off, (size_t)PK_N * B));
  TRY(dalloc(h, &l->d_meta, 1));
  TRY(dalloc(h, &l->d_pack_cursor, 1));
  TRY(halloc(h, &l->h_counts, (size_t)CNT_ROWS * B));
  TRY(halloc(h, &l->h_warnings, B));
  TRY(halloc(h, &l->h_prec, B));
  TRY(halloc(h, &l->h_meta, 1));
  TRY(halloc(h, &l->h_n_in, (size_t)B + 16));
  PCOP_CUDA_TRY(cudaMemset(l->d_counts, 0, sizeof(int) * CNT_ROWS * B));
  PCOP_CUDA_TRY(cudaMemset(l->d_pf, 0, sizeof(PlaneFrame) * B));
  for (int s = 0; s < PCOP_N_STAGES; ++s)
    for (int i = 0; i < 2; ++i) PCOP_CUDA_TRY(cudaEventCreate(&l->ev_stage[s][i]));
  PCOP_CUDA_TRY(cudaEventCreateWithFlags(&l->ev_lane_done, cudaEventDisableTiming));
  PCOP_CUDA_TRY(cudaEventCreateWithFlags(&l->ev_copied, cudaEventDisableTiming));
  PCOP_CUDA_TRY(cudaEventCreateWithFlags(&l->ev_meta, cudaEventDisableTiming));
  PCOP_CUDA_TRY(cudaEventCreateWithFlags(&l->ev_grids_copied, cudaEventDisableTiming));
  return PCOP_OK;
}

// Parameters of pcop_create and pcop_set_params (validated): every lane's buffers that depend on them are grown
// first (never shrunk), so a failure leaves the handle with its previous parameters; then the RANSAC table (16 KB of
// the seed's rnd() values), the crop + VoxelGrid plan and the lanes' partition-path stride and route history.
int apply_params(pcop_handle* h, const pcop_params& p) {
  const VoxFusedPlan plan = make_plan(p, (size_t)h->cap);
  const int gstride = plan.part_ok ? vox_part_group_bound(plan, h->cap) + 1 : 0;
  const int B = h->maxB;
  for (auto& lp : h->lanes) {
    Lane* l = lp.get();
    if (plan.part_ok && !l->d_vp_ne) {
      TRY(dalloc(h, &l->d_vp_hist, vox_part_hist_elems(B)));
      TRY(dalloc(h, &l->d_vp_bstart, vox_part_chunk_start_elems(B)));
      TRY(dalloc(h, &l->d_vp_nstart, vox_part_start_elems(B)));
      TRY(dalloc(h, &l->d_vp_ne, vox_part_bucket_elems(B)));
    }
    if (gstride > l->vp_gcap) {
      PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
      cudaFree(l->d_vp_grec);  // (not tracked in dev_allocs)
      cudaFree(l->d_vp_desc);
      l->d_vp_grec = nullptr;
      l->d_vp_desc = nullptr;
      l->vp_gcap = 0;
      PCOP_CUDA_TRY(cudaMalloc((void**)&l->d_vp_grec, sizeof(uint2) * B * gstride));
      PCOP_CUDA_TRY(cudaMalloc((void**)&l->d_vp_desc, sizeof(unsigned) * B * gstride));
      l->vp_gcap = gstride;
    }
    TRY(ensure_pack_capacity(l, effective_outputs(p)));
  }
  std::vector<int> tbl(RNG_TABLE);
  fill_rng_table(p.ransac_seed, tbl.data(), RNG_TABLE);
  PCOP_CUDA_TRY(cudaMemcpy(h->d_rng, tbl.data(), sizeof(int) * RNG_TABLE, cudaMemcpyHostToDevice));
  h->params = p;
  h->vplan = plan;
  for (auto& l : h->lanes) {  // (route history: the LSD-path countdown and the group hint start over, the sizes of the last wave are kept)
    if (plan.part_ok) {
      l->vp_gstride = gstride;
      l->vp_group_hint = gstride - 1;
    }
    l->vox_lsd_waves = 0;
  }
  return PCOP_OK;
}

}  // namespace

pcop::Lane::~Lane() {
  if (stream) cudaStreamSynchronize(stream);
  if (cstream) cudaStreamSynchronize(cstream);
  cudaFree(d_pack);  // (the buffers that grow are not tracked in dev_allocs)
  cudaFree(d_raw);
  cudaFree(d_occ_counts);
  cudaFree(d_occ_grids);
  cudaFree(d_vp_grec);
  cudaFree(d_vp_desc);
  cudaFree(d_pc2);
  if (h_pc2) cudaFreeHost(h_pc2);
  for (int i = 0; i < 2; ++i)
    if (h_pack_buf[i]) cudaFreeHost(h_pack_buf[i]);
  for (cudaEvent_t e : {ev_lane_done, ev_copied, ev_meta, ev_grids_copied})
    if (e) cudaEventDestroy(e);
  for (const TraceRec& r : trace_recs)  // (PCOP_TRACE)
    for (cudaEvent_t e : {r.meta, r.c0, r.c1})
      if (e) cudaEventDestroy(e);
  for (int s = 0; s < PCOP_N_STAGES; ++s)
    for (int i = 0; i < 2; ++i)
      if (ev_stage[s][i]) cudaEventDestroy(ev_stage[s][i]);
  if (cstream) cudaStreamDestroy(cstream);
  if (stream) cudaStreamDestroy(stream);
}

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

int pcop_create(const pcop_params* params, int device, size_t max_points, int max_batch, pcop_handle** out) {
  // (frame-major launches put the tile index in gridDim.y, and look-back descriptors carry 30-bit prefixes)
  if (!params || !out || max_points == 0 || max_points > (size_t)65535 * BT_TILE || max_batch < 1)
    return fail(nullptr, PCOP_ERR_BAD_PARAM, "pcop_create: bad argument (max_points must be in [1, 268431360])");
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
  pcop_handle* h = new pcop_handle();
  h->device = device;
  h->cap = (int)max_points;
  h->maxB = lane_batch;
  h->wave_frames = std::min(wave_frames, lane_batch);
  h->trace = getenv("PCOP_TRACE") != nullptr;
  h->ece_small_max = ece_small_limit();
  const int st = [&] {  // everything the handle allocates, then the parameters
    TRY(validate_params(h, *params));
    PCOP_CUDA_TRY(cudaSetDevice(h->device));
    TRY(dalloc(h, &h->d_acc, (size_t)h->cap));
    TRY(dalloc(h, &h->d_rng, RNG_TABLE));
    for (int i = 0; i < 2; ++i) PCOP_CUDA_TRY(cudaEventCreate(&h->ev_call[i]));
    for (int i = 0; i < n_lanes; ++i) {
      h->lanes.emplace_back(new Lane{h});
      TRY(init_lane(h->lanes.back().get()));
    }
    return apply_params(h, *params);
  }();
  if (st != PCOP_OK) {
    g_global_error = h->err;
    pcop_destroy(h);
    return st;
  }
  *out = h;
  return PCOP_OK;
}

void pcop_destroy(pcop_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  h->lanes.clear();  // (every lane waits for its streams first)
  for (void* p : h->dev_allocs) cudaFree(p);
  for (void* p : h->host_allocs) cudaFreeHost(p);
  if (h->d_occ) cudaFree(h->d_occ);
  if (h->d_shadow) cudaFree(h->d_shadow);
  if (h->kt.ev) {
    for (int i = 0; i < 2 * KernelTimers::MAX_SLOTS; ++i) cudaEventDestroy(h->kt.ev[i]);
    delete[] h->kt.ev;
  }
  for (int i = 0; i < 2; ++i)
    if (h->ev_call[i]) cudaEventDestroy(h->ev_call[i]);
  delete h;
}

int pcop_set_params(pcop_handle* h, const pcop_params* params) {
  if (!h || !params) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  TRY(validate_params(h, *params));
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  return apply_params(h, *params);
}

int pcop_process(pcop_handle* h, const float* xyzw, int32_t n, pcop_frame_result* out) {
  return process_impl(h, xyzw, (size_t)(n > 0 ? n : 1), &n, 1, out);
}

int pcop_process_batch(pcop_handle* h, const float* xyzw, size_t frame_stride_points, const int32_t* n, int32_t batch,
                       pcop_frame_result* out) {
  return process_impl(h, xyzw, frame_stride_points, n, batch, out);
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

// the grid request of a batched call: the handle's grid (PCOP_ERR_CAPACITY above PCOP_OCC_BATCH_MAX_CELLS) + poses
static int occ_call_of(pcop_handle* h, const char* who, const float* world_to_sensor16, const float* sensor_to_world16,
                       int8_t* grids, OccCall* oc) {
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
  OccCall oc{};
  TRY(occ_call_of(h, "pcop_process_batch_occupancy", world_to_sensor16, sensor_to_world16, grids, &oc));
  if (xyzw) return process_impl(h, xyzw, frame_stride_points, n, batch, out, &oc);
  // the accumulated cloud, consumed by this run (od.cpp:701), as pcop_process_accumulated
  const int32_t acc_n = h->acc_count;
  const int st = process_impl(h, reinterpret_cast<const float*>(h->d_acc), (size_t)(acc_n > 0 ? acc_n : 1), &acc_n, 1, out, &oc);
  h->acc_count = 0;
  return st;
}

// pcop_process_batch_pointcloud2_windows, and pcop_process_batch_pointcloud2 with one message per window (`who` names
// the entry point in error messages)
static int pointcloud2_windows(pcop_handle* h, const char* who, const pcop_pointcloud2_frame* msgs, int32_t n_msgs,
                               const int32_t* window_first, int32_t batch, const float* transform16,
                               const float* world_to_sensor16, const float* sensor_to_world16, int8_t* grids,
                               pcop_frame_result* out) {
  const std::string w(who);
  if (!out || batch < 0 || n_msgs < 0 || (!msgs && n_msgs > 0) || (!window_first && (batch > 0 || n_msgs > 0)) ||
      (grids && (!world_to_sensor16 || !sensor_to_world16)))
    return fail(h, PCOP_ERR_BAD_PARAM, w + ": null argument (grids need world_to_sensor16 and sensor_to_world16)");
  if (window_first && (window_first[0] != 0 || window_first[batch] != n_msgs))
    return fail(h, PCOP_ERR_BAD_PARAM, w + ": window_first must start at 0 and end at the message count");
  for (int f = 0; f < batch; ++f)  // (then every window lies inside [0, n_msgs))
    if (window_first[f + 1] < window_first[f])
      return fail(h, PCOP_ERR_BAD_PARAM, w + ": window_first decreases at window " + std::to_string(f));
  // window by window, message by message: with one message per window the checks run in the order of
  // pcop_process_batch_pointcloud2's per-frame checks
  std::vector<int32_t> n((size_t)batch + 1, 0);  // frame f = the concatenation of its window's messages
  for (int f = 0; f < batch; ++f) {
    long long total = 0;
    for (int m = window_first[f]; m < window_first[f + 1]; ++m) {
      const pcop_pointcloud2_frame& d = msgs[m];
      if (d.n_points < 0 || (!d.data && d.n_points > 0))
        return fail(h, PCOP_ERR_BAD_PARAM, w + ": message " + std::to_string(m) + ": bad count or NULL data");
      if (!pc2_layout_ok(d.point_step, d.off_x, d.off_y, d.off_z))
        return fail(h, PCOP_ERR_BAD_PARAM,
                    w + ": message " + std::to_string(m) + ": PointCloud2 field offsets do not fit point_step");
      total += d.n_points;
    }
    if (total > h->cap)
      return fail(h, PCOP_ERR_CAPACITY, w + ": window " + std::to_string(f) + " holds " + std::to_string(total) +
                                            " points, more than max_points");
    n[f] = (int32_t)total;
  }
  OccCall oc{};
  if (grids) TRY(occ_call_of(h, who, world_to_sensor16, sensor_to_world16, grids, &oc));
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  Pc2Call pc;
  pc.msgs = msgs;
  pc.window_first = window_first;
  pc.transform16 = transform16;
  pc.on_device.resize((size_t)n_msgs);
  PayloadClassifier on_device;
  for (int m = 0; m < n_msgs; ++m) pc.on_device[m] = msgs[m].n_points > 0 && on_device(msgs[m].data);
  return process_impl(h, nullptr, (size_t)h->cap, n.data(), batch, out, grids ? &oc : nullptr, &pc);
}

int pcop_process_batch_pointcloud2_windows(pcop_handle* h, const pcop_pointcloud2_frame* messages, int32_t n_messages,
                                           const int32_t* window_first, int32_t batch, const float* transform16,
                                           const float* world_to_sensor16, const float* sensor_to_world16,
                                           int8_t* grids, pcop_frame_result* out) {
  if (!h) return fail(nullptr, PCOP_ERR_BAD_PARAM, "null handle");
  return pointcloud2_windows(h, "pcop_process_batch_pointcloud2_windows", messages, n_messages, window_first, batch,
                             transform16, world_to_sensor16, sensor_to_world16, grids, out);
}

int pcop_process_batch_pointcloud2(pcop_handle* h, const pcop_pointcloud2_frame* frames, int32_t batch,
                                   const float* transform16, const float* world_to_sensor16,
                                   const float* sensor_to_world16, int8_t* grids, pcop_frame_result* out) {
  if (!h) return fail(nullptr, PCOP_ERR_BAD_PARAM, "null handle");
  std::vector<int32_t> first((size_t)std::max(batch, 0) + 1);
  for (size_t f = 0; f < first.size(); ++f) first[f] = (int32_t)f;
  return pointcloud2_windows(h, "pcop_process_batch_pointcloud2", frames, batch, first.data(), batch, transform16,
                             world_to_sensor16, sensor_to_world16, grids, out);
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
  const cudaStream_t s = h->lanes[0]->stream;
  if (bytes) PCOP_CUDA_TRY(cudaMemcpyAsync(dst, src_device, bytes, cudaMemcpyDefault, s));
  PCOP_CUDA_TRY(cudaStreamSynchronize(s));
  return PCOP_OK;
}

int64_t pcop_last_sort_pass_keys(const pcop_handle* h) { return h ? (int64_t)h->sort_pass_keys : 0; }
double pcop_last_d2h_bytes(const pcop_handle* h) { return h ? h->d2h_bytes : 0.0; }

// ---- accumulator ingest (od.cpp:691-698) -------------------------------------------------
static int transform_into(pcop_handle* h, const float* xyzw, int32_t n, const float* t16, int is_dense, float4* dst) {
  Lane* l = h->lanes[0].get();
  const float4* src;
  TRY(device_cloud(h, xyzw, n, &src));
  Mat34 t;
  const float ident[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
  memcpy(t.m, t16 ? t16 : ident, sizeof(t.m));
  Ctx c = make_ctx(l, 1, n);
  KL(c, "k_transform", k_transform<<<cdiv(n, 256), 256, 0, l->stream>>>(src, n, t, is_dense, dst));
  count_launch(c);
  return PCOP_OK;
}

int pcop_accumulate(pcop_handle* h, const float* xyzw, int32_t n, const float* transform16, int32_t is_dense, int32_t* total) {
  if (!h || (!xyzw && n > 0) || n < 0) return fail(h, PCOP_ERR_BAD_PARAM, "pcop_accumulate: bad argument");
  if ((long long)h->acc_count + n > h->cap) return fail(h, PCOP_ERR_CAPACITY, "accumulated cloud exceeds max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (n > 0) {
    TRY(transform_into(h, xyzw, n, transform16, is_dense, h->d_acc + h->acc_count));
    if (!is_device_pointer(xyzw)) PCOP_CUDA_TRY(cudaStreamSynchronize(h->lanes[0]->stream));  // the caller may reuse its buffer
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
  Lane* l = h->lanes[0].get();
  TRY(transform_into(h, xyzw, n, transform16, is_dense, l->d_crop));
  TRY(download(h, out_xyzw, l->d_crop, (size_t)n * 16));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
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
  Lane* l = h->lanes[0].get();
  TRY(pc2_ingest(h, data, n_points, point_step, off_x, off_y, off_z, nullptr, 1, l->d_crop));
  TRY(download(h, out_xyzw, l->d_crop, (size_t)n_points * 16));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  return PCOP_OK;
}

int pcop_cloud_to_pointcloud2(pcop_handle* h, const float* xyzw, int32_t n, int32_t point_step, int32_t off_x, int32_t off_y,
                              int32_t off_z, unsigned char* out_data) {
  if (!h || n < 0 || (n > 0 && (!xyzw || !out_data))) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (point_step < 12 || !pc2_layout_ok(point_step, off_x, off_y, off_z))
    return fail(h, PCOP_ERR_BAD_PARAM, "PointCloud2 field offsets do not fit point_step");
  if (n > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return PCOP_OK;
  Lane* l = h->lanes[0].get();
  const float4* src;
  TRY(device_cloud(h, xyzw, n, &src));
  const size_t bytes = (size_t)n * (size_t)point_step;
  unsigned char* dst = out_data;
  const bool out_on_device = is_device_pointer(out_data);
  if (!out_on_device) {  // staged through the raw-payload buffer of the ingest path
    TRY(ensure_raw(l, bytes));
    dst = l->d_raw;
  }
  Ctx c = make_ctx(l, 1, n);
  KL(c, "k_pc2_egress", k_pc2_egress<<<cdiv(n, 256), 256, 0, l->stream>>>(src, n, point_step, off_x, off_y, off_z, dst));
  count_launch(c);
  PCOP_CUDA_TRY(cudaGetLastError());
  if (!out_on_device) TRY(download(h, out_data, dst, bytes));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  return PCOP_OK;
}

int pcop_occupancy_dims(const pcop_handle* h, int32_t* width, int32_t* height) {
  if (!h || !width || !height || !(h->params.block_size > 0.0f)) return PCOP_ERR_BAD_PARAM;
  const pcop_params& p = h->params;  // od.cpp:958-959 (double: the unqualified fabs is ::fabs(double))
  *width = (int32_t)std::ceil((std::fabs((double)p.y_min) + std::fabs((double)p.y_max)) / (double)p.block_size);
  *height = (int32_t)std::ceil((std::fabs((double)p.x_min) + std::fabs((double)p.x_max)) / (double)p.block_size);
  return PCOP_OK;
}

int pcop_occupancy_grid(pcop_handle* h, const float* xyzw, int32_t n, int8_t* grid_data, int64_t* counts, int64_t* row_avg) {
  if (!h || !grid_data || n < 0) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  OccGrid g;
  TRY(occ_grid_of(h, &g));
  const int32_t H = g.H;
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  Lane* l = h->lanes[0].get();
  const float4* src;
  if (!xyzw) {  // the accumulated cloud
    src = h->d_acc;
    n = h->acc_count;
  } else {
    if (n > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
    TRY(device_cloud(h, xyzw, n, &src));
  }
  const size_t cells = (size_t)g.cells;
  const size_t need = cells * 8 + (size_t)H * 8 + cells;
  if (need > h->occ_cap) {
    PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
    if (h->d_occ) cudaFree(h->d_occ);
    h->d_occ = nullptr;
    h->occ_cap = 0;
    PCOP_CUDA_TRY(cudaMalloc((void**)&h->d_occ, need + 256));
    h->occ_cap = need;
  }
  unsigned long long* d_counts = reinterpret_cast<unsigned long long*>(h->d_occ);
  long long* d_avg = reinterpret_cast<long long*>(h->d_occ + cells * 8);
  signed char* d_grid = reinterpret_cast<signed char*>(h->d_occ + cells * 8 + (size_t)H * 8);
  Ctx c = make_ctx(l, 1, n);
  PCOP_CUDA_TRY(cudaMemsetAsync(d_counts, 0, cells * 8, l->stream));
  run_occ_count(c, src, n, g, d_counts);
  run_occ_finish(c, d_counts, g, d_avg, d_grid);
  TRY(download(h, grid_data, d_grid, cells));
  TRY(download(h, counts, d_counts, cells * 8));
  TRY(download(h, row_avg, d_avg, (size_t)H * 8));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  return PCOP_OK;
}

// Shadow casting + obstacle marking (od.cpp:467-672, 817-833) on a grid produced by pcop_occupancy_grid
int pcop_occupancy_shadows(pcop_handle* h, const float* remaining_xyzw, int32_t n_remaining, const int32_t* cluster_offsets,
                           const int32_t* cluster_indices, int32_t n_clusters, const float* world_to_sensor16,
                           const float* sensor_to_world16, int8_t* grid_data, int32_t* shadow_records, uint32_t* warnings) {
  if (!h || !grid_data || n_remaining < 0 || n_clusters < 0 || (n_remaining > 0 && !remaining_xyzw) ||
      (n_clusters > 0 && (!cluster_offsets || !cluster_indices || !world_to_sensor16 || !sensor_to_world16)))
    return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  OccGrid g;
  TRY(occ_grid_of(h, &g));
  if (n_remaining > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cloud has more points than max_points");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  Lane* l = h->lanes[0].get();
  const size_t cells = (size_t)g.cells;
  // the member list's length is the last CSR offset
  int32_t L = 0;
  if (n_clusters > 0) {
    if (is_device_pointer(cluster_offsets)) {
      PCOP_CUDA_TRY(cudaMemcpyAsync(&L, cluster_offsets + n_clusters, sizeof(int32_t), cudaMemcpyDeviceToHost, l->stream));
      PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
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
    PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
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
  TRY(device_cloud(h, remaining_xyzw, n_remaining, &a.cloud));
  a.offsets = cluster_offsets;
  a.indices = cluster_indices;
  if (n_clusters > 0 && !is_device_pointer(cluster_offsets)) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(d_off, cluster_offsets, ((size_t)n_clusters + 1) * 4, cudaMemcpyHostToDevice, l->stream));
    a.offsets = d_off;
  }
  if (n_clusters > 0 && L > 0 && !is_device_pointer(cluster_indices)) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(d_idx, cluster_indices, (size_t)L * 4, cudaMemcpyHostToDevice, l->stream));
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
  PCOP_CUDA_TRY(cudaMemcpyAsync(d_sizes, &up, sizeof(up), cudaMemcpyHostToDevice, l->stream));  // (pageable: staged before return)
  a.n_points = d_sizes;
  a.n_clusters = d_sizes + 1;
  a.mats = d_mats;
  const pcop_params& p = h->params;
  a.y_min = p.y_min;
  a.x_max = p.x_max;
  a.block_size = p.block_size;
  a.W = g.W;
  a.size = g.cells;
  a.opacity = p.grid_opacity;
  const bool grid_on_device = is_device_pointer(grid_data);
  a.grid = reinterpret_cast<signed char*>(grid_data);
  if (!grid_on_device) {
    PCOP_CUDA_TRY(cudaMemcpyAsync(h->d_shadow, grid_data, cells, cudaMemcpyHostToDevice, l->stream));
    a.grid = reinterpret_cast<signed char*>(h->d_shadow);
  }
  a.records = shadow_records ? d_rec : nullptr;
  a.warnings = d_warn;
  PCOP_CUDA_TRY(cudaMemsetAsync(d_warn, 0, sizeof(uint32_t), l->stream));
  Ctx c = make_ctx(l, 1, n_remaining);
  pcop::run_occ_shadows(c, a, n_clusters, n_remaining);
  PCOP_CUDA_TRY(cudaGetLastError());
  if (!grid_on_device) TRY(download(h, grid_data, a.grid, cells));
  if (shadow_records && n_clusters > 0) {
    if (is_device_pointer(shadow_records))
      PCOP_CUDA_TRY(cudaMemcpyAsync(shadow_records, d_rec, 6 * (size_t)n_clusters * 4, cudaMemcpyDeviceToDevice, l->stream));
    else
      TRY(download(h, shadow_records, d_rec, 6 * (size_t)n_clusters * 4));
  }
  uint32_t wv = 0;
  PCOP_CUDA_TRY(cudaMemcpyAsync(&wv, d_warn, sizeof(uint32_t), cudaMemcpyDeviceToHost, l->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  if (warnings) *warnings = wv;
  return PCOP_OK;
}

// ---- stage-isolated entry points -------------------------------------------------------
int pcop_crop(pcop_handle* h, const float* xyzw, int32_t n, float* out_xyzw, int32_t* kept_idx, int32_t* m) {
  if (!h || !xyzw || !m) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  TRY(upload_single(h, xyzw, n, CNT_IN));
  Lane* l = h->lanes[0].get();
  Ctx c = make_ctx(l, 1, n);
  run_crop(c, make_crop_args(l, l->d_in, h->cap, l->cnt(CNT_IN)));
  TRY(fetch_word(h, l->cnt(CNT_CROP), m));
  TRY(download(h, out_xyzw, l->d_crop, (size_t)*m * 16));
  TRY(download(h, kept_idx, l->d_crop_kept, (size_t)*m * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  return PCOP_OK;
}

int pcop_voxel(pcop_handle* h, const float* xyzw, int32_t m, float* out_xyzw, uint32_t* out_keys, int32_t* v,
               uint32_t* warnings) {
  if (!h || !xyzw || !v) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (!(h->params.downsample_size > 0.0f)) return fail(h, PCOP_ERR_BAD_PARAM, "downsample_size must be > 0");
  TRY(upload_single(h, xyzw, m, CNT_CROP));
  Lane* l = h->lanes[0].get();
  Ctx c = make_ctx(l, 1, m);
  run_minmax(c, l->d_in, h->cap, l->cnt(CNT_CROP), l->d_minmax);
  run_voxel(c, make_voxel_args(l, l->d_in, h->cap, l->cnt(CNT_CROP)));
  TRY(fetch_word(h, l->cnt(CNT_VOX), v));
  TRY(fetch_word(h, l->d_warnings, warnings));
  TRY(download(h, out_xyzw, l->d_vox, (size_t)*v * 16));
  TRY(download(h, out_keys, l->d_vox_keys, (size_t)*v * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  return PCOP_OK;
}

int pcop_sor(pcop_handle* h, const float* xyzw, int32_t v, float* out_xyzw, int32_t* kept_idx, int32_t* s,
             uint32_t* warnings) {
  if (!h || !xyzw || !s) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (h->params.statistical_outlier_meanK < 1 || h->params.statistical_outlier_meanK > 63)
    return fail(h, PCOP_ERR_BAD_PARAM, "statistical_outlier_meanK must be in [1, 63]");
  TRY(upload_single(h, xyzw, v, CNT_VOX));
  Lane* l = h->lanes[0].get();
  Ctx c = make_ctx(l, 1, v);
  run_sor(c, make_sor_args(l, l->d_in, h->cap, l->cnt(CNT_VOX)));
  TRY(fetch_word(h, l->cnt(CNT_SOR), s));
  TRY(fetch_word(h, l->d_warnings, warnings));
  TRY(download(h, out_xyzw, l->d_sor, (size_t)*s * 16));
  TRY(download(h, kept_idx, l->d_sor_kept, (size_t)*s * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  return PCOP_OK;
}

int pcop_plane(pcop_handle* h, const float* xyzw, int32_t s, float* remaining_xyzw, int32_t* remaining_src_idx,
               int32_t* p, int32_t* n_passes, int32_t* pass_points, int32_t* pass_inliers, float* pass_coeff,
               float* last_coeff, int32_t* inlier_idx, int32_t* n_inliers, uint32_t* warnings) {
  if (!h || !xyzw || !p) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  TRY(upload_single(h, xyzw, s, CNT_SOR));
  Lane* l = h->lanes[0].get();
  Ctx c = make_ctx(l, 1, s);
  PlaneArgs a = make_plane_args(l, l->d_in, h->cap, l->cnt(CNT_SOR));
  a.large_tier = 1;
  cudaError_t e = run_plane(c, a);
  if (e != cudaSuccess) return fail_cuda(h, e, "run_plane", __FILE__, __LINE__);
  KL(c, "k_plane_record", k_plane_record<<<1, 32, 0, l->stream>>>(l->d_pf, l->d_prec, l->cnt(CNT_NINL), l->cnt(CNT_CLUS), l->cnt(CNT_CLUS1), 1, 1));
  TRY(fetch_word(h, l->cnt(CNT_REM), p));
  TRY(fetch_word(h, l->d_warnings, warnings));
  PCOP_CUDA_TRY(cudaMemcpyAsync(l->h_prec, l->d_prec, sizeof(PlaneRecord), cudaMemcpyDeviceToHost, l->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  const PlaneRecord& r = l->h_prec[0];
  if (n_passes) *n_passes = r.n_passes;
  if (pass_points) memcpy(pass_points, r.pass_points, sizeof(r.pass_points));
  if (pass_inliers) memcpy(pass_inliers, r.pass_inliers, sizeof(r.pass_inliers));
  if (pass_coeff) memcpy(pass_coeff, r.pass_coeff, sizeof(r.pass_coeff));
  if (last_coeff) memcpy(last_coeff, &r.coeff, 16);
  if (n_inliers) *n_inliers = r.n_inliers_last;
  TRY(download(h, remaining_xyzw, l->d_rem, (size_t)*p * 16));
  TRY(download(h, remaining_src_idx, l->d_rem_src, (size_t)*p * 4));
  TRY(download(h, inlier_idx, l->d_inliers, (size_t)r.n_inliers_last * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  return PCOP_OK;
}

int pcop_cluster(pcop_handle* h, const float* xyzw, int32_t p, int32_t* cluster_offsets, int32_t* cluster_indices,
                 int32_t* c_out, int32_t* l_out) {
  if (!h || !xyzw || !c_out || !l_out) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (!(h->params.euc_cluster_tolerance > 0.0f)) return fail(h, PCOP_ERR_BAD_PARAM, "euc_cluster_tolerance must be > 0");
  TRY(upload_single(h, xyzw, p, CNT_REM));
  Lane* l = h->lanes[0].get();
  Ctx c = make_ctx(l, 1, p);
  run_cluster(c, make_cluster_args(l, l->d_in, h->cap, l->cnt(CNT_REM)), /*with_generic=*/true);
  TRY(fetch_word(h, l->cnt(CNT_CLUS), c_out));
  TRY(fetch_word(h, l->cnt(CNT_CLPTS), l_out));
  TRY(download(h, cluster_offsets, l->d_offsets, (size_t)(*c_out + 1) * 4));
  TRY(download(h, cluster_indices, l->d_indices, (size_t)*l_out * 4));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  return PCOP_OK;
}

int pcop_centroid_radius(pcop_handle* h, const float* xyzw, int32_t p, const int32_t* cluster_offsets,
                         const int32_t* cluster_indices, int32_t c_in, float* obstacles) {
  if (!h || !xyzw || !cluster_offsets || !cluster_indices || !obstacles || c_in < 0)
    return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  if (c_in > h->cap) return fail(h, PCOP_ERR_CAPACITY, "too many clusters");
  TRY(upload_single(h, xyzw, p, CNT_REM));
  Lane* l = h->lanes[0].get();
  const int len = cluster_offsets[c_in];
  if (len < 0 || len > h->cap) return fail(h, PCOP_ERR_CAPACITY, "cluster index list longer than max_points");
  l->h_n_in[1] = c_in;
  PCOP_CUDA_TRY(cudaMemcpyAsync(l->cnt(CNT_CLUS), l->h_n_in + 1, sizeof(int), cudaMemcpyHostToDevice, l->stream));
  PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_offsets, cluster_offsets, (size_t)(c_in + 1) * 4, cudaMemcpyDefault, l->stream));
  if (len > 0) PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_indices, cluster_indices, (size_t)len * 4, cudaMemcpyDefault, l->stream));
  Ctx c = make_ctx(l, 1, p);
  run_centroid_radius(c, make_cluster_args(l, l->d_in, h->cap, l->cnt(CNT_REM)));
  TRY(download(h, obstacles, l->d_obst, (size_t)c_in * 16));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  return PCOP_OK;
}

}  // extern "C"
