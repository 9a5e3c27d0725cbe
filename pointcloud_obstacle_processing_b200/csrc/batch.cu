// Wave scheduler of the batched calls, and the kernels it owns: input decode, result packing, metadata out.
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
#include <chrono>
#include <cstdio>

#include "handle.cuh"
#include "primitives.cuh"

using namespace pcop;

namespace {

// ---- small kernels owned by the wave scheduler -----------------------------------------
__global__ void k_copy_counts(const int* __restrict__ src, int* __restrict__ dst, int B) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < B) dst[f] = src[f];
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
// the decoded point of one record (PCL's transform coefficients in float, no FMA)
__device__ __forceinline__ float4 pc2_point(const Pc2Frame& d, float x, float y, float z) {
  float4 o = make_float4(x, y, z, 1.0f);
  const bool finite = fabsf(x) <= 3.402823466e+38f && fabsf(y) <= 3.402823466e+38f && fabsf(z) <= 3.402823466e+38f;
  if (d.apply_transform && (d.is_dense || finite)) {
    const Mat34& t = d.t;
    o.x = fadd(fadd(fadd(fmul(t.m[0], x), fmul(t.m[1], y)), fmul(t.m[2], z)), t.m[3]);
    o.y = fadd(fadd(fadd(fmul(t.m[4], x), fmul(t.m[5], y)), fmul(t.m[6], z)), t.m[7]);
    o.z = fadd(fadd(fadd(fmul(t.m[8], x), fmul(t.m[9], y)), fmul(t.m[10], z)), t.m[11]);
  }
  return o;
}
// Every decode of the library (pcop_accumulate_pointcloud2 / pcop_pointcloud2_to_xyz: one message; the batched
// PointCloud2 wave: every message of its windows).  A 1-D grid over record tiles of PC2_TILE records: message m owns
// tiles tile0 .. tile0 + cdiv(n, PC2_TILE) - 1 (empty messages own none), so a block finds its message by a binary
// search over tile0, and a tile never spans two messages.  Record i of message m goes to out[dst + i].  aligned = 1
// (point_step % 16 == 0, 16-byte aligned base, x / y / z inside one aligned 16-byte word of the record): one 16-byte
// load per record instead of three 4-byte (or twelve 1-byte) loads; a thread issues the loads of its PC2_ITEMS records
// before it stores.
__global__ void __launch_bounds__(PC2_THREADS)
    k_pc2_ingest(const Pc2Frame* __restrict__ msgs, int n_msgs, float4* __restrict__ out) {
  const int tile = blockIdx.x;
  int lo = 0, hi = n_msgs - 1;  // the last message whose first tile is <= tile
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (msgs[mid].tile0 <= tile) lo = mid;
    else hi = mid - 1;
  }
  const Pc2Frame& d = msgs[lo];
  const int base = (tile - d.tile0) * PC2_TILE;
  const int n = d.n - base;  // (> 0)
  const unsigned char* rec0 = d.data + (size_t)base * (size_t)d.point_step;
  float4* o = out + d.dst + base;
  if (d.aligned) {
    const int word = d.off_x & ~15, kx = (d.off_x & 15) >> 2, ky = (d.off_y & 15) >> 2, kz = (d.off_z & 15) >> 2;
    float4 v[PC2_ITEMS];
#pragma unroll
    for (int k = 0; k < PC2_ITEMS; ++k) {
      const int i = k * PC2_THREADS + threadIdx.x;
      if (i < n) v[k] = __ldg(reinterpret_cast<const float4*>(rec0 + (size_t)i * (size_t)d.point_step + word));
    }
#pragma unroll
    for (int k = 0; k < PC2_ITEMS; ++k) {
      const int i = k * PC2_THREADS + threadIdx.x;
      if (i < n) o[i] = pc2_point(d, pc2_lane(v[k], kx), pc2_lane(v[k], ky), pc2_lane(v[k], kz));
    }
  } else {
#pragma unroll
    for (int k = 0; k < PC2_ITEMS; ++k) {
      const int i = k * PC2_THREADS + threadIdx.x;
      if (i < n) {
        const unsigned char* rec = rec0 + (size_t)i * (size_t)d.point_step;
        o[i] = pc2_point(d, pc2_load_f32(rec + d.off_x), pc2_load_f32(rec + d.off_y), pc2_load_f32(rec + d.off_z));
      }
    }
  }
}

// the descriptor of one message whose payload sits at `src` on the device (validated by the caller); its place in the
// launch (dst, tile0) is set by the caller
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
  Lane* l;
  int stage;
  StageTimer(Lane* ll, int s) : l(ll), stage(s) {
    cudaEventRecord(l->ev_stage[s][0], l->stream);
    l->stage_used[s] = true;
  }
  ~StageTimer() { cudaEventRecord(l->ev_stage[stage][1], l->stream); }
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

int ensure_host_pack(Lane* l, size_t need) {
  if (need <= l->h_pack_cap) return PCOP_OK;
  size_t ncap = std::max<size_t>(need, l->h_pack_cap * 2);
  ncap = std::max<size_t>(ncap, 1 << 20);
  unsigned char* q = nullptr;
  cudaError_t e = cudaHostAlloc((void**)&q, ncap, cudaHostAllocMapped);
  if (e != cudaSuccess) return fail_cuda(l->h, e, "cudaHostAlloc(pack)", __FILE__, __LINE__);
  if (l->cstream) cudaStreamSynchronize(l->cstream);  // copies into the old buffer must have landed
  if (l->h_pack) {
    memcpy(q, l->h_pack, l->h_pack_cap);
    cudaFreeHost(l->h_pack);
  }
  l->h_pack = q;
  l->h_pack_cap = ncap;
  l->h_pack_buf[l->h_pack_sel] = q;
  l->h_pack_buf_cap[l->h_pack_sel] = ncap;
  return PCOP_OK;
}

// The first route of a wave whose largest frame has max_n points, from the handle's plan and knobs and the lane's
// history: the LSD voxel path while a partition-path decline is recent, a reduce grid sized by the frames seen lately,
// and the plane tiers and clustering kernels the last waves needed.
WaveRoute next_route(const Lane* l, int max_n) {
  const pcop_handle* h = l->h;
  WaveRoute r;
  if (h->vplan.part_ok && l->vox_lsd_waves <= 0) {
    r.vox = WaveRoute::VOX_PARTITION;
    r.vox_groups = std::min(l->vp_group_hint, vox_part_group_bound(h->vplan, max_n));
  } else if (h->vplan.ok) {
    r.vox = WaveRoute::VOX_LSD;
  }
  r.plane_large = l->expect_large_plane;
  r.cluster_generic = l->expect_big_remaining || h->ece_small_max <= 0;  // (no fused kernel at all: run_cluster)
  return r;
}

// The plane loop of one wave on the stage input recorded in the lane.  Tiers: see run_plane.
int run_wave_plane(Lane* l, int B, int max_n, const WaveRoute& r) {
  const pcop_params& p = l->h->params;
  Ctx c = make_ctx(l, B, max_n);  // (no frame holds more points than the largest input frame)
  StageTimer t(l, PCOP_STAGE_PLANE);
  if (p.enable_plane) {
    PlaneArgs a = make_plane_args(l, l->plane_in, l->plane_stride, l->plane_n);
    a.n_in_copy = p.enable_sor ? nullptr : l->cnt(CNT_SOR);
    a.large_tier = r.plane_large;
    if (!(effective_outputs(p) & PCOP_OUT_PLANE)) a.inlier_idx = nullptr;  // the inlier list is only written on request
    cudaError_t e = run_plane(c, a);
    if (e != cudaSuccess) return fail_cuda(l->h, e, "run_plane", __FILE__, __LINE__);
  } else {
    KL(c, "k_copy_counts", k_copy_counts<<<cdiv(B, 256), 256, 0, l->stream>>>(l->plane_n, l->cnt(CNT_REM), B));
    KL(c, "k_copy_cloud", k_copy_cloud<<<dim3(cdiv(c.grid_cap, CT_TILE), B), CT_THREADS, 0, l->stream>>>(
                              l->plane_in, l->plane_stride, l->plane_n, l->d_rem, l->d_rem_src, l->h->cap));
    count_launch(c, 2);
  }
  return PCOP_OK;
}

// All stages of one wave up to the plane loop.  `in`/`stride` already on the device; counts row CNT_IN already set.
int run_wave_stages(Lane* l, int B, const float4* in, size_t stride, int max_n, const WaveRoute& r) {
  pcop_handle* h = l->h;
  const pcop_params& p = h->params;
  Ctx c = make_ctx(l, B, max_n);  // no stage ever holds more points per frame than the largest input frame
  if (r.vox == WaveRoute::VOX_GENERIC || (effective_outputs(p) & PCOP_OUT_CROP)) {  // (the fused voxel path zeroes the warnings itself)
    KL(c, "k_zero_u32", k_zero_u32<<<cdiv(B, 256), 256, 0, l->stream>>>(l->d_warnings, B));
    count_launch(c);
  }

  const float4* cur = in;
  size_t cur_stride = stride;
  const int* cur_n = l->cnt(CNT_IN);
  bool have_minmax = false;

  if (r.vox == WaveRoute::VOX_PARTITION) {
    {
      StageTimer t(l, PCOP_STAGE_CROP);
      if (effective_outputs(p) & PCOP_OUT_CROP) run_crop(c, make_crop_args(l, cur, cur_stride, cur_n));
    }
    StageTimer t(l, PCOP_STAGE_VOXEL);
    VoxelPartArgs a{};
    a.in = cur;
    a.in_stride = cur_stride;
    a.n_in = cur_n;
    a.plan = h->vplan;
    a.leaf = p.downsample_size;
    a.minmax = l->d_minmax;
    a.vf = l->d_vf;
    a.ghist = l->d_vp_hist;
    a.chunk_start = l->d_vp_bstart;
    a.ne_bucket = l->d_vp_ne;
    a.ne_start = l->d_vp_nstart;
    a.grec = l->d_vp_grec;
    a.n_groups = l->cnt(CNT_GROUPS);
    a.part = l->d_sorted;  // (the search-grid point list of SOR / clustering is not live yet)
    a.desc = l->d_vp_desc;
    a.group_stride = l->vp_gstride;
    a.group_launch = r.vox_groups;
    a.flags = l->d_vf_flags;
    a.warnings = (effective_outputs(p) & PCOP_OUT_CROP) ? nullptr : l->d_warnings;  // zeroed by k_vp_init
    a.n_crop = l->cnt(CNT_CROP);
    a.out = l->d_vox;
    a.out_keys = l->d_vox_keys;
    a.n_out = l->cnt(CNT_VOX);
    a.want_keys = (effective_outputs(p) & PCOP_OUT_VOXEL) ? 1 : 0;
    run_voxel_part(c, a);
    cur = l->d_vox;
    cur_stride = h->cap;
    cur_n = l->cnt(CNT_VOX);
  } else if (r.vox == WaveRoute::VOX_LSD) {
    // crop + VoxelGrid in one pass over the input (stage_voxel_fused.cu); the cropped cloud itself is only
    // materialised when it is a requested output
    {
      StageTimer t(l, PCOP_STAGE_CROP);
      if (effective_outputs(p) & PCOP_OUT_CROP) run_crop(c, make_crop_args(l, cur, cur_stride, cur_n));
    }
    StageTimer t(l, PCOP_STAGE_VOXEL);
    VoxelFusedArgs a{};
    a.in = cur;
    a.in_stride = cur_stride;
    a.n_in = cur_n;
    a.plan = h->vplan;
    a.leaf = p.downsample_size;
    a.minmax = l->d_minmax;
    a.vf = l->d_vf;
    a.sort = l->sort;
    a.pair[0] = l->d_vf_pair[0];
    a.pair[1] = l->d_vf_pair[1];
    a.desc = l->d_desc;
    a.flags = l->d_vf_flags;
    a.warnings = (effective_outputs(p) & PCOP_OUT_CROP) ? nullptr : l->d_warnings;  // zeroed by k_vf_init
    a.n_crop = l->cnt(CNT_CROP);
    a.out = l->d_vox;
    a.out_keys = l->d_vox_keys;
    a.n_out = l->cnt(CNT_VOX);
    a.want_keys = (effective_outputs(p) & PCOP_OUT_VOXEL) ? 1 : 0;
    run_voxel_fused(c, a);
    cur = l->d_vox;
    cur_stride = h->cap;
    cur_n = l->cnt(CNT_VOX);
  } else {
    {
      StageTimer t(l, PCOP_STAGE_CROP);
      if (p.enable_crop) {
        run_crop(c, make_crop_args(l, cur, cur_stride, cur_n));
        cur = l->d_crop;
        cur_stride = h->cap;
        cur_n = l->cnt(CNT_CROP);
        have_minmax = true;
      } else {
        KL(c, "k_copy_counts", k_copy_counts<<<cdiv(B, 256), 256, 0, l->stream>>>(cur_n, l->cnt(CNT_CROP), B));
        count_launch(c);
      }
    }
    {
      StageTimer t(l, PCOP_STAGE_VOXEL);
      if (p.enable_voxel) {
        if (!have_minmax) run_minmax(c, cur, cur_stride, cur_n, l->d_minmax);
        run_voxel(c, make_voxel_args(l, cur, cur_stride, cur_n));
        cur = l->d_vox;
        cur_stride = h->cap;
        cur_n = l->cnt(CNT_VOX);
      } else {
        KL(c, "k_copy_counts", k_copy_counts<<<cdiv(B, 256), 256, 0, l->stream>>>(cur_n, l->cnt(CNT_VOX), B));
        count_launch(c);
      }
    }
  }
  {
    StageTimer t(l, PCOP_STAGE_SOR);
    if (p.enable_sor) {
      run_sor(c, make_sor_args(l, cur, cur_stride, cur_n));
      cur = l->d_sor;
      cur_stride = h->cap;
      cur_n = l->cnt(CNT_SOR);
    } else if (!p.enable_plane) {  // (with the plane stage on, its init kernel copies the count row)
      KL(c, "k_copy_counts", k_copy_counts<<<cdiv(B, 256), 256, 0, l->stream>>>(cur_n, l->cnt(CNT_SOR), B));
      count_launch(c);
    }
  }
  l->plane_in = cur;
  l->plane_stride = cur_stride;
  l->plane_n = cur_n;
  TRY(run_wave_plane(l, B, max_n, r));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail_cuda(h, e, "stage launches", __FILE__, __LINE__);
  return PCOP_OK;
}

// Clustering + centroid / radius of one wave.  The host does not know the remaining-cloud sizes yet; without
// r.cluster_generic only the fused small-cloud kernel runs (settle_wave repeats the stage with the generic kernels if a
// frame turned out larger, see run_cluster).
int run_wave_cluster(Lane* l, int B, int max_n, const WaveRoute& r) {
  pcop_handle* h = l->h;
  const pcop_params& p = h->params;
  Ctx c = make_ctx(l, B, max_n);
  ClusterArgs ca = make_cluster_args(l, l->d_rem, h->cap, l->cnt(CNT_REM));
  bool generic_centroid = false;
  {
    StageTimer t(l, PCOP_STAGE_CLUSTER);
    if (p.enable_cluster) {
      generic_centroid = run_cluster(c, ca, r.cluster_generic);  // the fused small-cloud kernel writes the obstacles itself
    } else {
      cudaMemsetAsync(l->cnt(CNT_CLUS), 0, sizeof(int) * B, l->stream);
      cudaMemsetAsync(l->cnt(CNT_CLPTS), 0, sizeof(int) * B, l->stream);
    }
  }
  {
    StageTimer t(l, PCOP_STAGE_CENTROID);
    if (p.enable_cluster && generic_centroid) run_centroid_radius(c, ca);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail_cuda(h, e, "stage launches", __FILE__, __LINE__);
  return PCOP_OK;
}

size_t pc2_payload_bytes(const pcop_pointcloud2_frame& m) { return (size_t)m.n_points * (size_t)m.point_step; }

// PointCloud2 wave, input half: the descriptors of every message of the wave's windows go up through the pinned staging
// (the lane's previous wave no longer reads it), every host payload into the lane's raw staging at a 256-byte aligned
// offset, device payloads are read in place; one k_pc2_ingest launch decodes (and transforms) every message into its
// frame's slot of d_in, after the messages before it in its window.  A repeat of the wave (voxel decline) decodes again
// from the same staging -- the plane stage has overwritten d_in, the staging is intact.
int enqueue_wave_decode(Lane* l, const Pc2Call& pc, int w0, int B, int max_n, bool repeat) {
  pcop_handle* h = l->h;
  if (!repeat) {
    const int m0 = pc.window_first[w0];
    size_t off = 0;
    int tiles = 0;
    for (int f = 0; f < B; ++f) {
      size_t dst = (size_t)f * (size_t)h->cap;
      for (int k = pc.window_first[w0 + f]; k < pc.window_first[w0 + f + 1]; ++k) {
        const pcop_pointcloud2_frame& m = pc.msgs[k];
        const size_t bytes = pc2_payload_bytes(m);
        const unsigned char* src = m.data;
        if (bytes > 0 && !pc.on_device[k]) {
          PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_raw + off, m.data, bytes, cudaMemcpyHostToDevice, l->stream));
          src = l->d_raw + off;
          off += (bytes + 255) & ~(size_t)255;
        }
        Pc2Frame& d = l->h_pc2[k - m0];
        d = make_pc2_frame(src, m.n_points, m.point_step, m.off_x, m.off_y, m.off_z,
                           pc.transform16 ? pc.transform16 + (size_t)k * 16 : nullptr, m.is_dense);
        d.dst = dst;
        d.tile0 = tiles;
        dst += (size_t)m.n_points;
        tiles += cdiv(m.n_points, PC2_TILE);
      }
    }
    l->pc2_msgs = pc.window_first[w0 + B] - m0;
    l->pc2_tiles = tiles;
    if (l->pc2_msgs > 0)
      PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_pc2, l->h_pc2, sizeof(Pc2Frame) * l->pc2_msgs, cudaMemcpyHostToDevice, l->stream));
  }
  if (l->pc2_tiles > 0) {  // (a wave of empty windows decodes nothing)
    Ctx c = make_ctx(l, B, max_n);
    KL(c, "k_pc2_ingest", k_pc2_ingest<<<l->pc2_tiles, PC2_THREADS, 0, l->stream>>>(l->d_pc2, l->pc2_msgs, l->d_in));
    count_launch(c);
  }
  return PCOP_OK;
}

// Second half of a wave: clustering, result packing, and the copy of the wave's counts / plane records / pack sizes
// into pinned memory, followed by ev_meta.
int enqueue_wave_pack(Lane* l, int B, int max_n, uint32_t mask, const WaveRoute& r) {
  pcop_handle* h = l->h;
  // pack the requested outputs of all frames of the wave
  Ctx c = make_ctx(l, B, max_n);
  StageTimer t(l, PCOP_STAGE_D2H);
  const bool dev_results = (mask & PCOP_OUT_DEVICE) != 0;  // the arrays stay in d_pack (bump-allocated over the call)
  if (!dev_results && l->wave_seq >= 1) PCOP_CUDA_TRY(cudaStreamWaitEvent(l->stream, l->ev_copied, 0));  // d_pack is free again
  KL(c, "k_pack_scan", k_pack_scan<<<1, 320, 0, l->stream>>>(l->d_counts, h->maxB, B, mask, l->d_pack_off, l->d_meta, l->d_pf, l->d_prec,
                                             h->params.enable_plane ? 1 : 0, dev_results ? l->d_pack_cursor : nullptr,
                                             (unsigned long long)l->pack_cap));
  count_launch(c);
  const void* srcs[PK_N] = {l->d_crop_kept, l->d_vox_keys, l->d_vox,     l->d_sor_kept, l->d_inliers,
                            l->d_rem,       l->d_rem_src,  l->d_offsets, l->d_indices,  l->d_obst};
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
    seg(l->d_counts, l->h_counts, sizeof(int) * CNT_ROWS * h->maxB);
    seg(l->d_warnings, l->h_warnings, sizeof(uint32_t) * B);
    seg(l->d_prec, l->h_prec, sizeof(PlaneRecord) * B);
    seg(l->d_meta, l->h_meta, sizeof(PackMeta));
    if (r.vox != WaveRoute::VOX_GENERIC) seg(l->d_vf_flags, l->h_vf_flags, sizeof(uint32_t) * B);
    static_assert(PK_N >= 5, "one pack block per metadata segment");
    if (any) {  // the (frame < 4, array k < 5) blocks of the pack kernel also carry metadata segment k out
      // (parts per (frame, array): 16 for the batched waves; a call of a few large frames gets enough to fill the GPU)
      const int gx = std::max(1, std::min(cdiv(c.grid_cap, 256 * 4), std::max(16, 592 / B)));
      m.frames = std::min(B, 4);
      KL(c, "k_pack", k_pack<<<dim3(gx, B, PK_N), 256, 0, l->stream>>>(ps, l->d_counts, h->maxB, l->d_pack_off, l->d_meta, l->d_pack, m));
      count_launch(c);
    } else {
      KL(c, "k_meta_out", k_meta_out<<<dim3(4, nseg), 256, 0, l->stream>>>(m));
      count_launch(c);
    }
  }
  if (h->trace) {
    if (l->trace_used == l->trace_recs.size()) {
      Lane::TraceRec r{};
      cudaEventCreate(&r.meta);
      cudaEventCreate(&r.c0);
      cudaEventCreate(&r.c1);
      l->trace_recs.push_back(r);
    }
    cudaEventRecord(l->trace_recs[l->trace_used].meta, l->stream);
  }
  PCOP_CUDA_TRY(cudaEventRecord(l->ev_meta, l->stream));
  return PCOP_OK;
}

// Grid product, first half: the wave's poses (from the pinned staging, which the lane's previous wave no longer
// reads) and the per-cell counts of every frame.  Runs before the plane stage, whose second ping-pong cloud is d_in.
int enqueue_wave_counts(Lane* l, const OccCall& oc, int w0, int B, const float4* in, size_t stride, int max_n) {
  pcop_handle* h = l->h;
  for (int f = 0; f < B; ++f) {
    memcpy(l->h_occ_mats[2 * f].m, oc.world_to_sensor16 + (size_t)(w0 + f) * 16, sizeof(Mat34));
    memcpy(l->h_occ_mats[2 * f + 1].m, oc.sensor_to_world16 + (size_t)(w0 + f) * 16, sizeof(Mat34));
  }
  PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_occ_mats, l->h_occ_mats, sizeof(Mat34) * 2 * B, cudaMemcpyHostToDevice, l->stream));
  PCOP_CUDA_TRY(cudaMemsetAsync(l->d_occ_counts, 0, sizeof(int) * (size_t)B * (size_t)oc.g.cells, l->stream));
  Ctx c = make_ctx(l, B, max_n);
  const cudaError_t e = run_occ_count_wave(c, in, stride, l->cnt(CNT_IN), oc.g, l->d_occ_counts);
  if (e != cudaSuccess) return fail_cuda(h, e, "run_occ_count_wave (shared-memory opt-in or launch)", __FILE__, __LINE__);
  return PCOP_OK;
}

// Grid product, second half (after clustering): threshold, shadows, obstacle marks.  Every repeat of the wave's back
// half rebuilds the grids from the counts, so the last repeat leaves exactly what one pass over the final clusters
// leaves.
int enqueue_wave_grids(Lane* l, const OccCall& oc, int B, int max_n) {
  pcop_handle* h = l->h;
  Ctx c = make_ctx(l, B, max_n);
  PCOP_CUDA_TRY(cudaStreamWaitEvent(l->stream, l->ev_grids_copied, 0));  // the previous wave's grids have left d_occ_grids
  run_occ_finish_wave(c, l->d_occ_counts, oc.g, l->d_occ_grids, l->d_warnings);
  OccShadowArgs a{};
  a.cloud = l->d_rem;
  a.cloud_stride = h->cap;
  a.n_points = l->cnt(CNT_REM);
  a.offsets = l->d_offsets;
  a.offsets_stride = (size_t)h->cap + 1;
  a.indices = l->d_indices;
  a.indices_stride = h->cap;
  a.n_clusters = l->cnt(CNT_CLUS);
  a.mats = l->d_occ_mats;
  a.y_min = oc.g.lim[2];
  a.x_max = oc.g.lim[1];
  a.block_size = oc.g.block_size;
  a.W = oc.g.W;
  a.size = oc.g.cells;
  a.opacity = h->params.grid_opacity;
  a.grid = l->d_occ_grids;
  a.warnings = l->d_warnings;
  // (the host does not know the cluster counts: a few blocks per frame, each taking every k-th cluster)
  run_occ_shadows(c, a, std::max(4, std::min(64, cdiv(2048, B))), max_n);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail_cuda(h, e, "grid launches", __FILE__, __LINE__);
  return PCOP_OK;
}

int enqueue_wave_back(Lane* l, const WaveInput& wi, int B, int max_n, uint32_t mask, const WaveRoute& r) {
  TRY(run_wave_cluster(l, B, max_n, r));
  if (wi.occ) TRY(enqueue_wave_grids(l, *wi.occ, B, max_n));
  return enqueue_wave_pack(l, B, max_n, mask, r);
}

// Enqueues one wave (largest frame: max_n points) on lane l along route r: input upload, all stages and
// enqueue_wave_back.  Returns without waiting for any of it.  repeat: the wave ran before (a voxel decline); its
// PointCloud2 payloads are staged already.
int enqueue_wave(Lane* l, const WaveInput& wi, int w0, int B, int max_n, uint32_t mask, const WaveRoute& r, bool repeat) {
  pcop_handle* h = l->h;
  for (int s = 0; s < PCOP_N_STAGES; ++s) l->stage_used[s] = false;
  const float4* in;
  size_t stride;
  const int32_t* n = wi.n;
  {
    StageTimer t(l, PCOP_STAGE_H2D);
    memcpy(l->h_n_in, n + w0, sizeof(int) * B);  // (the lane's previous wave has been collected: the staging is free)
    PCOP_CUDA_TRY(cudaMemcpyAsync(l->cnt(CNT_IN), l->h_n_in, sizeof(int) * B, cudaMemcpyHostToDevice, l->stream));
    if (wi.pc2) {  // from the decode on, the wave is a host-input wave
      TRY(enqueue_wave_decode(l, *wi.pc2, w0, B, max_n, repeat));
      in = l->d_in;
      stride = h->cap;
    } else if (wi.on_device) {
      in = reinterpret_cast<const float4*>(wi.xyzw) + (size_t)w0 * wi.frame_stride_points;
      stride = wi.frame_stride_points;
    } else {
      const float* src = wi.xyzw + (size_t)w0 * wi.frame_stride_points * 4;
      bool uniform = true;
      for (int f = 1; f < B; ++f) uniform = uniform && (n[w0 + f] == n[w0]);
      if (B > 0 && uniform && n[w0] > 0) {
        PCOP_CUDA_TRY(cudaMemcpy2DAsync(l->d_in, (size_t)h->cap * 16, src, wi.frame_stride_points * 16, (size_t)n[w0] * 16,
                                        B, cudaMemcpyHostToDevice, l->stream));
      } else {
        for (int f = 0; f < B; ++f)
          if (n[w0 + f] > 0)
            PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_in + (size_t)f * h->cap, src + (size_t)f * wi.frame_stride_points * 4,
                                          (size_t)n[w0 + f] * 16, cudaMemcpyHostToDevice, l->stream));
      }
      in = l->d_in;
      stride = h->cap;
    }
  }
  if (wi.occ) TRY(enqueue_wave_counts(l, *wi.occ, w0, B, in, stride, max_n));
  TRY(run_wave_stages(l, B, in, stride, max_n, r));
  l->pending = true;
  l->pend_w0 = w0;
  l->pend_B = B;
  l->pend_max_n = max_n;
  l->route = r;
  return enqueue_wave_back(l, wi, B, max_n, mask, r);
}

// Waits for the counts of the lane's wave in flight and corrects its route: each part of the wave a wrong guess left
// undone runs again, then the lane's history takes in what the wave needed.  The repeats, in this order:
//   - a frame the fused voxel path declined (a survivor with a NaN y or z: generic kernels; a bucket above the partition
//     path's limit: LSD path; more groups than the reduce grid covered: worst-case grid) repeats the whole wave;
//   - a plane-stage input above the small plane tier, when only that tier ran, repeats the wave from the plane stage on;
//   - a remaining cloud too large for the fused clustering kernel repeats the back half with the generic kernels.
int settle_wave(Lane* l, const WaveInput& wi, uint32_t mask) {
  pcop_handle* h = l->h;
  const pcop_params& p = h->params;
  const int w0 = l->pend_w0, B = l->pend_B, max_n = l->pend_max_n;
  const WaveRoute first = l->route;
  WaveRoute r = first;
  auto count = [&](int row, int f) { return l->h_counts[(size_t)row * h->maxB + f]; };
  PCOP_CUDA_TRY(cudaEventSynchronize(l->ev_meta));
  uint32_t vox_flags = 0u;
  int max_groups = 0;
  for (int f = 0; f < B && first.vox != WaveRoute::VOX_GENERIC; ++f) {
    vox_flags |= l->h_vf_flags[f];
    max_groups = std::max(max_groups, count(CNT_GROUPS, f));
  }
  if (vox_flags) {
    r.vox = (vox_flags & 1u) ? WaveRoute::VOX_GENERIC : ((vox_flags & 2u) ? WaveRoute::VOX_LSD : WaveRoute::VOX_PARTITION);
    r.vox_groups = l->vp_gstride - 1;
    TRY(enqueue_wave(l, wi, w0, B, max_n, mask, r, /*repeat=*/true));
    PCOP_CUDA_TRY(cudaEventSynchronize(l->ev_meta));
    for (int f = 0; f < B && r.vox != WaveRoute::VOX_GENERIC; ++f)  // (the repeat's flags came back with its metadata)
      if (l->h_vf_flags[f]) {
        l->pending = false;
        return fail(h, PCOP_ERR_INTERNAL, "the fused voxel path declined frame " + std::to_string(w0 + f) + " again on its repeat");
      }
  }
  bool large = false;
  for (int f = 0; f < B && p.enable_plane; ++f)  // (CNT_SOR = the plane stage's input size)
    large = large || count(CNT_SOR, f) > plane_small_tier_max();
  if (large && !r.plane_large) {
    r.plane_large = true;
    TRY(run_wave_plane(l, B, max_n, r));
    TRY(enqueue_wave_back(l, wi, B, max_n, mask, r));
    PCOP_CUDA_TRY(cudaEventSynchronize(l->ev_meta));
  }
  bool big = false;
  for (int f = 0; f < B && p.enable_cluster; ++f) big = big || count(CNT_REM, f) > h->ece_small_max;
  if (big && !r.cluster_generic && max_n > h->ece_small_max) {
    r.cluster_generic = true;
    TRY(enqueue_wave_back(l, wi, B, max_n, mask, r));
    PCOP_CUDA_TRY(cudaEventSynchronize(l->ev_meta));
  }

  // history (from the first run: the group count of the frames, the voxel-path flags)
  if (first.vox != WaveRoute::VOX_GENERIC) {
    if (h->vplan.part_ok)  // the next wave's reduce grid: 1.25 x the largest frame seen, >= 64
      l->vp_group_hint = std::min(l->vp_gstride - 1, std::max(64, max_groups + max_groups / 4 + 8));
    if (l->vox_lsd_waves > 0) --l->vox_lsd_waves;
    if (vox_flags & 2u) l->vox_lsd_waves = 64;  // dense buckets tend to come back: the next waves go straight to the LSD path
  }
  if (p.enable_plane) l->expect_large_plane = large;
  if (p.enable_cluster) l->expect_big_remaining = big;
  return PCOP_OK;
}

// Settles the lane's wave in flight, starts its payload copy and fills out[w0 .. w0 + B).  (Result pointers into
// the pinned buffer are stored as offsets and fixed up when the call ends: the buffer may still grow.)
int finish_wave(Lane* l, const WaveInput& wi, uint32_t mask, pcop_frame_result* out_all) {
  pcop_handle* h = l->h;
  if (!l->pending) return PCOP_OK;
  TRY(settle_wave(l, wi, mask));
  const int w0 = l->pend_w0, B = l->pend_B;
  l->pending = false;
  pcop_frame_result* out = out_all + w0;
  const bool dev_results = (mask & PCOP_OUT_DEVICE) != 0;
  const PackMeta meta = *l->h_meta;
  if (meta.overflow)
    return fail(h, PCOP_ERR_CAPACITY, "PCOP_OUT_DEVICE: the result arrays of this call do not fit the device pack buffer");
  const size_t base_off = (l->h_pack_used + 255) & ~(size_t)255;
  if (h->trace) cudaEventRecord(l->trace_recs[l->trace_used].c0, l->cstream);
  if (!dev_results) {
    // (when the buffer has to grow, grow it for all the waves this lane will see in the call: a pinned allocation
    // costs ~0.4 ms per MB, and every regrowth copies what is already there)
    if (base_off + meta.total_bytes + 256 > l->h_pack_cap)
      TRY(ensure_host_pack(l, base_off + (size_t)((double)(meta.total_bytes + 256) * 1.1 * std::max(1, l->call_lane_waves - l->wave_seq))));
    // payload copy on the copy stream (the pack kernels have finished: ev_meta follows them), in pieces: one large
    // device-to-host copy holds up the kernels of the other lanes for as long as it runs (measured: 6.4 ms per
    // 1024-frame call with one 17 MB copy per wave, 5.7 ms with 0.5-1 MB pieces, 5.9 / 6.2 ms with 2 / 4 MB pieces,
    // 6.3 ms with 256 KB pieces -- the host thread becomes the limit -- and 5.3 ms with no copy at all)
    const size_t piece = (size_t)1 << 20;
    for (size_t o = 0; o < meta.total_bytes; o += piece)
      PCOP_CUDA_TRY(cudaMemcpyAsync(l->h_pack + base_off + o, l->d_pack + o, std::min<size_t>(piece, meta.total_bytes - o),
                                    cudaMemcpyDeviceToHost, l->cstream));
    PCOP_CUDA_TRY(cudaEventRecord(l->ev_copied, l->cstream));
    l->h_pack_used = base_off + meta.total_bytes;
  }
  if (wi.occ) {  // the wave's grids, after its last repeat, on the copy stream beside the payload
    const size_t bytes = (size_t)B * (size_t)wi.occ->g.cells;
    int8_t* dst = wi.occ->grids + (size_t)w0 * (size_t)wi.occ->g.cells;
    const unsigned char* src = reinterpret_cast<const unsigned char*>(l->d_occ_grids);
    if (wi.occ->grids_on_device) {
      PCOP_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, l->cstream));
    } else {
      const size_t piece = (size_t)1 << 20;  // (pieces: as the payload above)
      for (size_t o = 0; o < bytes; o += piece)
        PCOP_CUDA_TRY(cudaMemcpyAsync(dst + o, src + o, std::min<size_t>(piece, bytes - o), cudaMemcpyDeviceToHost, l->cstream));
      h->d2h_bytes += (double)bytes;
    }
    PCOP_CUDA_TRY(cudaEventRecord(l->ev_grids_copied, l->cstream));
  }
  if (h->trace) {
    Lane::TraceRec& tr = l->trace_recs[l->trace_used++];
    cudaEventRecord(tr.c1, l->cstream);
    tr.w0 = w0;
    tr.B = B;
    tr.bytes = dev_results ? 0 : (size_t)meta.total_bytes;
  }
  h->d2h_bytes += (dev_results ? 0.0 : (double)meta.total_bytes) +
                  (double)(sizeof(int) * CNT_ROWS * h->maxB + sizeof(uint32_t) * B + sizeof(PlaneRecord) * B + sizeof(PackMeta));
  ++l->wave_seq;

  size_t run[PK_N] = {0};
  auto H = [&](int row, int f) { return l->h_counts[(size_t)row * h->maxB + f]; };
  for (int f = 0; f < B; ++f) {
    pcop_frame_result& r = out[f];
    memset(&r, 0, sizeof(r));
    r.status = PCOP_OK;
    r.warnings = l->h_warnings[f];
    r.n_input = H(CNT_IN, f);
    r.n_crop = H(CNT_CROP, f);
    r.n_voxel = H(CNT_VOX, f);
    r.n_sor = H(CNT_SOR, f);
    r.n_remaining = H(CNT_REM, f);
    r.n_clusters = H(CNT_CLUS, f);
    r.n_cluster_points = H(CNT_CLPTS, f);
    const PlaneRecord& pr = l->h_prec[f];
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
        *slots[k] = l->d_pack + (size_t)meta.base[k] + run[k] * kPkElem[k];
      } else {
        // store the byte offset now; turned into a pointer once the host buffer can no longer move
        const size_t off = base_off + (size_t)meta.base[k] + run[k] * kPkElem[k];
        *slots[k] = (const void*)(uintptr_t)(off + 1);  // +1 so that offset 0 is distinguishable from NULL
        l->fixups.push_back((size_t)((const unsigned char*)slots[k] - (const unsigned char*)out_all));
      }
      run[k] += (size_t)H(kPkCount[k], f);
    }
    // algorithmic bytes (SURVEY 8d)
    double b = 0.0;
    const pcop_params& p = h->params;
    if (wi.pc2)  // the decode: every message's payload in, PointXYZ out
      for (int k = wi.pc2->window_first[w0 + f]; k < wi.pc2->window_first[w0 + f + 1]; ++k)
        b += (double)(wi.pc2->msgs[k].point_step + 16) * wi.pc2->msgs[k].n_points;
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
    if (!l->stage_used[s]) continue;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, l->ev_stage[s][0], l->ev_stage[s][1]) == cudaSuccess) h->stage_us[s] += ms * 1000.f;
    else cudaGetLastError();
  }
  resolve_kernel_timers(h);
  return PCOP_OK;
}

static std::chrono::steady_clock::time_point g_trace_t0;
static double trace_host_us() {
  return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - g_trace_t0).count();
}

// occupancy grid scratch of one lane for waves of `frames` frames of `cells` cells (grown, never shrunk)
int ensure_occ_scratch(Lane* l, size_t frames, size_t cells) {
  pcop_handle* h = l->h;
  if (!l->d_occ_mats) {
    TRY(dalloc(h, &l->d_occ_mats, 2 * (size_t)h->maxB));
    TRY(halloc(h, &l->h_occ_mats, 2 * (size_t)h->maxB));
  }
  const size_t need = frames * cells;
  if (need <= l->occ_scratch_cells) return PCOP_OK;
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));
  PCOP_CUDA_TRY(cudaStreamSynchronize(l->cstream));
  if (l->d_occ_counts) cudaFree(l->d_occ_counts);  // (not tracked in dev_allocs)
  if (l->d_occ_grids) cudaFree(l->d_occ_grids);
  l->d_occ_counts = nullptr;
  l->d_occ_grids = nullptr;
  l->occ_scratch_cells = 0;
  PCOP_CUDA_TRY(cudaMalloc((void**)&l->d_occ_counts, sizeof(int) * need));
  PCOP_CUDA_TRY(cudaMalloc((void**)&l->d_occ_grids, need));
  l->occ_scratch_cells = need;
  return PCOP_OK;
}

}  // namespace

namespace pcop {

__global__ void k_zero_u32(uint32_t* p, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0u;
}

int process_impl(pcop_handle* h, const float* xyzw, size_t frame_stride_points, const int32_t* n, int32_t batch,
                 pcop_frame_result* out, const OccCall* occ, const Pc2Call* pc2) {
  if (!h) return fail(nullptr, PCOP_ERR_BAD_PARAM, "null handle");
  if ((!xyzw && !pc2) || !n || !out || batch < 0) return fail(h, PCOP_ERR_BAD_PARAM, "null argument");
  PCOP_CUDA_TRY(cudaSetDevice(h->device));
  for (int f = 0; f < batch; ++f) {
    if (n[f] < 0) return fail(h, PCOP_ERR_BAD_PARAM, "negative point count");
    if (n[f] > h->cap) return fail(h, PCOP_ERR_CAPACITY, "frame has more points than max_points");
    if ((size_t)n[f] > frame_stride_points && batch > 1) return fail(h, PCOP_ERR_BAD_PARAM, "frame_stride_points < n");
  }
  const uint32_t mask = effective_outputs(h->params);
  const WaveInput wi{xyzw, frame_stride_points, n, pc2 ? false : is_device_pointer(xyzw), pc2, occ};
  // lanes used by this call: per-kernel timing needs each kernel alone on the GPU, so it serialises the lanes
  std::vector<Lane*> lanes(1, h->lanes[0].get());
  if (!h->kt.enabled)
    for (size_t i = 1; i < h->lanes.size(); ++i) lanes.push_back(h->lanes[i].get());
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
  // PointCloud2 messages: host payload bytes of the largest wave, as staged (256-byte aligned), and its message count
  size_t raw_need = 0, pc2_need = 0;
  if (pc2)
    for (const auto& w : waves) {
      size_t bytes = 0;
      const int m0 = pc2->window_first[w.first], m1 = pc2->window_first[w.first + w.second];
      for (int k = m0; k < m1; ++k)
        if (!pc2->on_device[k]) bytes += (pc2_payload_bytes(pc2->msgs[k]) + 255) & ~(size_t)255;
      raw_need = std::max(raw_need, bytes);
      pc2_need = std::max(pc2_need, (size_t)(m1 - m0));
    }
  h->launches = 0;
  h->alg_bytes = 0.0;
  h->d2h_bytes = 0.0;
  h->kt.used = 0;
  h->sort_pass_keys = 0;
  for (int s = 0; s < PCOP_N_STAGES; ++s) h->stage_us[s] = 0.f;
  for (Lane* l : lanes) {
    if (occ && !waves.empty()) TRY(ensure_occ_scratch(l, (size_t)waves[0].second, (size_t)occ->g.cells));  // (the first wave is the largest)
    if (raw_need) TRY(ensure_raw(l, raw_need));
    if (pc2_need) TRY(ensure_pc2(l, pc2_need));
    l->h_pack_used = 0;
    l->h_pack_sel ^= 1;
    l->h_pack = l->h_pack_buf[l->h_pack_sel];
    l->h_pack_cap = l->h_pack_buf_cap[l->h_pack_sel];
    l->fixups.clear();
    l->wave_seq = 0;
    l->call_lane_waves = cdiv((int)waves.size(), (int)lanes.size());
    l->trace_used = 0;
    l->pending = false;
    TRY(ensure_pack_capacity(l, mask));
  }
  PCOP_CUDA_TRY(cudaEventRecord(h->ev_call[0], lanes[0]->stream));
  if (h->trace) g_trace_t0 = std::chrono::steady_clock::now();
  for (size_t l = 0; l < lanes.size(); ++l) {
    if (l > 0) PCOP_CUDA_TRY(cudaStreamWaitEvent(lanes[l]->stream, h->ev_call[0], 0));
    PCOP_CUDA_TRY(cudaMemsetAsync(lanes[l]->sort.stats, 0, sizeof(unsigned long long), lanes[l]->stream));
    if (mask & PCOP_OUT_DEVICE)
      PCOP_CUDA_TRY(cudaMemsetAsync(lanes[l]->d_pack_cursor, 0, sizeof(unsigned long long), lanes[l]->stream));
  }
  int status = PCOP_OK;
  for (size_t w = 0; w < waves.size() && status == PCOP_OK; ++w) {
    Lane* l = lanes[w % lanes.size()];
    const double th0 = h->trace ? trace_host_us() : 0.0;
    status = finish_wave(l, wi, mask, out);  // (the lane's previous wave, if any)
    const double th1 = h->trace ? trace_host_us() : 0.0;
    if (status == PCOP_OK) {  // (after the finish: the route follows the history the lane's previous wave left)
      const int w0 = waves[w].first, B = waves[w].second;
      int max_n = 1;
      for (int f = w0; f < w0 + B; ++f) max_n = std::max(max_n, (int)n[f]);
      status = enqueue_wave(l, wi, w0, B, max_n, mask, next_route(l, max_n), /*repeat=*/false);
    }
    if (h->trace)
      fprintf(stderr, "[pcop trace]   host: wave %4d+%-4d lane %zu: finish of the lane's previous wave %7.0f .. %7.0f us, enqueue .. %7.0f us\n",
              waves[w].first, waves[w].second, w % lanes.size(), th0, th1, trace_host_us());
  }
  // collect what is still in flight, oldest first
  for (size_t k = 0; k < lanes.size(); ++k) {
    const int st = finish_wave(lanes[(waves.size() + k) % lanes.size()], wi, mask, out);
    if (st != PCOP_OK && status == PCOP_OK) status = st;
  }
  for (Lane* l : lanes) {  // the call is done when every lane's last result copy has landed
    cudaMemcpyAsync(l->h_stats, l->sort.stats, sizeof(unsigned long long), cudaMemcpyDeviceToHost, l->stream);
    cudaEventRecord(l->ev_lane_done, l->cstream);
    cudaStreamWaitEvent(l->stream, l->ev_lane_done, 0);
    cudaEventRecord(l->ev_lane_done, l->stream);
    if (l != lanes[0]) cudaStreamWaitEvent(lanes[0]->stream, l->ev_lane_done, 0);
  }
  PCOP_CUDA_TRY(cudaEventRecord(h->ev_call[1], lanes[0]->stream));
  PCOP_CUDA_TRY(cudaEventSynchronize(h->ev_call[1]));
  if (status != PCOP_OK) return status;
  float ms = 0.f;
  PCOP_CUDA_TRY(cudaEventElapsedTime(&ms, h->ev_call[0], h->ev_call[1]));
  h->last_elapsed_us = ms * 1000.f;
  if (h->trace) {
    fprintf(stderr, "[pcop trace] call of %d frames: %.0f us on the device\n", batch, ms * 1000.f);
    for (size_t li = 0; li < lanes.size(); ++li) {
      for (size_t k = 0; k < lanes[li]->trace_used; ++k) {
        const Lane::TraceRec& tr = lanes[li]->trace_recs[k];
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
  for (Lane* l : lanes) {
    h->sort_pass_keys += *l->h_stats;
    // the host pack buffers are final now: turn the stored offsets into pointers
    for (size_t fx : l->fixups) {
      const void** slot = (const void**)((unsigned char*)out + fx);
      const size_t off = (size_t)(uintptr_t)(*slot) - 1;
      *slot = l->h_pack + off;
    }
  }
  return PCOP_OK;
}

int pc2_ingest(pcop_handle* h, const unsigned char* data, int32_t n, int32_t point_step, int32_t ox, int32_t oy,
               int32_t oz, const float* t16, int is_dense, float4* dst) {
  if (!pc2_layout_ok(point_step, ox, oy, oz)) return fail(h, PCOP_ERR_BAD_PARAM, "PointCloud2 field offsets do not fit point_step");
  Lane* l = h->lanes[0].get();
  const size_t bytes = (size_t)n * (size_t)point_step;
  const unsigned char* src = data;
  if (!is_device_pointer(data)) {
    TRY(ensure_raw(l, bytes));
    PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_raw, data, bytes, cudaMemcpyHostToDevice, l->stream));
    src = l->d_raw;
  }
  // the batched decode with one message; the descriptor goes up from pageable memory (staged before the call returns)
  TRY(ensure_pc2(l, 1));
  const Pc2Frame d = make_pc2_frame(src, n, point_step, ox, oy, oz, t16, is_dense);  // (dst = 0, tile0 = 0)
  PCOP_CUDA_TRY(cudaMemcpyAsync(l->d_pc2, &d, sizeof(d), cudaMemcpyHostToDevice, l->stream));
  Ctx c = make_ctx(l, 1, n);
  KL(c, "k_pc2_ingest", k_pc2_ingest<<<cdiv(n, PC2_TILE), PC2_THREADS, 0, l->stream>>>(l->d_pc2, 1, dst));
  count_launch(c);
  if (src != data) PCOP_CUDA_TRY(cudaStreamSynchronize(l->stream));  // the caller may reuse its buffer
  return PCOP_OK;
}

}  // namespace pcop
