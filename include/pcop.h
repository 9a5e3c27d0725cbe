/*
 * pcop.h — C ABI of the B200-native point-cloud obstacle-processing hot path.
 *
 * Drop-in boundary for the five PCL call sites of the reference ROS node
 * (minibot_cr18/src/obstacle_detection.cpp, "od.cpp" below):
 *
 *   od.cpp:727  build_initial_occupancy_grid_dataset  (crop loop od.cpp:195-215)  -> pcop_crop
 *   od.cpp:740  downsample_cloud                      (od.cpp:271-296)            -> pcop_voxel
 *   od.cpp:751  remove_statistical_outliers           (od.cpp:316-340)            -> pcop_sor
 *   od.cpp:778  segment_plane_and_extract_indices     (od.cpp:342-428)            -> pcop_plane
 *   od.cpp:796  extract_euclidian_clusters            (od.cpp:430-455, 791-792)   -> pcop_cluster
 *   msg/PointWithRad.msg:1-4, msg/PointIndicesArray.msg:1 (dead call od.cpp:806-814)
 *                                                                                 -> pcop_centroid_radius
 *   the whole stage sequence of cloud_cb (od.cpp:699-927)                         -> pcop_process / pcop_process_batch
 *   od.cpp:688-698  PointCloud2 decode + world transform + accumulate             -> pcop_accumulate_pointcloud2 / pcop_accumulate
 *   od.cpp:290-294  toROSMsg of the intermediate clouds (debug publishers)           -> pcop_cloud_to_pointcloud2
 *   od.cpp:727  build_initial_occupancy_grid_dataset  (grid part od.cpp:134-157, 184-269) -> pcop_occupancy_grid
 *   od.cpp:817-833  handle_shadow_casting per cluster (od.cpp:467-672) + obstacle marks   -> pcop_occupancy_shadows
 *   od.cpp:699-852  pipeline + occupancy grid of a batch of frames                        -> pcop_process_batch_occupancy
 *   od.cpp:688-696 + 699-852  the same for a batch of raw PointCloud2 messages with a pose each -> pcop_process_batch_pointcloud2
 *   od.cpp:688-701 + 699-852  ... with accumulate_count messages (or several sensors) per frame -> pcop_process_batch_pointcloud2_windows
 *
 * Plain C: POD structs, raw pointers and sizes, integer status codes.  No C++
 * exceptions, PCL, ROS or torch types cross this boundary.
 *
 * A point is a pcl::PointXYZ as PCL lays it out: four floats {x, y, z, pad},
 * 16-byte stride.  `cloud.points.data()` can be passed as-is.  Input pointers
 * may be host or device pointers (detected with cudaPointerGetAttributes).
 *
 * Threading: one handle = one device = one caller at a time (the reference
 * node is single-threaded, od.cpp:1014).  Different handles may be driven
 * concurrently from different threads.
 *
 * There is NO CPU fallback: every entry point that computes fails with
 * PCOP_ERR_CUDA when no sm_100-class device is usable.
 */
#ifndef PCOP_H_
#define PCOP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCOP_ABI_VERSION 1
#define PCOP_MAX_PLANE_PASSES_RECORDED 16
#define PCOP_MAX_HYPOTHESES 64

/* ---- status codes -------------------------------------------------------- */
enum {
  PCOP_OK = 0,
  PCOP_ERR_BAD_PARAM = 1,
  PCOP_ERR_CAPACITY = 2,  /* frame larger than max_points / batch larger than allowed */
  PCOP_ERR_CUDA = 3,
  PCOP_ERR_INTERNAL = 4
};

/* per-frame warning bits (pcop_frame_result.warnings) */
enum {
  PCOP_WARN_VOXEL_OVERFLOW_FALLBACK = 1, /* PCL: "Leaf size is too small": output = input   */
  PCOP_WARN_SOR_TOO_FEW_POINTS = 2,      /* V <= meanK: cloud passed through unchanged      */
  PCOP_WARN_PLANE_BREAK = 4,             /* od.cpp:383-387: no inliers, loop left early     */
  PCOP_WARN_RNG_TABLE_EXHAUSTED = 8,     /* >PCOP rng table draws needed (degenerate cloud) */
  PCOP_WARN_SHADOW_DEGENERATE = 16       /* pcop_occupancy_shadows: a shadow fan too long to draw was skipped */
};

/* which arrays pcop_process* copies back to the host (pcop_params.outputs) */
enum {
  PCOP_OUT_CROP = 1,       /* crop_kept_idx                               */
  PCOP_OUT_VOXEL = 2,      /* voxel_keys, voxel_centroids                 */
  PCOP_OUT_SOR = 4,        /* sor_kept_idx                                */
  PCOP_OUT_PLANE = 8,      /* plane_inlier_idx (last pass)                */
  PCOP_OUT_REMAINING = 16, /* remaining_cloud, remaining_src_idx          */
  PCOP_OUT_CLUSTERS = 32,  /* cluster_offsets, cluster_indices            */
  PCOP_OUT_OBSTACLES = 64, /* obstacles                                   */
  PCOP_OUT_DEFAULT = 16 | 32 | 64,
  PCOP_OUT_ALL = 127,
  /* Modifier: leave the requested arrays in device memory.  The pcop_frame_result pointers are then DEVICE pointers
   * (valid until the next pcop_process* call on the handle; counts, warnings and the plane record are still host
   * values) for a consumer that lives on the GPU: the next GPU stage, a peer-to-peer / NCCL transfer,
   * pcop_cloud_to_pointcloud2 or pcop_download.  The arrays of all waves of a call stay in the handle's pack buffers
   * (sized by pcop_create for the worst case of one wave); a call whose results do not fit returns PCOP_ERR_CAPACITY. */
  PCOP_OUT_DEVICE = 256
};

/* stage ids for pcop_stage_times_us */
enum {
  PCOP_STAGE_H2D = 0,
  PCOP_STAGE_CROP = 1,
  PCOP_STAGE_VOXEL = 2,
  PCOP_STAGE_SOR = 3,
  PCOP_STAGE_PLANE = 4,
  PCOP_STAGE_CLUSTER = 5,
  PCOP_STAGE_CENTROID = 6,
  PCOP_STAGE_D2H = 7,
  PCOP_N_STAGES = 8
};

/*
 * Parameters.  Field names are the params.yaml keys (minibot_cr18/params.yaml:1-31)
 * read at od.cpp:940-975.  Types follow the globals they are read into
 * (od.cpp:82-118): note plane_segment_angle is an `int` handed to
 * setEpsAngle() as radians (od.cpp:111, 371).
 */
typedef struct pcop_params {
  /* crop box, inclusive (od.cpp:197-199; params.yaml:2-7) */
  float x_min, x_max, y_min, y_max, z_min, z_max;
  /* VoxelGrid leaf (od.cpp:284; params.yaml:16) */
  float downsample_size;
  /* StatisticalOutlierRemoval (od.cpp:328-329; params.yaml:20-21) */
  int32_t statistical_outlier_meanK;
  float statistical_outlier_stdDevThres;
  /* SACSegmentation (od.cpp:365-372; params.yaml:23-24) */
  float plane_segment_dist_thres;
  int32_t plane_segment_angle;
  /* EuclideanClusterExtraction (od.cpp:447-449; params.yaml:26-28) */
  float euc_cluster_tolerance;
  int32_t euc_min_cluster_size;
  int32_t euc_max_cluster_size;

  /* hard-coded in the reference, exposed with the reference's values */
  float plane_axis[3];           /* od.cpp:769  (0,0,1)                        */
  double plane_keep_fraction;    /* od.cpp:379  0.3                            */
  int32_t plane_max_iterations;  /* PCL default 50                             */
  double plane_probability;      /* PCL default 0.99                           */
  uint32_t ransac_seed;          /* PCL SampleConsensusModel: mt19937(12345)   */
  int32_t optimize_coefficients; /* od.cpp:365 true                            */

  /* stage enables (the reference always runs all five; benches/configs 2-4 switch some off) */
  int32_t enable_crop, enable_voxel, enable_sor, enable_plane, enable_cluster;

  /* od.cpp:945 publish_point_clouds -> return intermediates; OR-ed into outputs as PCOP_OUT_ALL */
  int32_t publish_point_clouds;
  uint32_t outputs; /* PCOP_OUT_* mask */

  /* accepted and ignored, for surface compatibility (SURVEY 5.1) */
  int32_t accumulate_count;
  float block_size, dev_percent;
  int32_t grid_opacity;
  int32_t downsample_input_data; /* also covers the YAML misspelling downsame_input_data */
  int32_t passthrough_filter_enable;
  float convex_hull_alpha;
} pcop_params;

/* Code defaults of od.cpp:940-975 (note: inverted z range drops everything). */
void pcop_params_init_code_defaults(pcop_params* p);
/* Values of minibot_cr18/params.yaml:1-31. */
void pcop_params_init_params_yaml(pcop_params* p);

/*
 * Result of one frame.  All pointers point into pinned host memory owned by
 * the handle and stay valid until the next pcop_process* call on that handle.
 * Arrays whose PCOP_OUT_* bit is not requested are NULL.
 */
typedef struct pcop_frame_result {
  int32_t status;   /* PCOP_OK or error for this frame */
  uint32_t warnings;
  /* counts: N, M, V, S, P, C, L (SURVEY 8) */
  int32_t n_input, n_crop, n_voxel, n_sor, n_remaining, n_clusters, n_cluster_points;
  /* plane loop record */
  int32_t n_plane_passes; /* passes that removed inliers */
  int32_t plane_pass_points[PCOP_MAX_PLANE_PASSES_RECORDED];  /* P_k  */
  int32_t plane_pass_inliers[PCOP_MAX_PLANE_PASSES_RECORDED]; /* I_k  */
  float plane_pass_coeff[PCOP_MAX_PLANE_PASSES_RECORDED][4];  /* refined a,b,c,d */
  float plane_coeff[4];        /* coefficients of the last segment() call (pcl::ModelCoefficients) */
  int32_t n_plane_inliers;     /* size of `inliers` after the loop (last segment call)  */

  const int32_t* crop_kept_idx;      /* [M] index into the input                         */
  const uint32_t* voxel_keys;        /* [V] ascending                                     */
  const float* voxel_centroids;      /* [V][4]                                            */
  const int32_t* sor_kept_idx;       /* [S] index into the voxel cloud                    */
  const int32_t* plane_inlier_idx;   /* [n_plane_inliers] index into the last pass' input */
  const float* remaining_cloud;      /* [P][4] = planar_cloud_y (od.cpp:765), cluster indices index into it */
  const int32_t* remaining_src_idx;  /* [P] index into the plane-loop input cloud         */
  const int32_t* cluster_offsets;    /* [C+1] CSR                                         */
  const int32_t* cluster_indices;    /* [L]   -> std::vector<pcl::PointIndices>           */
  const float* obstacles;            /* [C][4] PointWithRad {x,y,z,r}                     */
} pcop_frame_result;

typedef struct pcop_handle pcop_handle;

/*
 * Create a handle on `device` able to process frames of up to `max_points`
 * points, `max_batch` frames per internal wave (larger batches are processed
 * in waves).  All device and pinned memory is allocated here.
 */
int pcop_create(const pcop_params* params, int device, size_t max_points, int max_batch, pcop_handle** out);
void pcop_destroy(pcop_handle* h);
const char* pcop_last_error(const pcop_handle* h);
/* Static error text for failures that happen before a handle exists. */
const char* pcop_global_error(void);
int pcop_abi_version(void);

/* Replace parameters (no reallocation; capacity unchanged). */
int pcop_set_params(pcop_handle* h, const pcop_params* params);

/* One frame through every enabled stage (cloud_cb process branch, od.cpp:699-927).
 * Host result arrays live in pinned buffers owned by the handle; the handle alternates between two of them, so the
 * pointers a call returns stay valid until the call AFTER the next one on the same handle (a consumer -- the next
 * pipeline stage, a multi-GPU gather -- may still read the results of call k while call k + 1 runs). */
int pcop_process(pcop_handle* h, const float* xyzw, int32_t n, pcop_frame_result* out);

/*
 * `batch` independent frames.  Frame f is `n[f]` points at `xyzw + f*frame_stride_points*4`
 * (host or device memory).  `out` has `batch` entries.
 */
int pcop_process_batch(pcop_handle* h, const float* xyzw, size_t frame_stride_points, const int32_t* n,
                       int32_t batch, pcop_frame_result* out);

/* Device time of the last pcop_process* call, CUDA events on the handle's stream. */
float pcop_last_elapsed_us(const pcop_handle* h);
/* Per-stage device time of the last call (summed over waves). */
int pcop_stage_times_us(const pcop_handle* h, float us[PCOP_N_STAGES]);
/* Kernel launches issued by the last call. */
int64_t pcop_last_launch_count(const pcop_handle* h);
/* Algorithmic bytes (SURVEY 8d table) of the last call, from its counts. */
double pcop_last_algorithmic_bytes(const pcop_handle* h);
/* Keys moved by radix-sort passes during the last call (each is 8 B read + 8 B written). */
int64_t pcop_last_sort_pass_keys(const pcop_handle* h);
/* ---- accumulator ingest (replaces od.cpp:691-698) --------------------------------------------------
 * The node transforms every incoming cloud into the world frame (pcl_ros::transformPointCloud, od.cpp:696) and
 * appends it to passthrough_input_cloud (od.cpp:697) until accumulate_count clouds have arrived; the next callback
 * runs the pipeline on the accumulated cloud (od.cpp:699 ff).  Here the accumulated cloud lives on the device:
 *   pcop_accumulate           transform (row-major 4x4 float, NULL = identity; PCL's coefficient formula in float)
 *                             + append; is_dense = 0 copies points with a non-finite coordinate unchanged (PCL's
 *                             behaviour for clouds with is_dense == false, e.g. Kinect clouds with NaN holes)
 *   pcop_accumulated_count    points accumulated so far
 *   pcop_process_accumulated  pcop_process on the accumulated cloud (never leaves the device), then reset
 *   pcop_accumulate_reset     drop what was accumulated
 *   pcop_transform            stage-isolated transform of one cloud (parity tests)
 * PCOP_ERR_CAPACITY when the accumulated cloud would exceed max_points. */
int pcop_accumulate(pcop_handle* h, const float* xyzw, int32_t n, const float* transform16, int32_t is_dense, int32_t* total);
int32_t pcop_accumulated_count(const pcop_handle* h);
int pcop_process_accumulated(pcop_handle* h, pcop_frame_result* out);
int pcop_accumulate_reset(pcop_handle* h);
int pcop_transform(pcop_handle* h, const float* xyzw, int32_t n, const float* transform16, int32_t is_dense, float* out_xyzw);

/* ---- PointCloud2 wire ingest (replaces od.cpp:688-689 + 691-698) ------------------------------------
 * pcl_conversions::toPCL + pcl::fromPCLPointCloud2<PointXYZ> extract the FLOAT32 fields x, y, z of every
 * point_step-byte record of the message payload (the author's second slowest step, od.cpp:721).  Here the raw
 * payload is uploaded once and ONE kernel decodes the records, applies the world transform and appends to the
 * accumulator (the PointXYZ padding float becomes 1.0f, as in a default-constructed pcl::PointXYZ).
 *   data        sensor_msgs/PointCloud2.data (host or device pointer), n_points = width * height records
 *   point_step  bytes per record; off_x/off_y/off_z = offsets of the FLOAT32 fields "x", "y", "z"
 * pcop_pointcloud2_to_xyz is the stage-isolated decode (no transform) for parity tests. */
int pcop_accumulate_pointcloud2(pcop_handle* h, const unsigned char* data, int32_t n_points, int32_t point_step,
                                int32_t off_x, int32_t off_y, int32_t off_z, const float* transform16, int32_t is_dense,
                                int32_t* total);
int pcop_pointcloud2_to_xyz(pcop_handle* h, const unsigned char* data, int32_t n_points, int32_t point_step, int32_t off_x,
                            int32_t off_y, int32_t off_z, float* out_xyzw);

/* ---- PointCloud2 wire egress (replaces the pcl::toROSMsg calls of the debug publishers, od.cpp:290-294, 332-339,
 * 401-426) -------------------------------------------------------------------------------------------------
 * pcl::toROSMsg(pcl::PointCloud<pcl::PointXYZ>) copies the PointXYZ records verbatim into sensor_msgs/PointCloud2.data:
 * point_step 16, fields x / y / z FLOAT32 (datatype 7, count 1) at offsets 0 / 4 / 8, the padding float travels along;
 * width = n, height = 1, row_step = 16 n, is_bigendian = false.  pcop_cloud_to_pointcloud2 writes that payload for
 * (point_step, offsets) = (16, 0, 4, 8); for any other layout it writes the three FLOAT32 fields of every record and
 * zeroes the other bytes.
 *   xyzw      the cloud (host or device pointer, e.g. a result array of a PCOP_OUT_DEVICE call), n records
 *   out_data  n * point_step bytes (host or device pointer) */
int pcop_cloud_to_pointcloud2(pcop_handle* h, const float* xyzw, int32_t n, int32_t point_step, int32_t off_x, int32_t off_y,
                              int32_t off_z, unsigned char* out_data);

/* ---- occupancy grid, initial data set (replaces od.cpp:134-157 + 175-269) ---------------------------------
 * The node's published product starts as a count of the crop survivors per block_size x block_size cell (rows along
 * -x from x_max, columns along +y from y_min), a per-row integer average and the threshold
 *   cell = (count < row_average * (1 - dev_percent)) ? 100 : 0        (float compare, od.cpp:258).
 * pcop_occupancy_dims: width/height as od.cpp:958-959.  pcop_occupancy_grid: xyzw = NULL takes the accumulated cloud
 * (pcop_accumulate*); grid_data[width*height] int8; counts[width*height] / row_avg[height] int64 are optional.
 * Shadow casting and the obstacle marks (od.cpp:467-672, 817-833): pcop_occupancy_shadows below. */
int pcop_occupancy_dims(const pcop_handle* h, int32_t* width, int32_t* height);
int pcop_occupancy_grid(pcop_handle* h, const float* xyzw, int32_t n, int8_t* grid_data, int64_t* counts, int64_t* row_avg);

/* ---- occupancy grid, shadow casting + obstacle marks (replaces od.cpp:467-672 and the loops of od.cpp:817-833) ----
 * For every cluster of >= 2 points (handle_shadow_casting, od.cpp:584-672): the members go into the sensor frame
 * (world_to_sensor16 = the "kinect2_link" <- "world" TF lookup of od.cpp:592, row-major 4x4 float, applied with
 * pcl::transformPointCloud's coefficient formula); the first member with the smallest sensor x starts the shadow, the
 * largest x and the y range give its height and width; calculate_shadow_cast (od.cpp:540-582) gives the end point,
 * which goes back to the world frame through sensor_to_world16 (od.cpp:570, 634); a fan of ceil(width / block_size) + 3
 * lines (traceShadow, od.cpp:467-538) is drawn with cells set to grid_opacity.  Afterwards every remaining point with
 * a non-NaN x marks its cell 100 (od.cpp:823-833).
 *   remaining_xyzw / cluster_offsets / cluster_indices   the arrays of a pcop_frame_result (host or device pointers)
 *   grid_data [height*width]   in/out (host or device pointer): the grid pcop_occupancy_grid produced
 *   shadow_records [C][6]      optional: start_x, start_y, end_x, end_y of the first line (grid cells, after the
 *                              half-width shift), lines drawn, skipped flag
 *   warnings                   optional: PCOP_WARN_SHADOW_DEGENERATE
 * Where the reference leaves the arithmetic to the platform or runs into undefined behaviour, this library defines:
 * unqualified fabs / sqrt / asin / tan / ceil are the double overloads (asin, tan: fixed IEEE operation sequences,
 * < 1e-15 from libm); the cell search of get_occupancy_grid_x_y stops after 2^20 steps; cell indices are 64-bit;
 * float/double -> int conversions saturate to INT_MIN like cvttss2si / cvttsd2si; a line longer than 65536 pixels or a
 * fan of more than 65536 lines is skipped (PCOP_WARN_SHADOW_DEGENERATE); the obstacle marks are bounds-checked. */
int pcop_occupancy_shadows(pcop_handle* h, const float* remaining_xyzw, int32_t n_remaining, const int32_t* cluster_offsets,
                           const int32_t* cluster_indices, int32_t n_clusters, const float* world_to_sensor16,
                           const float* sensor_to_world16, int8_t* grid_data, int32_t* shadow_records, uint32_t* warnings);

/* ---- the node's published product for a batch of frames (od.cpp:699-852 per frame) ----------------------------
 * Every frame of the batch through every enabled stage AND the occupancy grid it publishes, in one call: the initial
 * data set of pcop_occupancy_grid, then the shadows and obstacle marks of pcop_occupancy_shadows on the frame's own
 * remaining cloud and clusters.  Grid kernels run inside the batched pipeline; nothing returns to the host per frame.
 *   xyzw, frame_stride_points, n, batch, out   as pcop_process_batch; every out[f] equals what pcop_process_batch
 *                                              returns for the same frames (PCOP_OUT_DEVICE, pointer lifetime and
 *                                              alternating pinned buffers included), except that
 *                                              PCOP_WARN_SHADOW_DEGENERATE is set in the frames where a fan was skipped.
 *                                              xyzw = NULL with batch = 1 (n ignored): the accumulated cloud, which the
 *                                              call consumes like pcop_process_accumulated.
 *   world_to_sensor16, sensor_to_world16       [batch][16] row-major floats (host memory), frame f's two TF lookups
 *                                              (od.cpp:592 and od.cpp:570, 634); required
 *   grids                                      [batch][height][width] int8 (host or device pointer; width / height
 *                                              from pcop_occupancy_dims): frame f's grid equals, byte for byte,
 *                                              pcop_occupancy_grid(frame f) followed by pcop_occupancy_shadows(frame f's
 *                                              results, frame f's matrices).  Shadow records are not produced.
 *                                              Host grids should be pinned (cudaHostAlloc): a copy into pageable memory
 *                                              holds the calling thread until it lands, once per wave, so the lanes
 *                                              stop overlapping.
 * The handle keeps the counts (int32) and cells of one wave per lane, 5 bytes per cell and per frame of the largest
 * wave the lane has run (allocated by the first call, grown when pcop_set_params enlarges the grid or a call brings
 * larger waves): grids of more than PCOP_OCC_BATCH_MAX_CELLS cells give PCOP_ERR_CAPACITY (the single-frame calls
 * above take grids up to 2^26 cells).  pcop_last_d2h_bytes counts the grid bytes copied to host memory. */
#define PCOP_OCC_BATCH_MAX_CELLS (1 << 20)
int pcop_process_batch_occupancy(pcop_handle* h, const float* xyzw, size_t frame_stride_points, const int32_t* n,
                                 int32_t batch, const float* world_to_sensor16, const float* sensor_to_world16,
                                 int8_t* grids, pcop_frame_result* out);

/* ---- a batch of raw sensor_msgs/PointCloud2 messages (od.cpp:688-696 + 699-852 per message) ------------------------
 * A log replay, or several robots sharing one GPU, hands over sensor-frame messages, each with its own TF and its own
 * driver's record layout.  pcop_process_batch_pointcloud2 decodes every message (toPCL + fromPCLPointCloud2<PointXYZ>),
 * transforms it into the world frame (pcl_ros::transformPointCloud) and runs it through the batched pipeline -- and,
 * with grids != NULL, the grid product of pcop_process_batch_occupancy -- in one call.  Decode and transform run on the
 * GPU inside the batched pipeline; nothing returns to the host per message.
 *   frames             [batch] message descriptors (host memory); layouts may differ from message to message.  A
 *                      message with n_points == 0 may have data == NULL.  Payloads may be host or device pointers
 *                      (classified per allocation).  Host payloads should be pinned (cudaHostAlloc): a copy from pageable
 *                      memory holds the calling thread until it has been staged, once per message, so the lanes stop
 *                      overlapping.  Device payloads are read in place.
 *   transform16        [batch][16] row-major floats (host memory), message f's world <- sensor pose, applied with
 *                      pcl::transformPointCloud's coefficient formula (is_dense = 0: records with a non-finite x, y or z
 *                      are copied untransformed); NULL: no transform (payloads already in the world frame)
 *   world_to_sensor16, sensor_to_world16, grids    as pcop_process_batch_occupancy; grids = NULL: pipeline only (the two
 *                      matrices are then not read).  A replay of single messages passes the same array as transform16
 *                      and sensor_to_world16.
 *   out                [batch]
 * out[f] equals, byte for byte, what pcop_accumulate_reset + pcop_accumulate_pointcloud2(message f, transform16 + 16 f)
 * + pcop_process_accumulated return, i.e. pcop_process_batch on the decoded world clouds (padding float 1.0f); with grids,
 * results and grids equal pcop_process_batch_occupancy on those clouds with the same matrices.  PCOP_OUT_DEVICE, result
 * pointer lifetime and the alternating pinned result buffers behave as in pcop_process_batch.  The accumulator is neither
 * read nor changed.
 * Errors (the handle stays usable): PCOP_ERR_BAD_PARAM for a negative n_points, point_step < 4, a field offset with
 * off + 4 > point_step, NULL data with n_points > 0, frames = NULL with batch > 0, or grids without the two matrices;
 * PCOP_ERR_CAPACITY for n_points > max_points or a grid above PCOP_OCC_BATCH_MAX_CELLS.  batch = 0 does nothing.
 * Every lane of the handle stages the host payloads of one wave (allocated by the first call, grown to the largest wave's
 * payload bytes); pcop_stage_times_us counts the upload and the decode as PCOP_STAGE_H2D. */
typedef struct pcop_pointcloud2_frame {
  const unsigned char* data;   /* PointCloud2.data: host or device pointer                        */
  int32_t n_points;            /* width * height records                                           */
  int32_t point_step;          /* bytes per record                                                  */
  int32_t off_x, off_y, off_z; /* offsets of the FLOAT32 fields "x", "y", "z" (little-endian)       */
  int32_t is_dense;            /* 0: PCL's rule for is_dense == false, non-finite points untransformed */
} pcop_pointcloud2_frame;
int pcop_process_batch_pointcloud2(pcop_handle* h, const pcop_pointcloud2_frame* frames, int32_t batch,
                                   const float* transform16, const float* world_to_sensor16,
                                   const float* sensor_to_world16, int8_t* grids, pcop_frame_result* out);

/* ---- accumulation windows: one frame from several posed messages (od.cpp:688-701 per processing callback) ---------
 * The node appends accumulate_count posed messages to passthrough_input_cloud and runs the pipeline on the
 * concatenation; a rig with several sensors merges their messages into one cloud per time step the same way.
 * pcop_process_batch_pointcloud2_windows takes a whole message stream with one pose per message and returns, in one
 * call, what the node computes for every processing callback:
 *   messages, n_messages   [n_messages] descriptors as in pcop_process_batch_pointcloud2 (layouts and memory kinds may
 *                          differ from message to message; payloads are classified per allocation)
 *   window_first           [batch + 1] (host memory): frame f is the world-frame concatenation of messages
 *                          window_first[f] .. window_first[f + 1] - 1, in message order (an empty window is a frame of
 *                          0 points)
 *   transform16            [n_messages][16] or NULL: message m's world <- sensor pose (as pcop_process_batch_pointcloud2)
 *   world_to_sensor16, sensor_to_world16, grids    [batch] poses and grids, as pcop_process_batch_pointcloud2
 *   out                    [batch]
 * out[f] equals, byte for byte, what pcop_accumulate_reset + pcop_accumulate_pointcloud2(message m, transform16 + 16 m)
 * for every m of window f in order + pcop_process_accumulated return: n_input is the window's total and crop_kept_idx
 * indexes the concatenation.  With grids, frame f's results and grid equal pcop_process_batch_occupancy(NULL, ..., batch
 * 1, world_to_sensor16 + 16 f, sensor_to_world16 + 16 f) after the same accumulation.  PCOP_OUT_DEVICE, result pointer
 * lifetime and the alternating pinned result buffers behave as in pcop_process_batch.  The accumulator is neither read
 * nor changed.  pcop_process_batch_pointcloud2 is this call with windows of one message each.
 * Errors (the handle stays usable): PCOP_ERR_BAD_PARAM for every message check of pcop_process_batch_pointcloud2, for
 * window_first[0] != 0, a decreasing window_first, window_first[batch] != n_messages, or window_first = NULL with
 * batch > 0; PCOP_ERR_CAPACITY for a window of more than max_points records or a grid above PCOP_OCC_BATCH_MAX_CELLS.
 * batch = 0 does nothing.  Every lane of the handle keeps the decode descriptors of its largest wave's messages
 * (allocated by the first call, grown, never shrunk); the decode is one launch per wave whatever its message count. */
int pcop_process_batch_pointcloud2_windows(pcop_handle* h, const pcop_pointcloud2_frame* messages, int32_t n_messages,
                                           const int32_t* window_first, int32_t batch, const float* transform16,
                                           const float* world_to_sensor16, const float* sensor_to_world16,
                                           int8_t* grids, pcop_frame_result* out);

/* Copies `bytes` from a device result array (PCOP_OUT_DEVICE) to host memory, or device to device when dst is a device
 * pointer; synchronous. */
int pcop_download(pcop_handle* h, void* dst, const void* src_device, size_t bytes);

/* bytes copied device -> host by the last call (results, counts, records; padded rows of the early remaining-cloud copy included) */
double pcop_last_d2h_bytes(const pcop_handle* h);

/*
 * Optional per-kernel timing (CUDA events around every launch, on the handle's stream).  Totals
 * accumulate over calls from the moment timing is enabled; enabling again resets them.
 */
int pcop_enable_kernel_timing(pcop_handle* h, int enable);
int pcop_kernel_timing_count(const pcop_handle* h);
int pcop_kernel_timing_get(const pcop_handle* h, int i, const char** name, double* total_us, int64_t* launches);

/*
 * Stage-isolated entry points, one per reference wrapper, so a host can swap
 * one call site at a time and tests can check each stage against the oracle
 * fed with identical inputs.  Host pointers in, host pointers out; outputs
 * must have room for `n` elements.  Each returns a status; counts come back
 * through the int32_t* arguments.
 */
int pcop_crop(pcop_handle* h, const float* xyzw, int32_t n, float* out_xyzw, int32_t* kept_idx, int32_t* m);
int pcop_voxel(pcop_handle* h, const float* xyzw, int32_t m, float* out_xyzw, uint32_t* out_keys, int32_t* v,
               uint32_t* warnings);
int pcop_sor(pcop_handle* h, const float* xyzw, int32_t v, float* out_xyzw, int32_t* kept_idx, int32_t* s,
             uint32_t* warnings);
/* pass_* arrays hold PCOP_MAX_PLANE_PASSES_RECORDED entries; inlier_idx is the last pass' inlier list. */
int pcop_plane(pcop_handle* h, const float* xyzw, int32_t s, float* remaining_xyzw, int32_t* remaining_src_idx,
               int32_t* p, int32_t* n_passes, int32_t* pass_points, int32_t* pass_inliers, float* pass_coeff,
               float* last_coeff, int32_t* inlier_idx, int32_t* n_inliers, uint32_t* warnings);
int pcop_cluster(pcop_handle* h, const float* xyzw, int32_t p, int32_t* cluster_offsets, int32_t* cluster_indices,
                 int32_t* c, int32_t* l);
int pcop_centroid_radius(pcop_handle* h, const float* xyzw, int32_t p, const int32_t* cluster_offsets,
                         const int32_t* cluster_indices, int32_t c, float* obstacles);

#ifdef __cplusplus
}
#endif
#endif /* PCOP_H_ */
