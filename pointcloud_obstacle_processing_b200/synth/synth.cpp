// Synthetic LiDAR / depth-camera frame generators for the five BASELINE.json configs
// (SURVEY.md 8d).  Host-only helper used by tests and bench.py; neither oracle nor
// product.  Frames are pcl::PointXYZ arrays: {x, y, z, 1.0f}, 16-byte stride.
//
// PRNG: splitmix64 (in-repo, portable); seed = 0x5EED0000 + 4096*config + frame.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <vector>

#include "../../include/pcop.h"

namespace {

struct Rng {
  uint64_t s;
  explicit Rng(uint64_t seed) : s(seed) {}
  uint64_t next() {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  }
  double uni() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }  // [0,1)
  double uni(double a, double b) { return a + (b - a) * uni(); }
  double gauss() {
    double u1 = uni();
    if (u1 < 1e-300) u1 = 1e-300;
    return std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * uni());
  }
};

struct Box {
  double lo[3], hi[3];
};
struct Cyl {
  double cx, cy, r, z0, z1;
};
struct Sphere {
  double c[3], r;
};

struct Scene {
  std::vector<Box> boxes;
  std::vector<Cyl> cyls;
  std::vector<Sphere> spheres;
  bool ground = false;  // plane z = ground_z (normal +z)
  double ground_z = 0.0;
};

const double kInf = std::numeric_limits<double>::infinity();

double hit_box(const Box& b, const double o[3], const double d[3]) {
  double t0 = 0.0, t1 = kInf;
  for (int a = 0; a < 3; ++a) {
    if (std::fabs(d[a]) < 1e-12) {
      if (o[a] < b.lo[a] || o[a] > b.hi[a]) return kInf;
      continue;
    }
    double ta = (b.lo[a] - o[a]) / d[a], tb = (b.hi[a] - o[a]) / d[a];
    if (ta > tb) std::swap(ta, tb);
    if (ta > t0) t0 = ta;
    if (tb < t1) t1 = tb;
    if (t0 > t1) return kInf;
  }
  return t0 > 1e-6 ? t0 : kInf;
}

double hit_cyl(const Cyl& c, const double o[3], const double d[3]) {
  const double ox = o[0] - c.cx, oy = o[1] - c.cy;
  const double A = d[0] * d[0] + d[1] * d[1];
  double best = kInf;
  if (A > 1e-14) {
    const double B = ox * d[0] + oy * d[1];
    const double C = ox * ox + oy * oy - c.r * c.r;
    const double disc = B * B - A * C;
    if (disc >= 0.0) {
      const double t = (-B - std::sqrt(disc)) / A;
      if (t > 1e-6) {
        const double z = o[2] + t * d[2];
        if (z >= c.z0 && z <= c.z1) best = t;
      }
    }
  }
  if (std::fabs(d[2]) > 1e-12) {  // top cap
    const double t = (c.z1 - o[2]) / d[2];
    if (t > 1e-6 && t < best) {
      const double x = ox + t * d[0], y = oy + t * d[1];
      if (x * x + y * y <= c.r * c.r) best = t;
    }
  }
  return best;
}

double hit_sphere(const Sphere& s, const double o[3], const double d[3]) {
  const double oc[3] = {o[0] - s.c[0], o[1] - s.c[1], o[2] - s.c[2]};
  const double B = oc[0] * d[0] + oc[1] * d[1] + oc[2] * d[2];
  const double C = oc[0] * oc[0] + oc[1] * oc[1] + oc[2] * oc[2] - s.r * s.r;
  const double disc = B * B - C;
  if (disc < 0.0) return kInf;
  const double t = -B - std::sqrt(disc);
  return t > 1e-6 ? t : kInf;
}

double cast(const Scene& sc, const double o[3], const double d[3]) {
  double t = kInf;
  if (sc.ground && d[2] < -1e-12) {
    const double tg = (sc.ground_z - o[2]) / d[2];
    if (tg > 1e-6) t = tg;
  }
  for (const Box& b : sc.boxes) t = std::min(t, hit_box(b, o, d));
  for (const Cyl& c : sc.cyls) t = std::min(t, hit_cyl(c, o, d));
  for (const Sphere& s : sc.spheres) t = std::min(t, hit_sphere(s, o, d));
  return t;
}

inline void put(float* out, int i, double x, double y, double z) {
  out[4 * i + 0] = (float)x;
  out[4 * i + 1] = (float)y;
  out[4 * i + 2] = (float)z;
  out[4 * i + 3] = 1.0f;
}
inline void put_nan(float* out, int i) {
  const float q = std::numeric_limits<float>::quiet_NaN();
  out[4 * i + 0] = q;
  out[4 * i + 1] = q;
  out[4 * i + 2] = q;
  out[4 * i + 3] = 1.0f;
}

// spinning multi-beam lidar: rings x azimuths, ring-major-in-azimuth order (az outer, ring inner)
void lidar(const Scene& sc, const double origin[3], int rings, double elev_top_deg, double elev_bot_deg, int azimuths,
           double max_range, double range_sigma, double nan_frac, Rng& rng, float* out) {
  const double deg = 3.14159265358979323846 / 180.0;
  int i = 0;
  for (int a = 0; a < azimuths; ++a) {
    const double az = 2.0 * 3.14159265358979323846 * (double)a / (double)azimuths;
    for (int r = 0; r < rings; ++r, ++i) {
      const double el = (elev_top_deg + (elev_bot_deg - elev_top_deg) * (double)r / (double)(rings - 1)) * deg;
      const double d[3] = {std::cos(el) * std::cos(az), std::cos(el) * std::sin(az), std::sin(el)};
      double t = cast(sc, origin, d);
      const bool drop = rng.uni() < nan_frac;
      const double noise = rng.gauss() * range_sigma;
      if (drop || !(t < max_range)) {
        put_nan(out, i);
        continue;
      }
      t += noise;
      put(out, i, origin[0] + t * d[0], origin[1] + t * d[1], origin[2] + t * d[2]);
    }
  }
}

// config 1: VLP-16-style 30 000 returns inside the params.yaml arena
void gen_vlp16(uint64_t seed, float* out) {
  Rng rng(seed);
  Scene sc;
  sc.ground = true;
  sc.ground_z = 0.0;
  // arena walls just inside the crop box [0,4.5]x[0,3.78]
  sc.boxes.push_back({{0.02, 0.02, 0.0}, {0.06, 3.76, 0.6}});
  sc.boxes.push_back({{4.44, 0.02, 0.0}, {4.48, 3.76, 0.6}});
  sc.boxes.push_back({{0.02, 0.02, 0.0}, {4.48, 0.06, 0.6}});
  sc.boxes.push_back({{0.02, 3.72, 0.0}, {4.48, 3.76, 0.6}});
  const double origin[3] = {rng.uni(1.8, 2.6), rng.uni(1.5, 2.3), 0.3};
  const int nobj = 5 + (int)(rng.uni() * 6.0);
  for (int k = 0; k < nobj; ++k) {
    double cx, cy;
    do {
      cx = rng.uni(0.4, 4.1);
      cy = rng.uni(0.4, 3.4);
    } while (std::hypot(cx - origin[0], cy - origin[1]) < 0.7);
    const double sz = rng.uni(0.1, 0.4);
    if (rng.uni() < 0.5)
      sc.boxes.push_back({{cx - sz / 2, cy - sz / 2, 0.0}, {cx + sz / 2, cy + sz / 2, rng.uni(0.1, 0.4)}});
    else
      sc.cyls.push_back({cx, cy, sz / 2, 0.0, rng.uni(0.1, 0.4)});
  }
  lidar(sc, origin, 16, 15.0, -15.0, 1875, 100.0, 0.005, 0.01, rng, out);
}

// config 2/5: HDL-64-style 120 000 returns
void gen_hdl64(uint64_t seed, float* out) {
  Rng rng(seed);
  Scene sc;
  sc.ground = true;
  sc.ground_z = 0.0;
  const double origin[3] = {0.0, 0.0, 1.73};
  const int ncars = 12 + (int)(rng.uni() * 14.0);
  for (int k = 0; k < ncars; ++k) {
    double cx, cy;
    do {
      cx = rng.uni(-38.0, 38.0);
      cy = rng.uni(-38.0, 38.0);
    } while (std::hypot(cx, cy) < 5.0);
    const bool rot = rng.uni() < 0.5;
    const double lx = rot ? 1.8 : 4.0, ly = rot ? 4.0 : 1.8;
    sc.boxes.push_back({{cx - lx / 2, cy - ly / 2, 0.0}, {cx + lx / 2, cy + ly / 2, 1.5}});
  }
  const int ncyl = 8 + (int)(rng.uni() * 8.0);
  for (int k = 0; k < ncyl; ++k) {
    double cx, cy;
    do {
      cx = rng.uni(-30.0, 30.0);
      cy = rng.uni(-30.0, 30.0);
    } while (std::hypot(cx, cy) < 3.0);
    sc.cyls.push_back({cx, cy, 0.3, 0.0, 1.7});
  }
  lidar(sc, origin, 64, 2.0, -24.8, 1875, 80.0, 0.02, 0.0, rng, out);
}

// config 3: organized 640x480 depth image, camera frame (x right, y down, z forward)
// config 3's scene seen by a pinhole camera of W x H pixels: point v * W + u is pixel (u, v) in the camera frame
void gen_depth_camera(uint64_t seed, int W, int H, double fx, double fy, double cx, double cy, float* out) {
  Rng rng(seed);
  // build the scene in a z-up world, camera at the origin looking along world +x:
  //   cam z = world x, cam x = -world y, cam y = -world z
  Scene sc;
  sc.ground = true;
  sc.ground_z = -1.0;                                         // floor 1 m below the camera
  sc.boxes.push_back({{4.0, -6.0, -1.0}, {4.2, 6.0, 3.0}});   // back wall at z_cam = 4.0
  const int nobj = 10 + (int)(rng.uni() * 11.0);
  for (int k = 0; k < nobj; ++k) {
    const double wx = rng.uni(1.2, 3.6), wy = rng.uni(-1.8, 1.8), sz = rng.uni(0.12, 0.35);
    if (rng.uni() < 0.5)
      sc.boxes.push_back({{wx - sz / 2, wy - sz / 2, -1.0}, {wx + sz / 2, wy + sz / 2, -1.0 + rng.uni(0.15, 0.5)}});
    else
      sc.spheres.push_back({{wx, wy, -1.0 + sz / 2}, sz / 2});
  }
  const double o[3] = {0.0, 0.0, 0.0};
  int i = 0;
  for (int v = 0; v < H; ++v)
    for (int u = 0; u < W; ++u, ++i) {
      const double xc = ((double)u - cx) / fx, yc = ((double)v - cy) / fy;  // cam ray (xc, yc, 1)
      const double dw[3] = {1.0, -xc, -yc};                                 // world dir, un-normalised
      const double nrm = std::sqrt(dw[0] * dw[0] + dw[1] * dw[1] + dw[2] * dw[2]);
      const double d[3] = {dw[0] / nrm, dw[1] / nrm, dw[2] / nrm};
      const double t = cast(sc, o, d);
      const bool drop = rng.uni() < 0.10;
      const double g = rng.gauss();
      if (drop || !(t < 50.0)) {
        put_nan(out, i);
        continue;
      }
      double z = t * d[0];  // depth along the optical axis
      z += g * 0.0012 * z * z;
      if (!(z > 0.5 && z < 4.5)) {
        put_nan(out, i);
        continue;
      }
      put(out, i, xc * z, yc * z, z);
    }
}

void gen_depth(uint64_t seed, float* out) { gen_depth_camera(seed, 640, 480, 525.0, 525.0, 319.5, 239.5, out); }

// config 4: adversarial 1 M points: 3 dense blobs + a 50 k-point snake + 50 k noise
void gen_adversarial(uint64_t seed, float* out, int n) {
  Rng rng(seed);
  int i = 0;
  const int side = 67;  // 67^3 = 300 763 points per blob
  const double blob_org[3][3] = {{1.0, 1.0, 0.5}, {6.0, 2.0, 0.5}, {3.0, 12.0, 0.5}};
  const int n_snake = 50000, n_noise = 50000;
  const int n_blob_total = n - n_snake - n_noise;
  for (int b = 0; b < 3 && i < n_blob_total; ++b)
    for (int a = 0; a < side && i < n_blob_total; ++a)
      for (int c = 0; c < side && i < n_blob_total; ++c)
        for (int e = 0; e < side && i < n_blob_total; ++e, ++i)
          put(out, i, blob_org[b][0] + 0.02 * a + rng.uni(-0.004, 0.004),
              blob_org[b][1] + 0.02 * c + rng.uni(-0.004, 0.004),
              blob_org[b][2] + 0.02 * e + rng.uni(-0.004, 0.004));
  // any remainder of the blob budget goes to noise
  const int noise_extra = n_blob_total - i;
  // snake: Archimedean spiral in the plane z = 5, arc step 0.045 (0.9 * tol), turn spacing 0.1 (2 * tol)
  {
    double theta = 2.0 * 3.14159265358979323846 * 5.0;  // start at r = 0.5
    const double pitch = 0.1 / (2.0 * 3.14159265358979323846);
    for (int k = 0; k < n_snake; ++k, ++i) {
      const double r = pitch * theta;
      put(out, i, 9.0 + r * std::cos(theta), 9.0 + r * std::sin(theta), 5.0);
      theta += 0.045 / r;
    }
  }
  for (int k = 0; k < n_noise + noise_extra; ++k, ++i)
    put(out, i, rng.uni(0.0, 18.0), rng.uni(0.0, 18.0), rng.uni(0.0, 5.8));
  // shuffle so that index order carries no spatial structure (Fisher-Yates)
  for (int k = n - 1; k > 0; --k) {
    const int j = (int)(rng.next() % (uint64_t)(k + 1));
    float tmp[4];
    std::memcpy(tmp, out + 4 * k, 16);
    std::memcpy(out + 4 * k, out + 4 * j, 16);
    std::memcpy(out + 4 * j, tmp, 16);
  }
}

void base_params(pcop_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->plane_axis[0] = 0.0f;
  p->plane_axis[1] = 0.0f;
  p->plane_axis[2] = 1.0f;
  p->plane_keep_fraction = 0.3;
  p->plane_max_iterations = 50;
  p->plane_probability = 0.99;
  p->ransac_seed = 12345u;
  p->optimize_coefficients = 1;
  p->plane_segment_angle = 20;
  p->statistical_outlier_meanK = 15;
  p->statistical_outlier_stdDevThres = 4.0f;
  p->enable_crop = 1;
  p->enable_voxel = 1;
  p->enable_sor = 0;
  p->enable_plane = 1;
  p->enable_cluster = 1;
  p->outputs = PCOP_OUT_DEFAULT;
  p->accumulate_count = 1;
  p->block_size = 0.0375f;
  p->dev_percent = 0.9f;
  p->downsample_input_data = 1;
  p->passthrough_filter_enable = 1;
  p->convex_hull_alpha = 180.0f;
}

}  // namespace

extern "C" {

// number of points of one frame of `config` (1..5)
int32_t pcop_synth_points(int config) {
  switch (config) {
    case 1: return 30000;
    case 2: return 120000;
    case 3: return 640 * 480;
    case 4: return 1000000;
    case 5: return 120000;
    default: return 0;
  }
}

uint64_t pcop_synth_seed(int config, int frame) {
  return 0x5EED0000ull + 4096ull * (uint64_t)config + (uint64_t)frame;
}

// fills out[points*4]; returns the number of points or -1
int32_t pcop_synth_frame(int config, int frame, float* out) {
  const uint64_t seed = pcop_synth_seed(config, frame);
  switch (config) {
    case 1: gen_vlp16(seed, out); break;
    case 2: gen_hdl64(seed, out); break;
    case 3: gen_depth(seed, out); break;
    case 4: gen_adversarial(seed, out, 1000000); break;
    case 5: gen_hdl64(pcop_synth_seed(2, frame), out); break;  // config 5 = batch of config-2 frames
    default: return -1;
  }
  return pcop_synth_points(config);
}

// config 3's scene of frame `frame` through another pinhole camera (W x H points into out[W * H * 4])
void pcop_synth_depth_camera(int frame, int W, int H, double fx, double fy, double cx, double cy, float* out) {
  gen_depth_camera(pcop_synth_seed(3, frame), W, H, fx, fy, cx, cy, out);
}

// the parameter set each config runs with (SURVEY 8d table)
int pcop_synth_params(int config, pcop_params* p) {
  base_params(p);
  switch (config) {
    case 1:  // params.yaml verbatim
      p->x_min = 0.0f; p->x_max = 4.5f; p->y_min = 0.0f; p->y_max = 3.78f; p->z_min = -0.5f; p->z_max = 0.25f;
      p->downsample_size = 0.015f;
      p->enable_sor = 1;
      p->plane_segment_dist_thres = 0.040f;
      p->euc_cluster_tolerance = 0.4f; p->euc_min_cluster_size = 5; p->euc_max_cluster_size = 20000;
      p->accumulate_count = 200;
      p->publish_point_clouds = 1;
      break;
    case 2:
    case 5:
      p->x_min = -40.0f; p->x_max = 40.0f; p->y_min = -40.0f; p->y_max = 40.0f; p->z_min = -2.5f; p->z_max = 1.5f;
      p->downsample_size = 0.1f;
      p->plane_segment_dist_thres = 0.2f;
      p->euc_cluster_tolerance = 0.5f; p->euc_min_cluster_size = 10; p->euc_max_cluster_size = 100000;
      break;
    case 3:
      p->x_min = -10.0f; p->x_max = 10.0f; p->y_min = -10.0f; p->y_max = 10.0f; p->z_min = 0.3f; p->z_max = 4.5f;
      p->downsample_size = 0.02f;
      p->plane_segment_dist_thres = 0.03f;
      p->euc_cluster_tolerance = 0.05f; p->euc_min_cluster_size = 50; p->euc_max_cluster_size = 307200;
      break;
    case 4:
      p->x_min = -1.0f; p->x_max = 19.0f; p->y_min = -1.0f; p->y_max = 19.0f; p->z_min = -1.0f; p->z_max = 7.0f;
      p->downsample_size = 0.01f;
      p->enable_plane = 0;
      p->plane_segment_dist_thres = 0.05f;
      p->euc_cluster_tolerance = 0.05f; p->euc_min_cluster_size = 5; p->euc_max_cluster_size = 1000000;
      break;
    default: return -1;
  }
  return 0;
}

}  // extern "C"
