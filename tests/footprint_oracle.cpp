// ORACLE -- test infrastructure only.  The obstacle footprints of include/pcop.h (PCOP_OUT_FOOTPRINTS) restated for
// the host: the totalOrder box and Andrew's monotone chain over Shewchuk's filtered orient2d (the double evaluation with
// the ccwerrboundA filter, then an exact expansion; TwoProduct on std::fma).  The independent restatement in
// footprint_util.py (exact integers, quickhull) pins the same semantics.  Built like the pipeline oracle (g++ -O2
// -ffp-contract=off -fno-fast-math), so every double op is rounded in turn and none is contracted.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

namespace {

void two_sum(double a, double b, double& x, double& y) {
  x = a + b;
  const double bv = x - a, av = x - bv;
  y = (a - av) + (b - bv);
}
void two_diff(double a, double b, double& x, double& y) {
  x = a - b;
  const double bv = a - x, av = x + bv;
  y = (a - av) + (bv - b);
}
void two_product(double a, double b, double& x, double& y) {
  x = a * b;
  y = std::fma(a, b, -x);
}

// sign-carrying value of (ax - cx)(by - cy) - (ay - cy)(bx - cx) (Shewchuk's orient2d, the exact stage without the
// intermediate adaptive stages: every product of the exact differences into one nonoverlapping expansion)
double orient2d(double ax, double ay, double bx, double by, double cx, double cy) {
  const double detleft = (ax - cx) * (by - cy), detright = (ay - cy) * (bx - cx);
  const double det = detleft - detright;
  double detsum;
  if (detleft > 0.0) {
    if (detright <= 0.0) return det;
    detsum = detleft + detright;
  } else if (detleft < 0.0) {
    if (detright >= 0.0) return det;
    detsum = -detleft - detright;
  } else {
    return det;
  }
  const double ccwerrboundA = (3.0 + 16.0 * 0x1p-53) * 0x1p-53;
  const double errbound = ccwerrboundA * detsum;
  if (det >= errbound || -det >= errbound) return det;
  double d[4][2];  // the four differences, each as value + tail
  two_diff(ax, cx, d[0][0], d[0][1]);
  two_diff(by, cy, d[1][0], d[1][1]);
  two_diff(ay, cy, d[2][0], d[2][1]);
  two_diff(bx, cx, d[3][0], d[3][1]);
  std::vector<double> e;
  auto grow = [&](double q) {
    std::vector<double> h;
    for (double ei : e) {
      double x, y;
      two_sum(q, ei, x, y);
      q = x;
      if (y != 0.0) h.push_back(y);
    }
    if (q != 0.0) h.push_back(q);
    e.swap(h);
  };
  for (int i = 0; i < 2; ++i)
    for (int j = 0; j < 2; ++j) {
      double x, y;
      two_product(d[0][i], d[1][j], x, y);
      grow(y);
      grow(x);
      two_product(-d[2][i], d[3][j], x, y);
      grow(y);
      grow(x);
    }
  return e.empty() ? 0.0 : e.back();
}

uint32_t total_order_key(float f) {
  uint32_t u;
  std::memcpy(&u, &f, 4);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
float from_key(uint32_t k) {
  const uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  float f;
  std::memcpy(&f, &u, 4);
  return f;
}

struct P {
  float x, y;
  int32_t i;
};

}  // namespace

extern "C" double pcop_oracle_orient2d(float ax, float ay, float bx, float by, float cx, float cy) {
  return orient2d(ax, ay, bx, by, cx, cy);
}

// pcop_cluster_footprints on the host (arguments validated by the caller)
extern "C" int pcop_oracle_cluster_footprints(const float* xyzw, int32_t p, const int32_t* offsets, const int32_t* indices,
                                              int32_t c, float* boxes, int32_t* hull_offsets, int32_t* hull_indices,
                                              int32_t* n_hull) {
  (void)p;
  int32_t h = 0;
  for (int32_t k = 0; k < c; ++k) {
    hull_offsets[k] = h;
    const int32_t b = offsets[k], n = offsets[k + 1] - b;
    float* box = boxes + 8 * (size_t)k;
    std::memset(box, 0, 32);
    if (n == 0) continue;
    if (n == 1) {  // a singleton: its member copied, whatever it holds
      const float* q = xyzw + 4 * (size_t)indices[b];
      box[0] = box[4] = q[0];
      box[1] = box[5] = q[1];
      box[2] = box[6] = q[2];
      hull_indices[h++] = indices[b];
      continue;
    }
    uint32_t mn[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, mx[3] = {0u, 0u, 0u};
    std::vector<P> pts((size_t)n);
    for (int32_t j = 0; j < n; ++j) {
      const float* q = xyzw + 4 * (size_t)indices[b + j];
      for (int a = 0; a < 3; ++a) {
        mn[a] = std::min(mn[a], total_order_key(q[a]));
        mx[a] = std::max(mx[a], total_order_key(q[a]));
      }
      pts[(size_t)j] = P{q[0], q[1], indices[b + j]};
    }
    for (int a = 0; a < 3; ++a) {
      box[a] = from_key(mn[a]);
      box[4 + a] = from_key(mx[a]);
    }
    std::sort(pts.begin(), pts.end(), [](const P& u, const P& v) {
      if (u.x != v.x) return u.x < v.x;
      if (u.y != v.y) return u.y < v.y;
      return u.i < v.i;
    });
    std::vector<P> u;  // distinct (x, y), smallest index of each
    for (const P& q : pts)
      if (u.empty() || !(u.back().x == q.x && u.back().y == q.y)) u.push_back(q);
    auto turn = [](const P& a, const P& b2, const P& q) { return orient2d(a.x, a.y, b2.x, b2.y, q.x, q.y); };
    std::vector<P> st;
    for (const P& q : u) {
      while (st.size() >= 2 && turn(st[st.size() - 2], st.back(), q) <= 0.0) st.pop_back();
      st.push_back(q);
    }
    if (u.size() > 1) {
      const size_t lower = st.size();
      for (size_t j = u.size() - 1; j-- > 0;) {
        while (st.size() > lower && turn(st[st.size() - 2], st.back(), u[j]) <= 0.0) st.pop_back();
        st.push_back(u[j]);
      }
      st.pop_back();  // the first point again
    }
    for (const P& q : st) hull_indices[h++] = q.i;
  }
  hull_offsets[c] = h;
  *n_hull = h;
  return 0;
}
