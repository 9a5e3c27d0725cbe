// Micro-benchmark: host time of classifying the payload pointers of one batched PointCloud2 call, one
// cudaPointerGetAttributes per message (is_device_pointer) against one driver query per allocation (PayloadClassifier),
// both as the library compiles them.  Payloads as a caller lays them out: n messages of `bytes` bytes in one device
// allocation, in one pinned host allocation, and in pageable memory.  Prints one JSON line (median / min / max of 7 runs,
// microseconds per call).  tools/pointcloud2_windows_bench.py builds and runs it.
//   payload_classify <messages> <bytes per message>
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../pointcloud_obstacle_processing_b200/csrc/handle.cuh"

template <class F>
static void timed(const char* name, F fn, bool last) {
  std::vector<double> us;
  int dev = 0;
  for (int r = 0; r < 8; ++r) {
    const auto a = std::chrono::steady_clock::now();
    dev = fn();
    const double t = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - a).count();
    if (r > 0) us.push_back(t);  // (the first run loads the entry point)
  }
  std::sort(us.begin(), us.end());
  printf("\"%s\": {\"median\": %.2f, \"min\": %.2f, \"max\": %.2f, \"runs\": %zu, \"device\": %d}%s", name, us[us.size() / 2],
         us.front(), us.back(), us.size(), dev, last ? "" : ", ");
}

int main(int argc, char** argv) {
  const int n = argc > 1 ? atoi(argv[1]) : 1024;
  const size_t bytes = argc > 2 ? (size_t)atoll(argv[2]) : 4096;
  unsigned char *d = nullptr, *p = nullptr;
  if (cudaMalloc((void**)&d, n * bytes) != cudaSuccess || cudaHostAlloc((void**)&p, n * bytes, 0) != cudaSuccess) {
    fprintf(stderr, "payload_classify: no CUDA device\n");
    return 1;
  }
  std::vector<unsigned char> q(n * bytes);
  printf("{\"messages\": %d, \"bytes_per_message\": %zu, ", n, bytes);
  const struct { const char* name; unsigned char* base; } kinds[3] = {{"device", d}, {"pinned", p}, {"pageable", q.data()}};
  for (int k = 0; k < 3; ++k) {
    unsigned char* base = kinds[k].base;
    printf("\"%s\": {", kinds[k].name);
    timed("per_message", [&] {
      int c = 0;
      for (int m = 0; m < n; ++m) c += pcop::is_device_pointer(base + m * bytes);
      return c;
    }, false);
    timed("per_allocation", [&] {
      pcop::PayloadClassifier on_device;
      int c = 0;
      for (int m = 0; m < n; ++m) c += on_device(base + m * bytes);
      return c;
    }, true);
    printf("}%s", k < 2 ? ", " : "}\n");
  }
  cudaFree(d);
  cudaFreeHost(p);
  return 0;
}
