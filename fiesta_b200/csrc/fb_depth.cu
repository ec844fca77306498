// fiesta_b200 -- depth image -> point cloud on the device (SURVEY.md 8(f) "next #1": the step right before the hot path).
// Replaces Fiesta::DepthConversion (/root/reference/include/Fiesta.h:319-382): pin-hole back-projection of a uint16
// millimetre depth image and the temporal consistency filter against the previous image; the surviving points are
// compacted IN PIXEL ORDER (the order defines the ray indices of the serial ray casting that follows) and handed to the
// ray-casting kernels without leaving HBM: one 0.6 MB image goes up instead of a 3.7 MB cloud.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include "../../include/fiesta_b200.h"
#include "fb_common.cuh"

__global__ void k_depth_project(const uint16_t *img, const uint16_t *last, int rows, int cols, fiesta_depth_params p, int filter_on,
                                FbDepthRel rel, float *pts, uint8_t *flags) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)rows * cols) return;
  const int v = (int)(i / cols), u = (int)(i % cols);
  const double depth = img[i] / 1000.0;                                   // k_depth_scaling_factor (:328)
  const float px = (float)((u - p.center_x) * depth / p.focal_x), py = (float)((v - p.center_y) * depth / p.focal_y), pz = (float)depth;
  pts[3 * i] = px; pts[3 * i + 1] = py; pts[3 * i + 2] = pz;
  uint8_t keep = 1;
  if (filter_on) {                                                        // :353-378
    keep = 0;
    const bool in_margin = v >= p.depth_filter_margin && v < rows - p.depth_filter_margin && u >= p.depth_filter_margin && u < cols - p.depth_filter_margin;
    if (in_margin && !(depth > p.depth_filter_max_dist || depth < p.depth_filter_min_dist)) {
      double h[4];
#pragma unroll
      for (int r = 0; r < 4; ++r)
        h[r] = ((rel.m[4 * r] * (double)px + rel.m[4 * r + 1] * (double)py) + rel.m[4 * r + 2] * (double)pz) + rel.m[4 * r + 3] * 1.0;
      const double cx = h[0] / h[3], cy = h[1] / h[3], cz = h[2] / h[3];
      const double uu = cx * p.focal_x / cz + p.center_x, vv = cy * p.focal_y / cz + p.center_y;
      if (uu >= 0 && uu < cols && vv >= 0 && vv < rows)
        keep = fabs(last[(long long)(int)vv * cols + (int)uu] / 1000.0 - cz) < p.depth_filter_tolerance;
    }
  }
  flags[i] = keep;
}
__global__ void k_depth_gather(const float *pts, const uint32_t *sel, unsigned n, float *cloud) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = sel[i];
  cloud[3 * i] = pts[3 * s]; cloud[3 * i + 1] = pts[3 * s + 1]; cloud[3 * i + 2] = pts[3 * s + 2];
}

// d_img: this frame's image (device), d_last: previous one.  d_pts / d_cloud: rows*cols*3 floats each; d_flags rows*cols bytes;
// d_sel rows*cols u32.  Returns the number of points in d_cloud (pixel order).
cudaError_t fb_depth_to_cloud(const uint16_t *d_img, const uint16_t *d_last, int rows, int cols, const fiesta_depth_params &p, int filter_on,
                              const FbDepthRel &rel, float *d_pts, uint8_t *d_flags, uint32_t *d_sel, float *d_cloud, unsigned *d_count,
                              FbDev<uint8_t> &tmp, unsigned *h_n, cudaStream_t s) {
  const size_t N = (size_t)rows * cols;
  k_depth_project<<<(unsigned)((N + 255) / 256), 256, 0, s>>>(d_img, d_last, rows, cols, p, filter_on, rel, d_pts, d_flags);
  thrust::counting_iterator<uint32_t> it(0);
  size_t bytes = 0;
  cudaError_t e = cub::DeviceSelect::Flagged(nullptr, bytes, it, d_flags, d_sel, d_count, (int)N, s);
  if (e) return e;
  if ((e = tmp.reserve(bytes, s, false))) return e;
  if ((e = cub::DeviceSelect::Flagged(tmp.get(), bytes, it, d_flags, d_sel, d_count, (int)N, s))) return e;
  if ((e = cudaMemcpyAsync(h_n, d_count, 4, cudaMemcpyDeviceToHost, s))) return e;
  if ((e = cudaStreamSynchronize(s))) return e;
  if (*h_n) k_depth_gather<<<(*h_n + 255) / 256, 256, 0, s>>>(d_pts, d_sel, *h_n, d_cloud);
  return cudaGetLastError();
}
