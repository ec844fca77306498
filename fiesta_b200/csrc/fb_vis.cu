// fiesta_b200 -- device-side visualisation extraction (SURVEY.md 8(f) "next #2"): the step right after the hot path.
// Replaces the full-box triple loops of ESDFMap::GetPointCloud (/root/reference/src/ESDFMap.cpp:544-582) and
// ESDFMap::GetSliceMarker + RainbowColorMap (:584-699) with a flag pass + ordered stream compaction (CUB), so only the
// selected points cross PCIe.  Output order = the reference's loop order (x, then y, then z = increasing linear index).
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include "../../include/fiesta_b200.h"
#include "fb_common.cuh"

__global__ void k_vis_occ_flags(FbGeom g, const double *occ, double l_occ, int zlo, int zhi, uint8_t *flags) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= g.total) return;
  const int x = (int)(idx / g.gyz), y = (int)(idx % g.gyz / g.gz), z = (int)(idx % g.gz);
  // `if (!Exist(...) || z < vis_lower_bound || z > vis_upper_bound) continue;` inside the update box (:565-569)
  flags[idx] = fb_in_range(g, x, y, z) && z >= zlo && z <= zhi && occ[fb_ii(g, x, y, z)] > l_occ;
}
__global__ void k_vis_occ_points(FbGeom g, const uint32_t *sel, unsigned n, float *out) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long idx = sel[i];
  const int v[3] = {(int)(idx / g.gyz), (int)(idx % g.gyz / g.gz), (int)(idx % g.gz)};
#pragma unroll
  for (int k = 0; k < 3; ++k) out[3 * i + k] = (float)((v[k] + 0.5) * g.res + g.origin[k]);   // Vox2Pos (:79-82), Point32 is float
}
__device__ __forceinline__ double fb_slice_dist(const FbGeom &g, const uint32_t *cobs, int x, int y, int z) {
  const uint32_t raw = cobs[fb_ii(g, x, y, z)], c = raw & FB_CODE_MASK;
  if (c == FB_UNKNOWN) return -10000.0;
  if (c == FB_INF || (raw & FB_DINF)) return 10000.0;
  int ox, oy, oz; fb_unpack(c, ox, oy, oz);
  const double dx = (double)(ox - x), dy = (double)(oy - y), dz = (double)(oz - z);
  return sqrt((dx * dx + dy * dy) + dz * dz) * g.res;
}
__global__ void k_vis_slice_flags(FbGeom g, const uint32_t *cobs, int slice, uint8_t *flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.gx * g.gy) return;
  const int x = i / g.gy, y = i % g.gy;
  bool on = x >= g.min_vec[0] && x <= g.max_vec[0] && y >= g.min_vec[1] && y <= g.max_vec[1];
  if (on) { const double d = fb_slice_dist(g, cobs, x, y, slice); on = !(d < 0 || d >= 10000.0); }   // (:682-683)
  flags[i] = on;
}
__global__ void k_vis_slice_points(FbGeom g, const uint32_t *cobs, const uint32_t *sel, unsigned n, int slice, double max_dist, double *xyz, float *rgba) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int x = sel[i] / g.gy, y = sel[i] % g.gy;
  const int v[3] = {x, y, slice};
#pragma unroll
  for (int k = 0; k < 3; ++k) xyz[3 * i + k] = (v[k] + 0.5) * g.res + g.origin[k];
  const double d = fb_slice_dist(g, cobs, x, y, slice);
  // RainbowColorMap(h), s = v = 1 (:584-637)
  double h = d <= max_dist ? d / max_dist : 1;
  h -= floor(h);
  h *= 6;
  const int k6 = (int)floor(h);
  double f = h - k6;
  if (!(k6 & 1)) f = 1 - f;
  const double mm = 1.0 * (1 - 1.0), nn = 1.0 * (1 - 1.0 * f), vv = 1.0;
  double r = 1, gg = 0.5, b = 0.5;
  switch (k6) {
    case 6: case 0: r = vv; gg = nn; b = mm; break;
    case 1: r = nn; gg = vv; b = mm; break;
    case 2: r = mm; gg = vv; b = nn; break;
    case 3: r = mm; gg = nn; b = vv; break;
    case 4: r = nn; gg = mm; b = vv; break;
    case 5: r = vv; gg = mm; b = nn; break;
    default: break;
  }
  rgba[4 * i] = (float)r; rgba[4 * i + 1] = (float)gg; rgba[4 * i + 2] = (float)b; rgba[4 * i + 3] = 1.0f;
}

static cudaError_t vis_select(const uint8_t *flags, size_t n, uint32_t *sel, unsigned *count, cudaStream_t s) {
  FbDev<unsigned> d_cnt; FbDev<uint8_t> tmp; size_t bytes = 0;
  cudaError_t e = d_cnt.alloc(1);
  if (e) return e;
  thrust::counting_iterator<uint32_t> it(0);
  e = cub::DeviceSelect::Flagged(nullptr, bytes, it, flags, sel, d_cnt.get(), (int)n, s);
  if (!e) e = tmp.alloc(bytes ? bytes : 16);
  if (!e) e = cub::DeviceSelect::Flagged(tmp.get(), bytes, it, flags, sel, d_cnt.get(), (int)n, s);
  if (!e) e = cudaMemcpyAsync(count, d_cnt, 4, cudaMemcpyDeviceToHost, s);
  if (!e) e = cudaStreamSynchronize(s);
  return e;
}

cudaError_t fb_vis_point_cloud(const FbGeom &g, const double *occ, double l_occ, int zlo, int zhi, float *h_out, long long cap, long long *count, cudaStream_t s) {
  const size_t G = (size_t)g.total;
  FbDev<uint8_t> flags; FbDev<uint32_t> sel; FbDev<float> pts;
  cudaError_t e = flags.alloc(G);
  if (!e) e = sel.alloc(G);
  unsigned n = 0;
  if (!e) { k_vis_occ_flags<<<(unsigned)((G + 255) / 256), 256, 0, s>>>(g, occ, l_occ, zlo, zhi, flags); e = vis_select(flags, G, sel, &n, s); }
  *count = n;
  const unsigned m = (long long)n < cap ? n : (unsigned)(cap < 0 ? 0 : cap);
  if (!e && m) {
    e = pts.alloc((size_t)m * 3);
    if (!e) { k_vis_occ_points<<<(m + 255) / 256, 256, 0, s>>>(g, sel, m, pts); e = cudaMemcpyAsync(h_out, pts, (size_t)m * 12, cudaMemcpyDeviceToHost, s); }
    if (!e) e = cudaStreamSynchronize(s);
  }
  return e;
}

cudaError_t fb_vis_slice(const FbGeom &g, const uint32_t *cobs, int slice, double max_dist, double *h_xyz, float *h_rgba, long long cap, long long *count, cudaStream_t s) {
  *count = 0;
  if (slice < 0 || slice >= g.gz) return cudaSuccess;
  const size_t G = (size_t)g.gx * g.gy;
  FbDev<uint8_t> flags; FbDev<uint32_t> sel; FbDev<double> xyz; FbDev<float> rgba;
  cudaError_t e = flags.alloc(G);
  if (!e) e = sel.alloc(G);
  unsigned n = 0;
  if (!e) { k_vis_slice_flags<<<(unsigned)((G + 255) / 256), 256, 0, s>>>(g, cobs, slice, flags); e = vis_select(flags, G, sel, &n, s); }
  *count = n;
  const unsigned m = (long long)n < cap ? n : (unsigned)(cap < 0 ? 0 : cap);
  if (!e && m) {
    e = xyz.alloc((size_t)m * 3);
    if (!e) e = rgba.alloc((size_t)m * 4);
    if (!e) {
      k_vis_slice_points<<<(m + 255) / 256, 256, 0, s>>>(g, cobs, sel, m, slice, max_dist, xyz, rgba);
      e = cudaMemcpyAsync(h_xyz, xyz, (size_t)m * 24, cudaMemcpyDeviceToHost, s);
      if (!e) e = cudaMemcpyAsync(h_rgba, rgba, (size_t)m * 16, cudaMemcpyDeviceToHost, s);
    }
    if (!e) e = cudaStreamSynchronize(s);
  }
  return e;
}
