// fiesta_b200 -- C ABI (include/fiesta_b200.h), host-side map state, and the occupancy / query / export kernels.
//
// Host code mirrors what the reference does on the caller's thread with pure arithmetic (index conversions,
// update-range bookkeeping, sentinel returns: /root/reference/src/ESDFMap.cpp:46-118, 401-421, 792-824) and hands every
// per-voxel operation to the device.  There is NO CPU fallback: fiesta_create fails without an sm_100 device.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <memory>
#include <new>
#include "../../include/fiesta_b200.h"
#include "fb_common.cuh"
#include "fb_exact.h"

static thread_local std::string g_last_error;
static void set_error(const char *fmt, const char *a = "", const char *b = "") {
  char buf[512];
  snprintf(buf, sizeof(buf), fmt, a, b);
  g_last_error = buf;
}
#define CK(call)                                                                         \
  do {                                                                                   \
    cudaError_t e__ = (call);                                                            \
    if (e__ != cudaSuccess) { set_error("%s failed: %s", #call, cudaGetErrorString(e__)); return FIESTA_ERR_CUDA; } \
  } while (0)

struct fiesta_map {
  FbGeom g;
  int device;
  cudaStream_t stream;
  bool params_set;
  double l_hit, l_miss, l_min, l_max, l_occ;
  double l_cornor[3], r_cornor[3];
  // per-voxel state
  FbDev<uint32_t> cobs, cobs_b, stamp[2], occbits;
  FbDev<double> occ;
  FbDev<unsigned long long> cnt;
  // tiles
  FbDev<uint32_t> tile_flag, nb_flag, list[2], changed[2], changed_bbox[2];
  CUtensorMap tmap;
  int wf_blocks, rr_blocks;
  // queues
  FbDev<uint32_t> touch_flag, touch_list;
  unsigned touch_epoch;
  FbDev<uint32_t> ins, del;
  unsigned n_touch_tiles, n_ins, n_del;  // host view (valid after the last sync)
  FbDev<FbCounters> d_ctr;
  FbPinned<FbCounters> h_ctr;
  // per-call SetOccupancy staging
  FbPinned<uint32_t> h_ev;
  FbDev<uint32_t> d_ev;
  size_t n_ev;
  // ray casting
  FbDev<float> d_xyz;
  FbDev<uint32_t> ray_list;
  FbDev<int> ray_len, ray_reach;
  FbDev<unsigned> ray_dirty;
  unsigned frame_tag, owner_tag;
  // queries
  FbDev<double> d_qin, d_qout;
  cudaEvent_t ev[4];
  FbDev<unsigned long long> d_dbg;
  // depth front end (next #1): sized exactly for cap_img pixels
  FbDev<uint16_t> d_img[2]; size_t cap_img; unsigned image_cnt;
  FbDev<float> d_dpts, d_dcloud; FbDev<uint8_t> d_dflags; FbDev<uint32_t> d_dsel; FbDev<unsigned> d_dcount; FbDev<uint8_t> d_dtmp; unsigned last_cloud_n;
  int mode;
  int shard_rank, shard_world, tile_x_lo, tile_x_hi;
  FbDev<unsigned> d_halo_changed;
  FbExact X;
  fiesta_stats st;
  // pinned host mirror (next #3): union of the update boxes that were current while records could change
  struct fiesta_host_mirror *mirror;
  int dirty_lo[3], dirty_hi[3];
  bool dirty_any, pending_obs;      // pending_obs: observations counted under the current box and not integrated yet
  // No constructor, so `new fiesta_map()` zero-fills every plain member.  The buffers free themselves after this body.
  ~fiesta_map() {
    for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
    if (stream) cudaStreamDestroy(stream);
  }
};
static void mark_dirty(fiesta_map *m) {                                   // tracked without a mirror too: events staged before a mirror is
  const FbGeom &g = m->g;                                                   // created are integrated after it
  for (int i = 0; i < 3; ++i) {
    if (!m->dirty_any || g.min_vec[i] < m->dirty_lo[i]) m->dirty_lo[i] = g.min_vec[i];
    if (!m->dirty_any || g.max_vec[i] > m->dirty_hi[i]) m->dirty_hi[i] = g.max_vec[i];
  }
  m->dirty_any = true;
}

// ====================================================================== kernels
__global__ void k_reset_ray_ctr(FbCounters *c) {
  c->ray_work[0] = c->ray_work[1] = c->ray_work[2] = 0u;
  c->rays_cast = c->rays_dropped = c->ray_rounds = c->ray_error = 0;
  c->ray_voxels = 0;
}
__global__ void k_reset_esdf_ctr(FbCounters *c) {
  c->n_changed[0] = c->n_changed[1] = 0;
  c->next_work[0] = c->next_work[1] = c->next_work[2] = c->next_work[3] = 0;
  c->generations = 0;
  c->voxels_changed = c->voxels_reset = c->tile_visits = 0;
}
__global__ void k_reset_touched(FbCounters *c) { c->n_touched = 0; }
__global__ void k_reset_queues(FbCounters *c, int touched, int insdel) {
  if (touched) c->n_touch_tiles = 0;
  if (insdel) c->n_ins = c->n_del = 0;
}

// occupancy bitmap = Exist(idx) for every voxel (ESDFMap.cpp:46-48) under a new occupancy threshold
__global__ void k_rebuild_occbits(const double *occ, long long ptotal, double l_occ, uint32_t *occbits) {
  const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (w * 32 >= ptotal) return;
  uint32_t bits = 0;
  for (int k = 0; k < 32; ++k) { const long long v = w * 32 + k; if (v < ptotal && occ[v] > l_occ) bits |= 1u << k; }
  occbits[w] = bits;
}

// O1 counter part for per-call SetOccupancy events staged on the host (ESDFMap.cpp:424-435).
__global__ void k_apply_events(FbGeom g, const uint32_t *ev, size_t n, FbTouch t, unsigned long long key_base) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t e = ev[i];
  fb_touch(g, t, e & 0x7fffffffu, e >> 31, key_base + i);       // the i-th staged call = its position in the serial order
}

// SetOccupancy(Vector3i, occ) for events that are already on the device (ESDFMap.cpp:417-437).
__global__ void k_apply_vox_events(FbGeom g, const int *vox, const uint8_t *occ, long long n, FbTouch t) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int x = vox[3 * i], y = vox[3 * i + 1], z = vox[3 * i + 2];
  if (!fb_in_range(g, x, y, z) || !fb_in_grid(g, x, y, z)) return;       // `if (!VoxInRange(vox)) return idx;` (:420-421)
  fb_touch(g, t, (unsigned)fb_ii(g, x, y, z), occ[i] & 1u, 0ull);
}

// O2: ESDFMap::UpdateOccupancy (ESDFMap.cpp:235-271).  One 128-thread CTA streams the counters of one queued 8^3 tile
// (4 voxels = one 32-byte sector per thread); every voxel with pending observations is integrated exactly as the
// reference does.  Voxels are independent, so the queue order does not matter for the result.
// EXACT = order-exact mode: only the ORDER of the insert_queue_ / delete_queue_ pushes depends on the voxel's place in
// occupancy_queue_ (:263-267), so the few voxels that cross the threshold are emitted together with the serial time of their
// first observation (hundreds per LIDAR frame, against millions of touched voxels) and sorted afterwards; the local-map
// reset keeps the closest obstacle (flag bit FB_DINF, :256-259).
template <bool EXACT>
__global__ void __launch_bounds__(128) k_integrate(FbGeom g, const uint32_t *tiles, unsigned ntiles, unsigned long long *cnt, double *occ,
                                                   uint32_t *cobs, uint32_t *occbits, uint32_t *ins, uint32_t *del, unsigned *n_ins, unsigned *n_del,
                                                   FbCounters *ctr, const unsigned long long *tkey, unsigned long long *ins_key,
                                                   unsigned long long *del_key, int global_map, double l_hit, double l_miss, double l_min,
                                                   double l_max, double l_occ) {
  const int row = threadIdx.x >> 1, half = threadIdx.x & 1;
  const int lx = row >> 3, ly = row & 7;
  unsigned touched = 0;
  for (unsigned w = blockIdx.x; w < ntiles; w += gridDim.x) {
    const unsigned tile = tiles[w];
    const int tz = tile % g.tz, ty = (tile / g.tz) % g.ty, tx = tile / (g.tz * g.ty);
    const int x = tx * 8 + lx, y = ty * 8 + ly, z0 = tz * 8 + half * 4;
    unsigned long long c[4] = {0, 0, 0, 0};
    const bool inside = x < g.gx && y < g.gy && z0 < g.pz;             // pz is a multiple of 4: the 4 voxels are in the array
    const long long base = fb_ii(g, x, y, z0);
    if (inside) {
      const ulonglong2 a = reinterpret_cast<const ulonglong2 *>(cnt + base)[0], b = reinterpret_cast<const ulonglong2 *>(cnt + base)[1];
      c[0] = a.x; c[1] = a.y; c[2] = b.x; c[3] = b.y;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      bool push_ins = false, push_del = false;
      const uint32_t ii = (uint32_t)(base + k);
      if (c[k] != 0ull) {
        ++touched;
        const long long hit = (long long)(c[k] >> 32), tot = (long long)(c[k] & 0xffffffffull);
        cnt[ii] = 0ull;                                                     // num_hit_ = num_miss_ = 0
        const double upd = (hit >= tot - hit) ? l_hit : l_miss;             // majority vote, ties -> hit (:243)
        if (cobs[ii] == FB_UNKNOWN) cobs[ii] = FB_INF;                      // first observation: distance_ = +infinity_ (:246-249)
        double o = occ[ii];
        const bool was = o > l_occ;                                         // Exist(idx) before (:242)
        const bool skip = (upd >= 0 && o >= l_max) || (upd <= 0 && o <= l_min);   // already clamped in that direction (:250-255)
        if (!skip) {
          if (!global_map && !fb_in_last_range(g, x, y, z0 + k)) {          // local map (:256-259): occupancy 0, distance_ +infinity_
            o = 0;
            if (EXACT) { if ((cobs[ii] & FB_CODE_MASK) >= 2u) cobs[ii] |= FB_DINF; }   // ... and the closest obstacle is KEPT
            else cobs[ii] = FB_INF;
          }
          double s = o + upd;
          s = s > l_min ? s : l_min;
          s = s < l_max ? s : l_max;
          occ[ii] = s;
          const bool now = s > l_occ;
          if (now && !was) { push_ins = true; atomicOr(&occbits[ii >> 5], 1u << (ii & 31)); }          // insert_queue_.push (:263-264)
          else if (!now && was) { push_del = true; atomicAnd(&occbits[ii >> 5], ~(1u << (ii & 31))); }  // delete_queue_.push (:265-266)
        }
      }
      const unsigned si = fb_warp_append(n_ins, push_ins);
      if (push_ins) { ins[si] = ii; if (EXACT) ins_key[si] = FB_KEY_MASK - (tkey[ii] & FB_KEY_MASK); }
      const unsigned sd = fb_warp_append(n_del, push_del);
      if (push_del) { del[sd] = ii; if (EXACT) del_key[sd] = FB_KEY_MASK - (tkey[ii] & FB_KEY_MASK); }
    }
  }
  touched = __reduce_add_sync(0xffffffffu, touched);
  if ((threadIdx.x & 31) == 0 && touched) atomicAdd(&ctr->n_touched, touched);
}

// distance_buffer_ value of a record (ESDFMap.cpp:122-123, 198, 247): exact because the stored obstacle coordinate is exact.
// Host + device: the pinned host mirror (fiesta_host_mirror_*) evaluates the same expression on the same records.
__host__ __device__ __forceinline__ double fb_record_distance(uint32_t c, int x, int y, int z, double res) {
  const bool dinf = (c & FB_DINF) != 0u;                                    // between calls bit 31 is only ever set by EXACT mode's local-map reset
  c &= FB_CODE_MASK;
  if (c == FB_UNKNOWN) return (double)FIESTA_UNDEFINED;
  if (c == FB_INF || dinf) return (double)FIESTA_INFINITY;
  int ox, oy, oz;
  fb_unpack(c, ox, oy, oz);
  const double dx = (double)(ox - x), dy = (double)(oy - y), dz = (double)(oz - z);
  return sqrt((dx * dx + dy * dy) + dz * dz) * res;
}

__global__ void k_export(FbGeom g, const uint32_t *cobs, const double *occ, const unsigned long long *cnt, double *out_dist,
                         int *out_cobs, double *out_occ, int *out_hit, int *out_tot) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // reference linear index
  if (idx >= g.total) return;
  const int x = (int)(idx / g.gyz), y = (int)(idx % g.gyz / g.gz), z = (int)(idx % g.gz);
  const long long ii = fb_ii(g, x, y, z);
  if (out_dist) out_dist[idx] = fb_record_distance(cobs[ii], x, y, z, g.res);
  if (out_cobs) {
    const uint32_t c = cobs[ii] & FB_CODE_MASK;
    int ox = FIESTA_UNDEFINED, oy = FIESTA_UNDEFINED, oz = FIESTA_UNDEFINED;
    if (c >= 2u) fb_unpack(c, ox, oy, oz);
    out_cobs[3 * idx] = ox; out_cobs[3 * idx + 1] = oy; out_cobs[3 * idx + 2] = oz;
  }
  if (out_occ) out_occ[idx] = occ[ii];
  if (out_hit) { const unsigned long long c = cnt[ii]; out_hit[idx] = (int)(c >> 32); out_tot[idx] = (int)(c & 0xffffffffull); }
}

// GetDistance(Vector3i) (ESDFMap.cpp:477-479): unknown reads +infinity_.  Out-of-grid coordinates (undefined behaviour
// in the reference) also read +infinity_.
__host__ __device__ __forceinline__ uint32_t fb_ld_record(const uint32_t *p) {
#ifdef __CUDA_ARCH__
  return __ldg(p);
#else
  return *p;
#endif
}
__host__ __device__ __forceinline__ double fb_get_distance_vox(const FbGeom &g, const uint32_t *cobs, int x, int y, int z) {
  if (!fb_in_grid(g, x, y, z)) return (double)FIESTA_INFINITY;
  const double d = fb_record_distance(fb_ld_record(&cobs[fb_ii(g, x, y, z)]), x, y, z, g.res);
  return d < 0 ? (double)FIESTA_INFINITY : d;
}
__host__ __device__ __forceinline__ bool fb_pos_in_map(const FbGeom &g, const double *p) {
  if (p[0] < g.min_range[0] || p[1] < g.min_range[1] || p[2] < g.min_range[2]) return false;
  if (p[0] > g.max_range[0] || p[1] > g.max_range[1] || p[2] > g.max_range[2]) return false;
  return true;
}
// GetDistance(Vector3d) (ESDFMap.cpp:467-475)
__host__ __device__ __forceinline__ double fb_query_distance(const FbGeom &g, const uint32_t *cobs, const double *p) {
  if (!fb_pos_in_map(g, p)) return (double)FIESTA_UNDEFINED;
  const int x = (int)floor((p[0] - g.origin[0]) / g.res), y = (int)floor((p[1] - g.origin[1]) / g.res), z = (int)floor((p[2] - g.origin[2]) / g.res);
  return fb_get_distance_vox(g, cobs, x, y, z);
}
// GetDistWithGradTrilinear (ESDFMap.cpp:481-540), operation for operation (fp64, no contraction: -fmad=false on the device,
// no FMA target on the host).
__host__ __device__ __forceinline__ double fb_query_trilinear(const FbGeom &g, const uint32_t *cobs, const double *p, double *grad) {
  if (!fb_pos_in_map(g, p)) { grad[0] = grad[1] = grad[2] = 0.0; return -1.0; }
  int b[3];
  double bp[3], f[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double pm = p[k] - 0.5 * g.res * 1.0;                           // pos - 0.5*resolution_*Ones()
    b[k] = (int)floor((pm - g.origin[k]) / g.res);
    bp[k] = (b[k] + 0.5) * g.res + g.origin[k];                           // Vox2Pos
    f[k] = (p[k] - bp[k]) * g.res_inv;
  }
  double c[2][2][2];
#pragma unroll
  for (int x = 0; x < 2; ++x)
#pragma unroll
    for (int y = 0; y < 2; ++y)
#pragma unroll
      for (int z = 0; z < 2; ++z) c[x][y][z] = fb_get_distance_vox(g, cobs, b[0] + x, b[1] + y, b[2] + z);
  const double v00 = (1 - f[0]) * c[0][0][0] + f[0] * c[1][0][0];
  const double v01 = (1 - f[0]) * c[0][0][1] + f[0] * c[1][0][1];
  const double v10 = (1 - f[0]) * c[0][1][0] + f[0] * c[1][1][0];
  const double v11 = (1 - f[0]) * c[0][1][1] + f[0] * c[1][1][1];
  const double v0 = (1 - f[1]) * v00 + f[1] * v10;
  const double v1 = (1 - f[1]) * v01 + f[1] * v11;
  grad[2] = (v1 - v0) * g.res_inv;
  grad[1] = ((1 - f[2]) * (v10 - v00) + f[2] * (v11 - v01)) * g.res_inv;
  double g0 = (1 - f[2]) * (1 - f[1]) * (c[1][0][0] - c[0][0][0]);
  g0 += (1 - f[2]) * f[1] * (c[1][1][0] - c[0][1][0]);
  g0 += f[2] * (1 - f[1]) * (c[1][0][1] - c[0][0][1]);
  g0 += f[2] * f[1] * (c[1][1][1] - c[0][1][1]);
  g0 *= g.res_inv;
  grad[0] = g0;
  return (1 - f[2]) * v0 + f[2] * v1;
}

// mode 0: GetDistance(Vector3d)  (ESDFMap.cpp:467-475)      out[i]
// mode 1: GetDistWithGradTrilinear (ESDFMap.cpp:481-540)    out[i], grad[3i..]
// mode 2: GetOccupancy(Vector3d)  (ESDFMap.cpp:452-460)      out[i] = 0/1/-10000
__global__ void k_query(FbGeom g, const uint32_t *cobs, const double *occ, double l_occ, const double *pos, long long n, int mode,
                        double *out, double *grad) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double p[3] = {pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]};
  if (mode == 0) { out[i] = fb_query_distance(g, cobs, p); return; }
  if (mode == 2) {
    if (!fb_pos_in_map(g, p)) { out[i] = (double)FIESTA_UNDEFINED; return; }
    const int x = (int)floor((p[0] - g.origin[0]) / g.res), y = (int)floor((p[1] - g.origin[1]) / g.res), z = (int)floor((p[2] - g.origin[2]) / g.res);
    out[i] = fb_in_grid(g, x, y, z) ? (occ[fb_ii(g, x, y, z)] > l_occ ? 1.0 : 0.0) : 0.0;
    return;
  }
  double gr[3];
  out[i] = fb_query_trilinear(g, cobs, p, gr);
  grad[3 * i] = gr[0]; grad[3 * i + 1] = gr[1]; grad[3 * i + 2] = gr[2];
}

// ====================================================================== host helpers
static void set_box_flag(FbGeom &g) {
  g.box_is_full = g.min_vec[0] == 0 && g.min_vec[1] == 0 && g.min_vec[2] == 0 && g.max_vec[0] == g.gx - 1 &&
                  g.max_vec[1] == g.gy - 1 && g.max_vec[2] == g.gz - 1;
}
static bool host_pos_in_map(const FbGeom &g, const double *p) {
  for (int i = 0; i < 3; ++i) if (p[i] < g.min_range[i]) return false;
  for (int i = 0; i < 3; ++i) if (p[i] > g.max_range[i]) return false;
  return true;
}
static void host_pos2vox(const FbGeom &g, const double *p, int *v) {
  for (int i = 0; i < 3; ++i) v[i] = (int)floor((p[i] - g.origin[i]) / g.res);
}
static int fetch_counters(fiesta_map *m) {
  CK(cudaMemcpyAsync(m->h_ctr, m->d_ctr, sizeof(FbCounters), cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  m->n_touch_tiles = m->h_ctr->n_touch_tiles;
  if (m->mode == FIESTA_MODE_FAST) { m->n_ins = m->h_ctr->n_ins; m->n_del = m->h_ctr->n_del; }
  return FIESTA_OK;
}
static int flush_events(fiesta_map *m) {
  if (m->n_ev == 0) return FIESTA_OK;
  CK(cudaMemcpyAsync(m->d_ev, m->h_ev, m->n_ev * sizeof(uint32_t), cudaMemcpyHostToDevice, m->stream));
  if (m->mode == FIESTA_MODE_EXACT && m->X.key_base + m->n_ev >= FB_KEY_MASK) { set_error("more than 2^44 observations between two UpdateOccupancy calls"); return FIESTA_ERR_LIMIT; }
  FbTouch t = {m->cnt, m->touch_flag, m->touch_list, m->touch_epoch, m->d_ctr, m->mode == FIESTA_MODE_EXACT ? m->X.tkey.get() : nullptr, m->X.key_hi};
  k_apply_events<<<(unsigned)((m->n_ev + 255) / 256), 256, 0, m->stream>>>(m->g, m->d_ev, m->n_ev, t, m->X.key_base);
  m->X.key_base += m->n_ev;
  m->st.kernel_launches++;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(m->stream));                                   // the pinned buffer is reused immediately
  m->n_ev = 0;
  return FIESTA_OK;
}
static inline int stage_event(fiesta_map *m, const int *v, int occ) {
  if (m->n_ev == m->h_ev.size()) { int r = flush_events(m); if (r) return r; }
  const long long ii = fb_ii(m->g, v[0], v[1], v[2]);
  m->pending_obs = true;
  m->h_ev[m->n_ev++] = (uint32_t)ii | ((uint32_t)occ << 31);
  return FIESTA_OK;
}
// ESDFMap::SetOccupancy(Vector3i, int) (ESDFMap.cpp:417-437) -- host half: index + range test + staged event.
static inline int host_set_occupancy_vox(fiesta_map *m, const int *v, int occ, int *ret) {
  const FbGeom &g = m->g;
  *ret = v[0] * g.gyz + v[1] * g.gz + v[2];                               // Vox2Idx (:91), returned even when not counted
  if (!fb_in_range(g, v[0], v[1], v[2])) return FIESTA_OK;                // :420-421
  if (!fb_in_grid(g, v[0], v[1], v[2])) return FIESTA_OK;                 // cannot happen for a box set through SetUpdateRange
  return stage_event(m, v, occ & 1);
}

// ====================================================================== C ABI
extern "C" {

const char *fiesta_last_error(void) { return g_last_error.c_str(); }

void fiesta_host_mirror_destroy(struct fiesta_host_mirror *p);
void fiesta_destroy(fiesta_map *m) {
  if (!m) return;
  cudaSetDevice(m->device);                                               // its buffers are freed on the device that holds them
  if (m->mirror) fiesta_host_mirror_destroy(m->mirror);                   // a mirror still attached goes with its map
  if (m->stream) cudaStreamSynchronize(m->stream);
  delete m;
}

int fiesta_create(const fiesta_config *cfg, fiesta_map **out) {
  if (!cfg || !out) { set_error("fiesta_create: null argument"); return FIESTA_ERR_INVALID; }
  *out = nullptr;
  if (!(cfg->resolution > 0)) { set_error("fiesta_create: resolution must be > 0"); return FIESTA_ERR_INVALID; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || cfg->device < 0 || cfg->device >= ndev) {
    set_error("fiesta_create: no CUDA device %s(this library has no CPU fallback)", ""); return FIESTA_ERR_NO_DEVICE;
  }
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) { set_error("fiesta_create: device is not sm_100 (%s); this build only contains sm_100a code", prop.name); return FIESTA_ERR_NO_DEVICE; }
  CK(cudaSetDevice(cfg->device));
  std::unique_ptr<fiesta_map> m(new (std::nothrow) fiesta_map());       // freed on every error return below
  if (!m) { set_error("out of host memory"); return FIESTA_ERR_INVALID; }
  m->device = cfg->device;
  m->mode = cfg->mode == FIESTA_MODE_FAST ? FIESTA_MODE_FAST : FIESTA_MODE_EXACT;
  if (const char *em = getenv("FIESTA_B200_MODE")) {                    // documented override (include/fiesta_b200.h)
    if (!strcmp(em, "fast")) m->mode = FIESTA_MODE_FAST; else if (!strcmp(em, "exact")) m->mode = FIESTA_MODE_EXACT;
  }
  m->shard_rank = 0; m->shard_world = 1;
  FbGeom &g = m->g;
  int gs[3];
  for (int i = 0; i < 3; ++i) {                                           // ctor, ESDFMap.cpp:171-186
    g.origin[i] = cfg->origin[i];
    gs[i] = (int)ceil(cfg->map_size[i] / cfg->resolution);
    g.min_range[i] = cfg->origin[i];
    g.max_range[i] = cfg->origin[i] + cfg->map_size[i];
    m->l_cornor[i] = cfg->origin[i];
    m->r_cornor[i] = cfg->origin[i] + cfg->map_size[i];
  }
  g.res = cfg->resolution; g.res_inv = 1 / cfg->resolution;
  if (gs[0] < 1 || gs[1] < 1 || gs[2] < 1 || gs[0] > FB_MAX_GX || gs[1] > FB_MAX_GY || gs[2] > FB_MAX_GZ) {
    set_error("fiesta_create: grid exceeds the supported 2046 x 1024 x 1024 voxels"); return FIESTA_ERR_LIMIT;
  }
  g.gx = gs[0]; g.gy = gs[1]; g.gz = gs[2]; g.pz = (g.gz + 3) & ~3;
  g.gyz = g.gy * g.gz;
  const long long total = (long long)g.gx * g.gyz;
  g.ptotal = (long long)g.gx * g.gy * g.pz;
  if (total > 0x7fffffffLL || g.ptotal > (long long)FB_LIST_IDX_MASK) { set_error("fiesta_create: more than 2^30 voxels"); return FIESTA_ERR_LIMIT; }
  g.total = (int)total;
  g.tx = (g.gx + 7) / 8; g.ty = (g.gy + 7) / 8; g.tz = (g.gz + 7) / 8; g.ntiles = g.tx * g.ty * g.tz;
  for (int i = 0; i < 3; ++i) { g.min_vec[i] = g.last_min_vec[i] = 0; }   // SetOriginalRange, ESDFMap.cpp:819-822
  g.max_vec[0] = g.last_max_vec[0] = g.gx - 1; g.max_vec[1] = g.last_max_vec[1] = g.gy - 1; g.max_vec[2] = g.last_max_vec[2] = g.gz - 1;
  set_box_flag(g);
  m->tile_x_lo = 0; m->tile_x_hi = g.tx;

  CK(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
  for (int i = 0; i < 4; ++i) CK(cudaEventCreate(&m->ev[i]));
  const size_t P = (size_t)g.ptotal;
  const size_t nbits = (P + 31) / 32;
  CK(m->cobs.alloc(P)); CK(m->cobs_b.alloc(P));
  CK(m->stamp[0].alloc(P)); CK(m->stamp[1].alloc(P));
  CK(m->occbits.alloc(nbits));
  CK(m->occ.alloc(P)); CK(m->cnt.alloc(P));
  CK(m->touch_flag.alloc(g.ntiles)); CK(m->touch_list.alloc(g.ntiles));
  CK(m->tile_flag.alloc(g.ntiles)); CK(m->nb_flag.alloc(g.ntiles));
  for (int k = 0; k < 2; ++k) {
    CK(m->list[k].alloc(g.ntiles));
    CK(m->changed[k].alloc(g.ntiles));
    CK(m->changed_bbox[k].alloc(g.ntiles));
  }
  CK(m->d_ctr.alloc(1));
  CK(m->h_ctr.alloc(1));
  CK(m->h_ev.alloc(1u << 22)); CK(m->d_ev.alloc(1u << 22));
  CK(cudaMemsetAsync(m->cobs, 0, P * 4, m->stream)); CK(cudaMemsetAsync(m->cobs_b, 0, P * 4, m->stream));
  CK(cudaMemsetAsync(m->stamp[0], 0, P * 4, m->stream)); CK(cudaMemsetAsync(m->stamp[1], 0, P * 4, m->stream));
  CK(cudaMemsetAsync(m->occbits, 0, nbits * 4, m->stream));
  CK(cudaMemsetAsync(m->occ, 0, P * 8, m->stream)); CK(cudaMemsetAsync(m->cnt, 0, P * 8, m->stream));
  CK(cudaMemsetAsync(m->tile_flag, 0, (size_t)g.ntiles * 4, m->stream)); CK(cudaMemsetAsync(m->nb_flag, 0, (size_t)g.ntiles * 4, m->stream));
  CK(cudaMemsetAsync(m->touch_flag, 0, (size_t)g.ntiles * 4, m->stream));
  m->touch_epoch = 1;
  memset(m->h_ctr, 0, sizeof(FbCounters));
  m->h_ctr->gen_stamp = 1;
  CK(cudaMemcpyAsync(m->d_ctr, m->h_ctr, sizeof(FbCounters), cudaMemcpyHostToDevice, m->stream));
  m->frame_tag = 0; m->owner_tag = 0;
  char err[256];
  if (fb_esdf_make_tensor_map(&m->tmap, g, m->cobs, err, sizeof(err)) != cudaSuccess) { set_error("%s", err); return FIESTA_ERR_CUDA; }
  m->wf_blocks = fb_esdf_wavefront_blocks(m->device);
  m->rr_blocks = fb_ray_resolve_blocks(m->device);
  if (m->wf_blocks <= 0 || m->rr_blocks <= 0) { set_error("cooperative kernels do not fit on this device"); return FIESTA_ERR_CUDA; }
  if (m->mode == FIESTA_MODE_EXACT && fb_exact_init(&m->X, g, m->device, m->stream) != cudaSuccess) { set_error("exact mode init: %s", m->X.err); return FIESTA_ERR_CUDA; }
  CK(cudaStreamSynchronize(m->stream));
  *out = m.release();
  return FIESTA_OK;
}

int fiesta_set_parameters(fiesta_map *m, double p_hit, double p_miss, double p_min, double p_max, double p_occ) {
  if (!m) return FIESTA_ERR_INVALID;
  const double old_occ = m->l_occ;
  m->l_hit = log(p_hit / (1 - p_hit)); m->l_miss = log(p_miss / (1 - p_miss));     // Logit, ESDFMap.cpp:12-14
  m->l_min = log(p_min / (1 - p_min)); m->l_max = log(p_max / (1 - p_max)); m->l_occ = log(p_occ / (1 - p_occ));
  if (m->params_set && m->l_occ != old_occ) {                              // Exist() (ESDFMap.cpp:46-48) compares with the CURRENT threshold:
    CK(cudaSetDevice(m->device));                                         // bring the occupancy bitmap the ESDF kernels read in line with it
    const size_t words = ((size_t)m->g.ptotal + 31) / 32;
    k_rebuild_occbits<<<(unsigned)((words + 255) / 256), 256, 0, m->stream>>>(m->occ, m->g.ptotal, m->l_occ, m->occbits);
    m->st.kernel_launches++;
    CK(cudaGetLastError());
  }
  m->params_set = true;
  return FIESTA_OK;
}
int fiesta_grid_total_size(const fiesta_map *m) { return m ? m->g.total : 0; }
int fiesta_grid_size(const fiesta_map *m, int out[3]) {
  if (!m || !out) return FIESTA_ERR_INVALID;
  out[0] = m->g.gx; out[1] = m->g.gy; out[2] = m->g.gz;
  return FIESTA_OK;
}

int fiesta_set_occupancy_vox(fiesta_map *m, const int vox[3], int occ) {
  int ret = FIESTA_UNDEFINED;
  if (!m || !vox) return FIESTA_UNDEFINED;
  if (host_set_occupancy_vox(m, vox, occ, &ret) != FIESTA_OK) return FIESTA_UNDEFINED;
  return ret;
}
int fiesta_set_occupancy_pos(fiesta_map *m, const double pos[3], int occ) {
  if (!m || !pos) return FIESTA_UNDEFINED;
  if (occ != 1 && occ != 0) return FIESTA_UNDEFINED;                      // "occ value error!", ESDFMap.cpp:402-405
  if (!host_pos_in_map(m->g, pos)) return FIESTA_UNDEFINED;               // :407-410
  int v[3];
  host_pos2vox(m->g, pos, v);
  return fiesta_set_occupancy_vox(m, v, occ);
}
int fiesta_set_occupancy_batch_vox(fiesta_map *m, const int *vox, const uint8_t *occ, int64_t n, int *out_idx) {
  if (!m || (n > 0 && (!vox || !occ))) return FIESTA_ERR_INVALID;
  for (int64_t i = 0; i < n; ++i) {
    int ret;
    int r = host_set_occupancy_vox(m, vox + 3 * i, occ[i], &ret);
    if (r) return r;
    if (out_idx) out_idx[i] = ret;
  }
  return FIESTA_OK;
}
int fiesta_set_occupancy_batch_pos(fiesta_map *m, const double *pos, const uint8_t *occ, int64_t n, int *out_idx) {
  if (!m || (n > 0 && (!pos || !occ))) return FIESTA_ERR_INVALID;
  for (int64_t i = 0; i < n; ++i) {
    int ret = FIESTA_UNDEFINED;
    if ((occ[i] == 0 || occ[i] == 1) && host_pos_in_map(m->g, pos + 3 * i)) {
      int v[3];
      host_pos2vox(m->g, pos + 3 * i, v);
      int r = host_set_occupancy_vox(m, v, occ[i], &ret);
      if (r) return r;
    }
    if (out_idx) out_idx[i] = ret;
  }
  return FIESTA_OK;
}

int fiesta_set_occupancy_batch_vox_device(fiesta_map *m, const int *d_vox, const uint8_t *d_occ, int64_t n) {
  if (!m || n < 0 || (n > 0 && (!d_vox || !d_occ))) return FIESTA_ERR_INVALID;
  if (m->mode != FIESTA_MODE_FAST) { set_error("fiesta_set_occupancy_batch_vox_device: FAST mode only (device events carry no serial order)"); return FIESTA_ERR_INVALID; }
  if (n == 0) return FIESTA_OK;
  CK(cudaSetDevice(m->device));
  m->pending_obs = true;
  FbTouch t = {m->cnt, m->touch_flag, m->touch_list, m->touch_epoch, m->d_ctr, nullptr, 0ull};
  k_apply_vox_events<<<(unsigned)((n + 255) / 256), 256, 0, m->stream>>>(m->g, d_vox, d_occ, n, t);
  m->st.kernel_launches++;
  CK(cudaGetLastError());
  int r;
  if ((r = fetch_counters(m))) return r;
  return FIESTA_OK;
}

int fiesta_raycast_frame_device(fiesta_map *m, const float *d_xyz, int64_t n, const double T[16], const fiesta_raycast_params *p) {
  if (!m || !T || !p || n < 0 || (n > 0 && !d_xyz)) { set_error("fiesta_raycast_frame: bad argument"); return FIESTA_ERR_INVALID; }
  if (n >= (int64_t)FB_RAY_MASK) { set_error("fiesta_raycast_frame: more than 2^19-2 (524286) points per frame"); return FIESTA_ERR_LIMIT; }
  CK(cudaSetDevice(m->device));
  m->st.rays_cast = m->st.rays_dropped = m->st.ray_voxels = m->st.raycast_rounds = 0; m->st.ms_raycast = 0;
  { int fr = flush_events(m); if (fr) return fr; }                         // per-call SetOccupancy events issued before this frame come first in occupancy_queue_
  if (m->mode == FIESTA_MODE_EXACT && m->X.key_base + (1ull << 30) >= FB_KEY_MASK) {
    set_error("fiesta_raycast_frame: more than 16383 frames between two UpdateOccupancy calls (order-exact mode)"); return FIESTA_ERR_LIMIT;
  }
  if (n == 0) return FIESTA_OK;
  m->pending_obs = true;
  const FbGeom &g = m->g;
  FbRayArgs a;
  memset(&a, 0, sizeof(a));
  a.xyz = d_xyz; a.n = n;
  memcpy(a.T, T, sizeof(double) * 16);
  for (int k = 0; k < 3; ++k) {
    a.org[k] = T[4 * k + 3] / T[15];                                      // raycast_origin_, Fiesta.h:420
    a.start[k] = a.org[k] / g.res;                                        // Fiesta.h:233-236
    a.bmin[k] = m->l_cornor[k] / g.res;
    a.bmax[k] = m->r_cornor[k] / g.res;
  }
  a.min_len = p->min_ray_length; a.max_len = p->max_ray_length;
  // Lattice fast path: the DDA walks floor(world/res) voxels while the map uses floor((world-origin)/res) (ESDFMap.cpp:74-77).
  // If, for every DDA coordinate c inside the box and every axis, the voxel centre (c+0.5)*res lies in the map and maps to
  // c - off (checked here with the reference's own fp64 expressions), the per-voxel divisions can be skipped exactly.
  a.lattice_ok = 1;
  for (int k = 0; k < 3 && a.lattice_ok; ++k) {
    const int G = k == 0 ? g.gx : (k == 1 ? g.gy : g.gz);
    const long long clo = (long long)ceil(a.bmin[k]), chi = (long long)ceil(a.bmax[k]);   // integers c with bmin <= c < bmax
    if (chi - clo > 4096 || chi <= clo) { a.lattice_ok = 0; break; }
    const double c0 = ((double)clo + 0.5) * g.res;
    const long long off = clo - (long long)floor((c0 - g.origin[k]) / g.res);
    a.lattice_off[k] = (int)off;
    for (long long c = clo; c < chi; ++c) {
      const double ctr = ((double)c + 0.5) * g.res;
      const long long v = (long long)floor((ctr - g.origin[k]) / g.res);
      if (ctr < g.min_range[k] || ctr > g.max_range[k] || v != c - off || v < 0 || v >= G) { a.lattice_ok = 0; break; }
    }
  }
  double capd = ceil(1.7320508075688772 * (p->max_ray_length / g.res)) + 8.0;
  if (!(capd < 1500.0)) capd = 1500.0;
  if (capd < 1.0) capd = 1.0;
  a.cap = (int)capd;
  a.max_rounds = FB_MAX_ROUNDS;
  if (m->frame_tag >= FB_MAX_CLAIM_FRAME) {                               // claim frame tags exhausted: clear and restart
    CK(cudaMemsetAsync(m->stamp[0], 0, (size_t)g.ptotal * 4, m->stream));
    m->frame_tag = 0;
  }
  if (m->owner_tag >= FB_MAX_OWNER_FRAME) {
    CK(cudaMemsetAsync(m->stamp[1], 0, (size_t)g.ptotal * 4, m->stream));
    m->owner_tag = 0;
  }
  a.frame_tag = ++m->frame_tag;
  a.owner_tag = ++m->owner_tag;
  int r;
  CK(m->ray_len.reserve((size_t)n, m->stream, false));
  CK(m->ray_reach.reserve((size_t)n, m->stream, false));
  CK(m->ray_dirty.reserve((size_t)n, m->stream, false));
  CK(m->ray_list.reserve((size_t)a.cap * (size_t)n, m->stream, false));
  a.cnt = m->cnt; a.stamp[0] = m->stamp[0]; a.stamp[1] = m->stamp[1];
  a.touch_flag = m->touch_flag; a.touch_list = m->touch_list; a.touch_epoch = m->touch_epoch;
  a.tkey = m->mode == FIESTA_MODE_EXACT ? m->X.tkey.get() : nullptr; a.key_hi = m->X.key_hi; a.key_base = m->X.key_base;
  m->X.key_base += 1ull << 30;                                            // (point index << 11) + position along the ray < 2^30
  a.ray_list = m->ray_list; a.ray_len = m->ray_len; a.ray_reach = m->ray_reach; a.ray_dirty = m->ray_dirty; a.ctr = m->d_ctr;
  static const bool dbg_ray = getenv("FIESTA_DEBUG_RAY") != nullptr;
  a.dbg = nullptr;
  if (dbg_ray) { if (!m->d_dbg) CK(m->d_dbg.alloc(2048)); CK(cudaMemsetAsync(m->d_dbg, 0, 2048 * 8, m->stream)); a.dbg = m->d_dbg; }
  CK(cudaEventRecord(m->ev[0], m->stream));
  k_reset_ray_ctr<<<1, 1, 0, m->stream>>>(m->d_ctr);
  int launches = 1;
  CK(fb_ray_frame(g, a, m->rr_blocks, m->stream, &launches));
  m->st.kernel_launches += launches;
  CK(cudaEventRecord(m->ev[1], m->stream));
  if ((r = fetch_counters(m))) return r;
  CK(cudaEventElapsedTime(&m->st.ms_raycast, m->ev[0], m->ev[1]));
  m->st.rays_cast = m->h_ctr->rays_cast; m->st.rays_dropped = m->h_ctr->rays_dropped;
  m->st.ray_voxels = (int64_t)m->h_ctr->ray_voxels; m->st.raycast_rounds = m->h_ctr->ray_rounds;
  m->st.touched_voxels = (int64_t)m->n_touch_tiles * 512;
  if (a.dbg) {
    unsigned long long h[1024];
    CK(cudaMemcpy(h, m->d_dbg, sizeof(h), cudaMemcpyDeviceToHost));
    fprintf(stderr, "[ray] rounds=%u counts %.0fus", m->h_ctr->ray_rounds, h[0] * 1e-3);
    for (unsigned r2 = 1; r2 <= m->h_ctr->ray_rounds && r2 < 300; ++r2) fprintf(stderr, " | %llu %.0fus", h[3 * r2], h[3 * r2 + 2] * 1e-3);
    fprintf(stderr, "\n");
  }
  if (m->h_ctr->ray_error == 3) { set_error("fiesta_raycast_frame: stamp resolution did not converge"); return FIESTA_ERR_LIMIT; }
  return FIESTA_OK;
}

int fiesta_raycast_frame(fiesta_map *m, const float *xyz, int64_t n, const double T[16], const fiesta_raycast_params *p) {
  if (!m || n < 0 || (n > 0 && !xyz)) { set_error("fiesta_raycast_frame: bad argument"); return FIESTA_ERR_INVALID; }
  CK(cudaSetDevice(m->device));
  CK(m->d_xyz.reserve((size_t)n * 3, m->stream, false));
  if (n) CK(cudaMemcpyAsync(m->d_xyz, xyz, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, m->stream));
  return fiesta_raycast_frame_device(m, m->d_xyz, n, T, p);
}

int fiesta_depth_frame(fiesta_map *m, const uint16_t *depth, int rows, int cols, const fiesta_depth_params *dp, const double T[16],
                       const double m_rel[16], const fiesta_raycast_params *rp, int64_t *n_points) {
  if (!m || !depth || !dp || !T || !rp || rows <= 0 || cols <= 0) { set_error("fiesta_depth_frame: bad argument"); return FIESTA_ERR_INVALID; }
  CK(cudaSetDevice(m->device));
  const size_t N = (size_t)rows * cols;
  if (N > m->cap_img) {                                                   // exact sizes: a larger image restarts the depth filter
    m->cap_img = 0;
    CK(m->d_img[0].alloc(N)); CK(m->d_img[1].alloc(N));
    CK(m->d_dpts.alloc(N * 3)); CK(m->d_dcloud.alloc(N * 3));
    CK(m->d_dflags.alloc(N)); CK(m->d_dsel.alloc(N));
    if (!m->d_dcount) CK(m->d_dcount.alloc(4));
    m->cap_img = N; m->image_cnt = 0;
  }
  ++m->image_cnt;                                                          // Fiesta.h:321-323: img_[image_cnt_ & 1] is the current image
  uint16_t *cur = m->d_img[m->image_cnt & 1], *last = m->d_img[!(m->image_cnt & 1)];
  CK(cudaMemcpyAsync(cur, depth, N * 2, cudaMemcpyHostToDevice, m->stream));
  unsigned n = 0;
  if (dp->use_depth_filter && m->image_cnt == 1) {                         // :353: the first image only primes the filter
    m->last_cloud_n = 0;
    if (n_points) *n_points = 0;
    CK(cudaStreamSynchronize(m->stream));
    return FIESTA_OK;
  }
  FbDepthRel rel;
  for (int k = 0; k < 16; ++k) rel.m[k] = (dp->use_depth_filter && m_rel) ? m_rel[k] : (k % 5 == 0 ? 1.0 : 0.0);
  CK(fb_depth_to_cloud(cur, last, rows, cols, *dp, dp->use_depth_filter ? 1 : 0, rel, m->d_dpts, m->d_dflags, m->d_dsel, m->d_dcloud, m->d_dcount,
                       m->d_dtmp, &n, m->stream));
  m->st.kernel_launches += 3;
  m->last_cloud_n = n;
  if (n_points) *n_points = n;
  if (n == 0) return FIESTA_OK;                                            // `if (cloud_.points.size() == 0) continue;` (Fiesta.h:430-433)
  return fiesta_raycast_frame_device(m, m->d_dcloud, n, T, rp);
}
int fiesta_last_depth_cloud(fiesta_map *m, float *out, int64_t cap, int64_t *n_points) {
  if (!m || !n_points) return FIESTA_ERR_INVALID;
  *n_points = m->last_cloud_n;
  const int64_t k = m->last_cloud_n < cap ? m->last_cloud_n : cap;
  if (k > 0 && out) CK(cudaMemcpy(out, m->d_dcloud, (size_t)k * 12, cudaMemcpyDeviceToHost));
  return FIESTA_OK;
}

int fiesta_check_update(fiesta_map *m) {
  if (!m) return 0;
  return (m->n_ev > 0 || m->n_touch_tiles > 0) ? 1 : 0;                       // !occupancy_queue_.empty(), ESDFMap.cpp:229
}

int fiesta_update_occupancy(fiesta_map *m, int global_map) {
  if (!m) return -FIESTA_ERR_INVALID;
  if (!m->params_set) { set_error("fiesta_update_occupancy: SetParameters was never called"); return -FIESTA_ERR_INVALID; }
  if (cudaSetDevice(m->device) != cudaSuccess) return -FIESTA_ERR_CUDA;
  int r;
  mark_dirty(m);
  m->pending_obs = false;
  cudaEventRecord(m->ev[0], m->stream);
  if ((r = flush_events(m))) return -r;
  if ((r = fetch_counters(m))) return -r;
  const unsigned n = m->n_touch_tiles;
  m->st.occupancy_updates = 0;
  if (m->mode == FIESTA_MODE_EXACT) {
    if (n) {
      FbExact &X = m->X;
      k_reset_touched<<<1, 1, 0, m->stream>>>(m->d_ctr);
      cudaMemsetAsync(X.d_count, 0, 8, m->stream);
      const unsigned blocks = n < 148u * 16u ? n : 148u * 16u;
      // crossings are staged (voxel, first-observation time) in arrays that are scratch between two k_x_relax launches
      unsigned long long *ikey = reinterpret_cast<unsigned long long *>(X.SUM.get()), *dkey = ikey + m->g.ptotal;
      k_integrate<true><<<blocks, 128, 0, m->stream>>>(m->g, m->touch_list, n, m->cnt, m->occ, m->cobs, m->occbits, X.touched, X.emask, X.d_count, X.d_count + 1,
                                                       m->d_ctr, X.tkey, ikey, dkey, global_map, m->l_hit, m->l_miss, m->l_min, m->l_max, m->l_occ);
      k_reset_queues<<<1, 1, 0, m->stream>>>(m->d_ctr, 1, 0);
      m->touch_epoch++;
      m->st.kernel_launches += 3;
      int launches = 0;
      if (fb_exact_queue_crossings(&X, ikey, X.touched, dkey, X.emask, m->ins, &m->n_ins, m->del, &m->n_del, m->stream, &launches) != cudaSuccess) {
        set_error("exact UpdateOccupancy: %s", X.err); return -FIESTA_ERR_CUDA;
      }
      m->st.kernel_launches += launches;
      if ((r = fb_exact_next_epoch(&X, m->g, m->stream))) { set_error("exact UpdateOccupancy: %s", X.err); return -FIESTA_ERR_CUDA; }
    }
    cudaEventRecord(m->ev[1], m->stream);
    if ((r = fetch_counters(m))) return -r;
    cudaEventElapsedTime(&m->st.ms_update_occupancy, m->ev[0], m->ev[1]);
    if (n) m->st.occupancy_updates = m->h_ctr->n_touched;
    m->st.touched_voxels = 0;
    return (m->n_ins > 0 || m->n_del > 0) ? 1 : 0;
  }
  if (n) {
    cudaError_t e = m->ins.reserve((size_t)m->n_ins + (size_t)n * 512, m->stream, true);   // pushes not yet consumed by UpdateESDF stay
    if (e == cudaSuccess) e = m->del.reserve((size_t)m->n_del + (size_t)n * 512, m->stream, true);
    if (e != cudaSuccess) { set_error("UpdateOccupancy: growing the queues failed: %s", cudaGetErrorString(e)); return -FIESTA_ERR_CUDA; }
    k_reset_touched<<<1, 1, 0, m->stream>>>(m->d_ctr);
    const unsigned blocks = n < 148u * 16u ? n : 148u * 16u;
    k_integrate<false><<<blocks, 128, 0, m->stream>>>(m->g, m->touch_list, n, m->cnt, m->occ, m->cobs, m->occbits, m->ins, m->del, &m->d_ctr->n_ins, &m->d_ctr->n_del,
                                                     m->d_ctr, nullptr, nullptr, nullptr, global_map, m->l_hit, m->l_miss, m->l_min, m->l_max, m->l_occ);
    k_reset_queues<<<1, 1, 0, m->stream>>>(m->d_ctr, 1, 0);
    m->touch_epoch++;
    m->st.kernel_launches += 3;
    if (cudaGetLastError() != cudaSuccess) { set_error("k_integrate launch failed"); return -FIESTA_ERR_CUDA; }
  }
  cudaEventRecord(m->ev[1], m->stream);
  if ((r = fetch_counters(m))) return -r;
  cudaEventElapsedTime(&m->st.ms_update_occupancy, m->ev[0], m->ev[1]);
  if (n) m->st.occupancy_updates = m->h_ctr->n_touched;
  m->st.touched_voxels = 0;
  return (m->n_ins > 0 || m->n_del > 0) ? 1 : 0;                          // :270
}

int fiesta_update_esdf(fiesta_map *m) {
  if (!m) return FIESTA_ERR_INVALID;
  CK(cudaSetDevice(m->device));
  m->st.inserts = m->n_ins; m->st.deletes = m->n_del;
  m->st.voxels_changed = m->st.voxels_reset = m->st.tile_visits = m->st.generations = m->st.expansions = 0;
  m->st.ms_update_esdf = m->st.ms_esdf_delete_scan = m->st.ms_esdf_wavefront = 0;
  if (m->n_ins == 0 && m->n_del == 0) return FIESTA_OK;
  mark_dirty(m);
  if (m->n_del) {                                                          // dependants of a deleted obstacle are reset wherever they lie,
    m->dirty_lo[0] = m->dirty_lo[1] = m->dirty_lo[2] = 0;                   // also outside the update box (ESDFMap.cpp:301-334)
    m->dirty_hi[0] = m->g.gx - 1; m->dirty_hi[1] = m->g.gy - 1; m->dirty_hi[2] = m->g.gz - 1;
  }
  if (m->mode == FIESTA_MODE_EXACT) {
    FbExactStats xs;
    int launches = 0;
    CK(cudaEventRecord(m->ev[0], m->stream));
    if (fb_exact_update_esdf(&m->X, m->g, m->cobs, m->cobs_b, m->occ, m->occbits, m->l_occ, m->ins, m->n_ins, m->del, m->n_del, m->stream, &xs,
                             &launches) != cudaSuccess) { set_error("exact UpdateESDF: %s", m->X.err); return FIESTA_ERR_CUDA; }
    CK(cudaEventRecord(m->ev[3], m->stream));
    CK(cudaStreamSynchronize(m->stream));
    CK(cudaEventElapsedTime(&m->st.ms_update_esdf, m->ev[0], m->ev[3]));
    m->st.kernel_launches += launches;
    m->st.voxels_changed = (int64_t)xs.voxels_changed; m->st.expansions = (int64_t)xs.expansions; m->st.voxels_reset = xs.dependants;
    m->st.generations = xs.generations; m->st.tile_visits = 0;
    m->n_ins = m->n_del = 0;
    return FIESTA_OK;
  }
  FbEsdfArgs a;
  a.cobs = m->cobs; a.cobs_b = m->cobs_b; a.occ = m->occ; a.occbits = m->occbits; a.tile_flag = m->tile_flag; a.nb_flag = m->nb_flag;
  for (int k = 0; k < 2; ++k) { a.list[k] = m->list[k]; a.changed[k] = m->changed[k]; a.changed_bbox[k] = m->changed_bbox[k]; }
  a.ctr = m->d_ctr; a.l_occ = m->l_occ;
  a.tile_x_lo = m->tile_x_lo; a.tile_x_hi = m->tile_x_hi;
  a.dbg = nullptr;
  static const bool dbg_wf = getenv("FIESTA_DEBUG_WF") != nullptr;
  if (dbg_wf) { if (!m->d_dbg) CK(m->d_dbg.alloc(2048)); CK(cudaMemsetAsync(m->d_dbg, 0, 2048 * 8, m->stream)); a.dbg = m->d_dbg; }
  CK(cudaEventRecord(m->ev[0], m->stream));
  k_reset_esdf_ctr<<<1, 1, 0, m->stream>>>(m->d_ctr);
  m->st.kernel_launches++;
  if (m->n_ins) { CK(fb_esdf_seed_inserts(m->g, a, m->ins, m->n_ins, m->stream)); m->st.kernel_launches++; }   // E1
  CK(cudaEventRecord(m->ev[1], m->stream));
  if (m->n_del) { CK(fb_esdf_delete_scan(m->g, a, m->stream)); m->st.kernel_launches++; }                      // E2
  CK(cudaEventRecord(m->ev[2], m->stream));
  CK(fb_esdf_wavefront(m->g, a, m->tmap, m->wf_blocks, m->stream));                                           // E3
  m->st.kernel_launches++;
  if (m->shard_world > 1) {                                               // FRESH flags the seed / delete scan left in the ghost layers
    const int x0 = m->tile_x_lo * 8, x1 = m->tile_x_hi * 8 < m->g.gx ? m->tile_x_hi * 8 : m->g.gx;
    if (m->shard_rank > 0) CK(fb_esdf_halo_retire(m->g, m->cobs, x0 - 2, 2, m->stream));
    if (m->shard_rank + 1 < m->shard_world) CK(fb_esdf_halo_retire(m->g, m->cobs, x1, 2, m->stream));
  }
  k_reset_queues<<<1, 1, 0, m->stream>>>(m->d_ctr, 0, 1);
  m->st.kernel_launches++;
  CK(cudaEventRecord(m->ev[3], m->stream));
  int r;
  if ((r = fetch_counters(m))) return r;
  CK(cudaEventElapsedTime(&m->st.ms_update_esdf, m->ev[0], m->ev[3]));
  CK(cudaEventElapsedTime(&m->st.ms_esdf_delete_scan, m->ev[1], m->ev[2]));
  CK(cudaEventElapsedTime(&m->st.ms_esdf_wavefront, m->ev[2], m->ev[3]));
  m->st.voxels_changed = (int64_t)m->h_ctr->voxels_changed; m->st.voxels_reset = (int64_t)m->h_ctr->voxels_reset;
  m->st.tile_visits = (int64_t)m->h_ctr->tile_visits; m->st.generations = m->h_ctr->generations;
  if (a.dbg) {
    unsigned long long h[1024];
    CK(cudaMemcpy(h, m->d_dbg, sizeof(h), cudaMemcpyDeviceToHost));
    fprintf(stderr, "[wf] gens=%u", m->h_ctr->generations);
    for (unsigned gI = 0; gI < m->h_ctr->generations && gI < 256; ++gI) fprintf(stderr, " | %llu/%llu %.0f+%.0fus", h[4 * gI], h[4 * gI + 1], h[4 * gI + 2] * 1e-3, h[4 * gI + 3] * 1e-3);
    fprintf(stderr, "\n");
  }
  return FIESTA_OK;
}

int fiesta_set_update_range(fiesta_map *m, const double min_pos[3], const double max_pos[3], int new_vec) {
  if (!m || !min_pos || !max_pos) return FIESTA_ERR_INVALID;
  if (m->pending_obs) mark_dirty(m);                                      // observations counted under the old box are integrated later
  FbGeom &g = m->g;
  double lo[3], hi[3];
  for (int i = 0; i < 3; ++i) {                                           // ESDFMap.cpp:794-800
    lo[i] = min_pos[i] > g.min_range[i] ? min_pos[i] : g.min_range[i];
    hi[i] = max_pos[i] < g.max_range[i] ? max_pos[i] : g.max_range[i];
  }
  if (new_vec) for (int i = 0; i < 3; ++i) { g.last_min_vec[i] = g.min_vec[i]; g.last_max_vec[i] = g.max_vec[i]; }
  host_pos2vox(g, lo, g.min_vec);
  for (int i = 0; i < 3; ++i) hi[i] = hi[i] - g.res / 2;                   // :807-809
  host_pos2vox(g, hi, g.max_vec);
  set_box_flag(g);
  return FIESTA_OK;
}
int fiesta_set_original_range(fiesta_map *m) {
  if (!m) return FIESTA_ERR_INVALID;
  if (m->pending_obs) mark_dirty(m);
  FbGeom &g = m->g;
  for (int i = 0; i < 3; ++i) g.min_vec[i] = g.last_min_vec[i] = 0;
  g.max_vec[0] = g.last_max_vec[0] = g.gx - 1; g.max_vec[1] = g.last_max_vec[1] = g.gy - 1; g.max_vec[2] = g.last_max_vec[2] = g.gz - 1;
  set_box_flag(g);
  return FIESTA_OK;
}

// ---- queries
static int run_query(fiesta_map *m, const double *pos, int64_t n, int mode, double *out, double *grad) {
  if (n <= 0) return FIESTA_OK;
  CK(cudaSetDevice(m->device));
  CK(m->d_qin.reserve((size_t)n * 3, m->stream, false));
  CK(m->d_qout.reserve((size_t)n * 4, m->stream, false));                 // [dist n][grad 3n]
  CK(cudaMemcpyAsync(m->d_qin, pos, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice, m->stream));
  k_query<<<(unsigned)((n + 127) / 128), 128, 0, m->stream>>>(m->g, m->cobs, m->occ, m->l_occ, m->d_qin, n, mode, m->d_qout, m->d_qout + n);
  m->st.kernel_launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, m->d_qout, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  if (grad) CK(cudaMemcpyAsync(grad, m->d_qout + n, (size_t)n * 3 * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  return FIESTA_OK;
}
double fiesta_get_distance_pos(fiesta_map *m, const double pos[3]) {
  double d = FIESTA_UNDEFINED;
  if (!m || run_query(m, pos, 1, 0, &d, nullptr)) return FIESTA_UNDEFINED;
  return d;
}
double fiesta_get_distance_vox(fiesta_map *m, const int vox[3]) {
  if (!m) return FIESTA_INFINITY;
  const FbGeom &g = m->g;
  if (!fb_in_grid(g, vox[0], vox[1], vox[2])) return FIESTA_INFINITY;
  double p[3];
  for (int i = 0; i < 3; ++i) p[i] = (vox[i] + 0.5) * g.res + g.origin[i];          // voxel centre maps back to the same voxel
  int v[3];
  host_pos2vox(g, p, v);
  if (v[0] == vox[0] && v[1] == vox[1] && v[2] == vox[2] && host_pos_in_map(g, p)) return fiesta_get_distance_pos(m, p);
  uint32_t c = 0;                                                         // pathological origin/resolution: read the record directly
  if (cudaMemcpy(&c, m->cobs + fb_ii(g, vox[0], vox[1], vox[2]), 4, cudaMemcpyDeviceToHost) != cudaSuccess) return FIESTA_INFINITY;
  if (c & FB_DINF) return FIESTA_INFINITY;
  c &= FB_CODE_MASK;
  if (c < 2u) return FIESTA_INFINITY;
  int ox, oy, oz; fb_unpack(c, ox, oy, oz);
  const double dx = ox - vox[0], dy = oy - vox[1], dz = oz - vox[2];
  return sqrt((dx * dx + dy * dy) + dz * dz) * g.res;
}
int fiesta_get_occupancy_pos(fiesta_map *m, const double pos[3]) {
  double d = FIESTA_UNDEFINED;
  if (!m || run_query(m, pos, 1, 2, &d, nullptr)) return FIESTA_UNDEFINED;
  return (int)d;
}
int fiesta_get_occupancy_vox(fiesta_map *m, const int vox[3]) {
  if (!m || !fb_in_grid(m->g, vox[0], vox[1], vox[2])) return 0;
  double o = 0;
  if (cudaMemcpy(&o, m->occ + fb_ii(m->g, vox[0], vox[1], vox[2]), 8, cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
  return o > m->l_occ ? 1 : 0;
}
double fiesta_get_dist_grad_trilinear(fiesta_map *m, const double pos[3], double grad[3]) {
  double d = -1;
  if (!m || run_query(m, pos, 1, 1, &d, grad)) return -1;
  return d;
}
int fiesta_get_distance_batch_pos(fiesta_map *m, const double *pos, int64_t n, double *out) {
  if (!m || (n > 0 && (!pos || !out))) return FIESTA_ERR_INVALID;
  return run_query(m, pos, n, 0, out, nullptr);
}
int fiesta_get_dist_grad_trilinear_batch(fiesta_map *m, const double *pos, int64_t n, double *out, double *grad) {
  if (!m || (n > 0 && (!pos || !out || !grad))) return FIESTA_ERR_INVALID;
  return run_query(m, pos, n, 1, out, grad);
}

// ---- planner query plan: fixed batch size, pinned host buffers, the copy-in / kernel / copy-out sequence captured once as a
// CUDA graph; a run is one graph launch + one stream synchronisation (SURVEY.md 8(f) #3).
struct fiesta_query_plan {
  fiesta_map *m;
  int64_t n;
  FbPinned<double> h_pos, h_out;  // [3n] positions; [n] distances followed by [3n] gradients.  The graph captured these
  FbDev<double> d_pos, d_out;     // addresses (and the map's cobs / occ): none of them is ever reallocated
  cudaGraph_t graph;
  cudaGraphExec_t exec;
  ~fiesta_query_plan() {
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
  }
};
void fiesta_query_plan_destroy(fiesta_query_plan *p) {
  if (!p) return;
  cudaSetDevice(p->m->device);
  cudaStreamSynchronize(p->m->stream);
  delete p;
}
int fiesta_query_plan_create(fiesta_map *m, int64_t n, fiesta_query_plan **out) {
  if (!m || !out || n <= 0) { set_error("fiesta_query_plan_create: bad argument"); return FIESTA_ERR_INVALID; }
  if (!m->params_set) { set_error("fiesta_query_plan_create: call SetParameters first (the occupancy threshold is captured)"); return FIESTA_ERR_INVALID; }
  *out = nullptr;
  CK(cudaSetDevice(m->device));
  std::unique_ptr<fiesta_query_plan> p(new (std::nothrow) fiesta_query_plan());
  if (!p) return FIESTA_ERR_INVALID;
  p->m = m; p->n = n;
  CK(p->h_pos.alloc((size_t)n * 3));
  CK(p->h_out.alloc((size_t)n * 4));
  CK(p->d_pos.alloc((size_t)n * 3));
  CK(p->d_out.alloc((size_t)n * 4));
  CK(cudaStreamSynchronize(m->stream));
  CK(cudaStreamBeginCapture(m->stream, cudaStreamCaptureModeThreadLocal));
  cudaMemcpyAsync(p->d_pos, p->h_pos, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice, m->stream);
  k_query<<<(unsigned)((n + 127) / 128), 128, 0, m->stream>>>(m->g, m->cobs, m->occ, m->l_occ, p->d_pos, n, 1, p->d_out, p->d_out + n);
  cudaMemcpyAsync(p->h_out, p->d_out, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToHost, m->stream);
  CK(cudaStreamEndCapture(m->stream, &p->graph));
  CK(cudaGraphInstantiate(&p->exec, p->graph, 0));
  *out = p.release();
  return FIESTA_OK;
}
double *fiesta_query_plan_positions(fiesta_query_plan *p) { return p ? p->h_pos.get() : nullptr; }
const double *fiesta_query_plan_distances(const fiesta_query_plan *p) { return p ? p->h_out.get() : nullptr; }
const double *fiesta_query_plan_gradients(const fiesta_query_plan *p) { return p ? p->h_out + p->n : nullptr; }
int fiesta_query_plan_run(fiesta_query_plan *p) {
  if (!p) return FIESTA_ERR_INVALID;
  CK(cudaSetDevice(p->m->device));
  CK(cudaGraphLaunch(p->exec, p->m->stream));
  p->m->st.kernel_launches++;
  CK(cudaStreamSynchronize(p->m->stream));
  return FIESTA_OK;
}

// ---- pinned host mirror of the distance records (SURVEY.md 8(f) #3): planners that call GetDistance / GetDistWithGradTrilinear one
// position at a time (ESDFMap.cpp:467-540) read page-locked host memory instead of paying a device round trip per call.  The
// mirror holds the packed 4-byte records in the device layout; a refresh diffs the dirty box against a device-side shadow of what
// the host already has, ships only the changed (index, record) pairs and patches them in.  Every record is one aligned 32-bit
// word, so a reader racing a refresh sees the old or the new record of a voxel, never a torn one.
struct fiesta_host_mirror {
  fiesta_map *m;
  FbPinned<uint32_t> h_rec;       // [ptotal]; fiesta_host_mirror_records hands this address out: never reallocated
  FbDev<uint32_t> d_shadow;       // [ptotal]: the records the host holds
  FbDev<uint2> d_chg;             // change list, device + pinned
  FbPinned<uint2> h_chg;
  FbDev<unsigned> d_n;
  FbPinned<unsigned> h_n;
  int64_t last_changed, last_scanned, refreshes, full_copies;
};
__global__ void k_mirror_diff(FbGeom g, const uint32_t *cobs, uint32_t *shadow, int lx, int ly, int lz, int ex, int ey, int ez, uint2 *chg,
                              unsigned cap, unsigned *n) {
  const long long vol = (long long)ex * ey * ez;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < vol; t += (long long)gridDim.x * blockDim.x) {
    const int z = lz + (int)(t % ez), y = ly + (int)(t / ez % ey), x = lx + (int)(t / ((long long)ez * ey));
    const long long ii = fb_ii(g, x, y, z);
    const uint32_t c = cobs[ii];
    const bool diff = c != shadow[ii];
    if (diff) shadow[ii] = c;
    const unsigned slot = fb_warp_append(n, diff);
    if (diff && slot < cap) chg[slot] = make_uint2((unsigned)ii, c);      // on overflow the host falls back to one full copy
  }
}
void fiesta_host_mirror_destroy(fiesta_host_mirror *p) {
  if (!p) return;
  cudaSetDevice(p->m->device);
  cudaStreamSynchronize(p->m->stream);
  if (p->m->mirror == p) p->m->mirror = nullptr;
  delete p;
}
static int mirror_full_copy(fiesta_host_mirror *p) {
  fiesta_map *m = p->m;
  const size_t P = (size_t)m->g.ptotal;
  CK(cudaMemcpyAsync(p->d_shadow, m->cobs, P * 4, cudaMemcpyDeviceToDevice, m->stream));
  CK(cudaMemcpyAsync(p->h_rec, m->cobs, P * 4, cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  p->full_copies++;
  return FIESTA_OK;
}
int fiesta_host_mirror_create(fiesta_map *m, fiesta_host_mirror **out) {
  if (!m || !out) { set_error("fiesta_host_mirror_create: null argument"); return FIESTA_ERR_INVALID; }
  *out = nullptr;
  if (m->mirror) { set_error("fiesta_host_mirror_create: this map already has a host mirror"); return FIESTA_ERR_INVALID; }
  CK(cudaSetDevice(m->device));
  std::unique_ptr<fiesta_host_mirror> p(new (std::nothrow) fiesta_host_mirror());
  if (!p) return FIESTA_ERR_INVALID;
  p->m = m;
  const size_t P = (size_t)m->g.ptotal;
  size_t cap_chg = P / 32 > (1u << 20) ? P / 32 : (1u << 20);
  if (cap_chg > P) cap_chg = P;
  if (const char *e = getenv("FIESTA_MIRROR_CAP")) { const long v = atol(e); if (v > 0 && (size_t)v < cap_chg) cap_chg = (size_t)v; }   // tests: force the bulk-copy path
  CK(p->h_rec.alloc(P));
  CK(p->h_chg.alloc(cap_chg));
  CK(p->h_n.alloc(1));
  CK(p->d_shadow.alloc(P));
  CK(p->d_chg.alloc(cap_chg));
  CK(p->d_n.alloc(1));
  int r = flush_events(m);
  if (!r) r = mirror_full_copy(p.get());
  if (r) return r;
  p->full_copies = 0;
  m->mirror = p.release();                                                // the dirty box is kept: the first refresh rescans it
  *out = m->mirror;
  return FIESTA_OK;
}
int fiesta_host_mirror_refresh(fiesta_host_mirror *p, int64_t *n_changed) {
  if (!p) return FIESTA_ERR_INVALID;
  fiesta_map *m = p->m;
  CK(cudaSetDevice(m->device));
  p->last_changed = p->last_scanned = 0;
  p->refreshes++;
  if (n_changed) *n_changed = 0;
  if (!m->dirty_any) return FIESTA_OK;
  const FbGeom &g = m->g;
  int lo[3], ex[3];
  const int gs[3] = {g.gx, g.gy, g.gz};
  bool empty = false;
  for (int i = 0; i < 3; ++i) {
    lo[i] = m->dirty_lo[i] < 0 ? 0 : m->dirty_lo[i];
    const int hi = m->dirty_hi[i] > gs[i] - 1 ? gs[i] - 1 : m->dirty_hi[i];
    ex[i] = hi - lo[i] + 1;
    if (ex[i] <= 0) empty = true;
  }
  m->dirty_any = false;
  if (empty) return FIESTA_OK;
  const long long vol = (long long)ex[0] * ex[1] * ex[2];
  p->last_scanned = vol;
  CK(cudaMemsetAsync(p->d_n, 0, 4, m->stream));
  const long long want = (vol + 255) / 256;
  const unsigned blocks = (unsigned)(want < 148ll * 16 ? want : 148ll * 16);
  k_mirror_diff<<<blocks, 256, 0, m->stream>>>(g, m->cobs, p->d_shadow, lo[0], lo[1], lo[2], ex[0], ex[1], ex[2], p->d_chg, (unsigned)p->d_chg.size(), p->d_n);
  m->st.kernel_launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(p->h_n, p->d_n, 4, cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  const size_t n = *p->h_n;
  p->last_changed = (int64_t)n;
  if (n_changed) *n_changed = (int64_t)n;
  if (n == 0) return FIESTA_OK;
  if (n > p->d_chg.size()) return mirror_full_copy(p);                    // the shadow is already current; one bulk copy brings the host up
  CK(cudaMemcpyAsync(p->h_chg, p->d_chg, n * sizeof(uint2), cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  for (size_t i = 0; i < n; ++i) {
    volatile uint32_t *dst = p->h_rec + p->h_chg[i].x;                     // one aligned 32-bit store per record
    *dst = p->h_chg[i].y;
  }
  return FIESTA_OK;
}
double fiesta_host_mirror_get_distance_pos(const fiesta_host_mirror *p, const double pos[3]) {
  return p ? fb_query_distance(p->m->g, p->h_rec, pos) : (double)FIESTA_UNDEFINED;
}
double fiesta_host_mirror_get_distance_vox(const fiesta_host_mirror *p, const int vox[3]) {
  return p ? fb_get_distance_vox(p->m->g, p->h_rec, vox[0], vox[1], vox[2]) : (double)FIESTA_INFINITY;
}
double fiesta_host_mirror_get_dist_grad_trilinear(const fiesta_host_mirror *p, const double pos[3], double grad[3]) {
  if (!p) { grad[0] = grad[1] = grad[2] = 0; return -1.0; }
  return fb_query_trilinear(p->m->g, p->h_rec, pos, grad);
}
int fiesta_host_mirror_get_distance_batch_pos(const fiesta_host_mirror *p, const double *pos, int64_t n, double *out) {
  if (!p || (n > 0 && (!pos || !out))) return FIESTA_ERR_INVALID;
  for (int64_t i = 0; i < n; ++i) out[i] = fb_query_distance(p->m->g, p->h_rec, pos + 3 * i);
  return FIESTA_OK;
}
int fiesta_host_mirror_get_dist_grad_trilinear_batch(const fiesta_host_mirror *p, const double *pos, int64_t n, double *out, double *grad) {
  if (!p || (n > 0 && (!pos || !out || !grad))) return FIESTA_ERR_INVALID;
  for (int64_t i = 0; i < n; ++i) out[i] = fb_query_trilinear(p->m->g, p->h_rec, pos + 3 * i, grad + 3 * i);
  return FIESTA_OK;
}
const uint32_t *fiesta_host_mirror_records(const fiesta_host_mirror *p) { return p ? p->h_rec.get() : nullptr; }
int fiesta_host_mirror_stats(const fiesta_host_mirror *p, int64_t out[4]) {
  if (!p || !out) return FIESTA_ERR_INVALID;
  out[0] = p->last_changed; out[1] = p->last_scanned; out[2] = p->refreshes; out[3] = p->full_copies;
  return FIESTA_OK;
}

// ---- exports
static int run_export(fiesta_map *m, double *dist, int *cobs3, double *occ, int *hit, int *tot) {
  CK(cudaSetDevice(m->device));
  const size_t G = (size_t)m->g.total;
  FbDev<double> dd, dof; FbDev<int> dc, dh, dt;
  cudaError_t e = cudaSuccess;
  if (dist) e = dd.alloc(G);
  if (!e && occ) e = dof.alloc(G);
  if (!e && cobs3) e = dc.alloc(G * 3);
  if (!e && hit) { e = dh.alloc(G); if (!e) e = dt.alloc(G); }
  if (!e) {
    k_export<<<(unsigned)((G + 255) / 256), 256, 0, m->stream>>>(m->g, m->cobs, m->occ, m->cnt, dd, dc, dof, dh, dt);
    m->st.kernel_launches++;
    e = cudaGetLastError();
  }
  if (!e && dist) e = cudaMemcpyAsync(dist, dd, G * 8, cudaMemcpyDeviceToHost, m->stream);
  if (!e && occ) e = cudaMemcpyAsync(occ, dof, G * 8, cudaMemcpyDeviceToHost, m->stream);
  if (!e && cobs3) e = cudaMemcpyAsync(cobs3, dc, G * 12, cudaMemcpyDeviceToHost, m->stream);
  if (!e && hit) { e = cudaMemcpyAsync(hit, dh, G * 4, cudaMemcpyDeviceToHost, m->stream); if (!e) e = cudaMemcpyAsync(tot, dt, G * 4, cudaMemcpyDeviceToHost, m->stream); }
  if (!e) e = cudaStreamSynchronize(m->stream);
  if (e != cudaSuccess) { set_error("export failed: %s", cudaGetErrorString(e)); return FIESTA_ERR_CUDA; }
  return FIESTA_OK;
}
int fiesta_export_distance(fiesta_map *m, double *out) { return (!m || !out) ? FIESTA_ERR_INVALID : run_export(m, out, nullptr, nullptr, nullptr, nullptr); }
int fiesta_export_closest_obstacle(fiesta_map *m, int *out) { return (!m || !out) ? FIESTA_ERR_INVALID : run_export(m, nullptr, out, nullptr, nullptr, nullptr); }
int fiesta_export_occupancy(fiesta_map *m, double *out) { return (!m || !out) ? FIESTA_ERR_INVALID : run_export(m, nullptr, nullptr, out, nullptr, nullptr); }
int fiesta_export_counters(fiesta_map *m, int *hit, int *tot) {
  if (!m || !hit || !tot) return FIESTA_ERR_INVALID;
  int r = flush_events(m);
  if (r) return r;
  return run_export(m, nullptr, nullptr, nullptr, hit, tot);
}

// ---- x-slab sharding
static void fill_esdf_args(fiesta_map *m, FbEsdfArgs &a) {
  a.cobs = m->cobs; a.cobs_b = m->cobs_b; a.occ = m->occ; a.occbits = m->occbits; a.tile_flag = m->tile_flag; a.nb_flag = m->nb_flag;
  for (int k = 0; k < 2; ++k) { a.list[k] = m->list[k]; a.changed[k] = m->changed[k]; a.changed_bbox[k] = m->changed_bbox[k]; }
  a.ctr = m->d_ctr; a.l_occ = m->l_occ; a.tile_x_lo = m->tile_x_lo; a.tile_x_hi = m->tile_x_hi; a.dbg = nullptr;
}
int fiesta_set_shard(fiesta_map *m, int rank, int world, fiesta_shard_info *out) {
  if (!m || world < 1 || rank < 0 || rank >= world) { set_error("fiesta_set_shard: bad rank/world"); return FIESTA_ERR_INVALID; }
  if (m->mode != FIESTA_MODE_FAST) { set_error("fiesta_set_shard: sharding is implemented for FIESTA_MODE_FAST only"); return FIESTA_ERR_INVALID; }
  if (world > m->g.tx) { set_error("fiesta_set_shard: more ranks than 8-voxel tile columns"); return FIESTA_ERR_LIMIT; }
  for (int r = 0; r < world; ++r) {                                       // every slab exchanges 2 x-layers per internal face
    const int lo = (int)((long long)m->g.tx * r / world) * 8, hi = (int)((long long)m->g.tx * (r + 1) / world) * 8;
    if ((hi < m->g.gx ? hi : m->g.gx) - lo < 2) { set_error("fiesta_set_shard: a slab would be thinner than the 2-layer ghost exchanged per face (too many ranks for grid_x)"); return FIESTA_ERR_LIMIT; }
  }
  m->shard_rank = rank; m->shard_world = world;
  m->tile_x_lo = (int)((long long)m->g.tx * rank / world);
  m->tile_x_hi = (int)((long long)m->g.tx * (rank + 1) / world);
  if (!m->d_halo_changed) CK(m->d_halo_changed.alloc(4));
  if (out) {
    out->rank = rank; out->world = world;
    out->x_begin = m->tile_x_lo * 8; out->x_end = m->tile_x_hi * 8 < m->g.gx ? m->tile_x_hi * 8 : m->g.gx;
    out->has_lo = rank > 0; out->has_hi = rank + 1 < world;
    out->layer_words = 2ll * m->g.gy * m->g.pz;
  }
  return FIESTA_OK;
}
int fiesta_shard_pack(fiesta_map *m, uint32_t *d_lo, uint32_t *d_hi) {
  if (!m) return FIESTA_ERR_INVALID;
  CK(cudaSetDevice(m->device));
  const long long per = (long long)m->g.gy * m->g.pz;
  const int x0 = m->tile_x_lo * 8, x1 = m->tile_x_hi * 8 < m->g.gx ? m->tile_x_hi * 8 : m->g.gx;
  if (d_lo && m->shard_rank > 0) CK(cudaMemcpyAsync(d_lo, m->cobs + (long long)x0 * per, 2 * per * 4, cudaMemcpyDeviceToDevice, m->stream));
  if (d_hi && m->shard_rank + 1 < m->shard_world) CK(cudaMemcpyAsync(d_hi, m->cobs + (long long)(x1 - 2) * per, 2 * per * 4, cudaMemcpyDeviceToDevice, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  return FIESTA_OK;
}
int fiesta_shard_ingest(fiesta_map *m, const uint32_t *d_from_lo, const uint32_t *d_from_hi, int64_t *changed) {
  if (!m || !changed) return FIESTA_ERR_INVALID;
  CK(cudaSetDevice(m->device));
  mark_dirty(m);
  FbEsdfArgs a; fill_esdf_args(m, a);
  const int x0 = m->tile_x_lo * 8, x1 = m->tile_x_hi * 8 < m->g.gx ? m->tile_x_hi * 8 : m->g.gx;
  CK(cudaMemsetAsync(m->d_halo_changed, 0, 4, m->stream));
  if (d_from_lo && m->shard_rank > 0) { CK(fb_esdf_halo_ingest(m->g, a, d_from_lo, x0 - 2, 2, m->tile_x_lo, m->d_halo_changed, m->stream)); m->st.kernel_launches++; }
  if (d_from_hi && m->shard_rank + 1 < m->shard_world) { CK(fb_esdf_halo_ingest(m->g, a, d_from_hi, x1, 2, m->tile_x_hi - 1, m->d_halo_changed, m->stream)); m->st.kernel_launches++; }
  unsigned h = 0;
  CK(cudaMemcpyAsync(&h, m->d_halo_changed, 4, cudaMemcpyDeviceToHost, m->stream));
  CK(cudaStreamSynchronize(m->stream));
  *changed = h;
  return FIESTA_OK;
}
int fiesta_shard_relax(fiesta_map *m, int64_t *changed) {
  if (!m || !changed) return FIESTA_ERR_INVALID;
  CK(cudaSetDevice(m->device));
  mark_dirty(m);
  FbEsdfArgs a; fill_esdf_args(m, a);
  k_reset_esdf_ctr<<<1, 1, 0, m->stream>>>(m->d_ctr);
  CK(fb_esdf_wavefront(m->g, a, m->tmap, m->wf_blocks, m->stream));
  const int x0 = m->tile_x_lo * 8, x1 = m->tile_x_hi * 8 < m->g.gx ? m->tile_x_hi * 8 : m->g.gx;
  if (m->shard_rank > 0) CK(fb_esdf_halo_retire(m->g, m->cobs, x0 - 2, 2, m->stream));
  if (m->shard_rank + 1 < m->shard_world) CK(fb_esdf_halo_retire(m->g, m->cobs, x1, 2, m->stream));
  m->st.kernel_launches += 4;
  int r;
  if ((r = fetch_counters(m))) return r;
  *changed = (int64_t)m->h_ctr->voxels_changed;
  m->st.voxels_changed += *changed; m->st.generations += m->h_ctr->generations; m->st.tile_visits += (int64_t)m->h_ctr->tile_visits;
  return FIESTA_OK;
}

int fiesta_get_point_cloud(fiesta_map *m, int lo, int hi, float *out, int64_t cap, int64_t *count) {
  if (!m || !count || (cap > 0 && !out)) return FIESTA_ERR_INVALID;
  CK(cudaSetDevice(m->device));
  long long c = 0;
  CK(fb_vis_point_cloud(m->g, m->occ, m->l_occ, lo, hi, out, cap, &c, m->stream));
  m->st.kernel_launches += 3;
  *count = c;
  return FIESTA_OK;
}
int fiesta_get_slice_marker(fiesta_map *m, int slice, double max_dist, double *xyz, float *rgba, int64_t cap, int64_t *count) {
  if (!m || !count || (cap > 0 && (!xyz || !rgba))) return FIESTA_ERR_INVALID;
  CK(cudaSetDevice(m->device));
  long long c = 0;
  CK(fb_vis_slice(m->g, m->cobs, slice, max_dist, xyz, rgba, cap, &c, m->stream));
  m->st.kernel_launches += 3;
  *count = c;
  return FIESTA_OK;
}

int fiesta_get_stats(fiesta_map *m, fiesta_stats *out) {
  if (!m || !out) return FIESTA_ERR_INVALID;
  *out = m->st;
  return FIESTA_OK;
}
int fiesta_synchronize(fiesta_map *m) {
  if (!m) return FIESTA_ERR_INVALID;
  CK(cudaSetDevice(m->device));
  CK(cudaStreamSynchronize(m->stream));
  return FIESTA_OK;
}

}  // extern "C"
