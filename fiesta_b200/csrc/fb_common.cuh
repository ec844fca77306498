// fiesta_b200 -- shared device/host definitions for the sm_100a kernels.
//
// HBM layout (all arrays dense, z fastest, index ii = (x*Gy + y)*Pz + z with Pz = Gz rounded up to 4 so that the
// TMA global strides are 16-byte multiples; ii equals the reference's linear index (ESDFMap.cpp:91) when Gz % 4 == 0):
//   cobs   u32   closest-obstacle record.  0 = never observed (reference distance_ = -10000, ESDFMap.cpp:198),
//                1 = observed, no obstacle yet (+10000, ESDFMap.cpp:247), >= 2 = packed obstacle coordinate
//                ((x+1)<<20 | y<<10 | z) in bits 0..30.  The distance is NOT stored: it is |voxel - obstacle| * resolution
//                (ESDFMap.cpp:122-123) recomputed from the integer coordinates, which is exact.
//                Bit 31 (FB_FRESH) = "this record changed in the previous wavefront generation", the device form of
//                "this voxel is in update_queue_" (ESDFMap.cpp:339-392); it is only ever set while UpdateESDF runs.
//   cobs_b u32   staging copy written by the wavefront kernel for tiles that changed in a generation.
//   occ    f64   log-odds occupancy_buffer_ (ESDFMap.h:84).
//   cnt    u64   {num_hit_:32 | num_miss_(=all observations):32} so one 64-bit atomicAdd counts an event (ESDFMap.cpp:424-425).
//   stamp  2xu32 per-frame ray stamps, the device form of Fiesta's set_free_/set_occ_ (Fiesta.h:60-64,107-110).
//   occbit u32/32 voxels  Exist() bitmap (ESDFMap.cpp:16-22), kept L2-resident for the dependant scan.
// The occupancy queue (occupancy_queue_, ESDFMap.h:96) is kept at 8^3-tile granularity: the first observation of a voxel
// since the last integration marks its tile; UpdateOccupancy then streams the counters of the marked tiles.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "fb_buf.h"

#define FB_UNKNOWN 0u
#define FB_INF 1u
#define FB_TILE 8
#define FB_HALO 2
#define FB_BOX (FB_TILE + 2 * FB_HALO)            // 12 : x and y extent of the staged box
#define FB_ZPAD 4                                 // TMA needs the innermost start coordinate 16-byte aligned: the box
#define FB_BOXZ (FB_TILE + 2 * FB_ZPAD)           // 16   starts at z0 - 4 (not z0 - 2) and is 16 voxels long in z
#define FB_BOX_WORDS (FB_BOX * FB_BOX * FB_BOXZ)  // 2304
#define FB_FRESH 0x80000000u
// EXACT mode (which never uses FRESH) keeps in the same bit, between calls, "distance_ forced to +infinity_ while the closest
// obstacle and its dependant-list link are kept" -- the state UpdateOccupancy(false) leaves behind for a voxel outside the
// previous update box (ESDFMap.cpp:256-259).  Cleared by the next write of the record.
#define FB_DINF 0x80000000u
#define FB_CODE_MASK 0x7fffffffu
#define FB_MAX_GX 2046
#define FB_MAX_GY 1024
#define FB_MAX_GZ 1024
// free-space claim word (stamp[0]): [frame tag:2 | ray index:19 | position in that ray's list:11]; 0 = never claimed.
// endpoint owner word (stamp[1]):   [owner frame tag:13 | ~ray index:19], atomicMax keeps the newest frame / lowest ray.
#define FB_RAY_BITS 19
#define FB_RAY_MASK ((1u << FB_RAY_BITS) - 1u)
#define FB_POS_BITS 11
#define FB_POS_MASK ((1u << FB_POS_BITS) - 1u)
#define FB_CLAIM_FRAME_SHIFT (FB_RAY_BITS + FB_POS_BITS)
#define FB_MAX_CLAIM_FRAME 3u
#define FB_MAX_OWNER_FRAME ((1u << (32 - FB_RAY_BITS)) - 1u)
#define FB_MAX_ROUNDS 2000u
#define FB_LIST_IDX_MASK 0x3fffffffu
#define FB_CLS_COUNT 0u   // NORMAL voxel inside the update box: counted + stamp logic (Fiesta.h:248-275)
#define FB_CLS_SKIP 1u    // len > max_ray_length or centre not in map: `continue` (Fiesta.h:245, 253)
#define FB_CLS_STOP 2u    // len < min_ray_length: `break` (Fiesta.h:243)
#define FB_CLS_STAMP 3u   // in map but outside the update box: stamp logic only (ESDFMap.cpp:420-421)

struct FbGeom {
  int gx, gy, gz, pz;          // grid_size_ and padded z pitch
  int gyz;                     // grid_size_yz_ (reference linear index)
  int total;                   // grid_total_size_
  long long ptotal;            // gx*gy*pz, size of the device arrays
  int tx, ty, tz, ntiles;      // 8^3 tile grid
  double origin[3], res, res_inv;
  double min_range[3], max_range[3];
  int min_vec[3], max_vec[3], last_min_vec[3], last_max_vec[3];
  int box_is_full;             // update box == whole grid (SetOriginalRange)
};

struct FbCounters {
  unsigned n_touched, n_ins, n_del;   // n_touched: voxels integrated by the last UpdateOccupancy
  unsigned n_touch_tiles;      // tiles holding pending observations (the occupancy queue)
  unsigned pad_x0;
  unsigned n_list[2];          // active-tile work lists (ping-pong)
  unsigned n_changed[2];       // changed-tile lists by generation parity
  unsigned next_work[4];       // dynamic tile fetch counters: [phase1 even, phase1 odd, phase2 even, phase2 odd]
  unsigned gen_stamp;          // monotonically increasing generation stamp for tile_flag dedupe
  unsigned generations;
  unsigned ray_work[3];        // number of rays that have to walk in a round, rotating per round
  unsigned ray_pad0;
  unsigned rays_cast, rays_dropped, ray_rounds, ray_error;
  unsigned long long ray_voxels;
  unsigned long long voxels_changed, voxels_reset, tile_visits;
};

__host__ __device__ __forceinline__ uint32_t fb_pack(int x, int y, int z) {
  return ((uint32_t)(x + 1) << 20) | ((uint32_t)y << 10) | (uint32_t)z;
}
__host__ __device__ __forceinline__ void fb_unpack(uint32_t c, int &x, int &y, int &z) {
  x = (int)((c & FB_CODE_MASK) >> 20) - 1; y = (int)((c >> 10) & 1023u); z = (int)(c & 1023u);
}
__host__ __device__ __forceinline__ long long fb_ii(const FbGeom &g, int x, int y, int z) {
  return ((long long)x * g.gy + y) * g.pz + z;
}
__host__ __device__ __forceinline__ bool fb_in_grid(const FbGeom &g, int x, int y, int z) {
  return x >= 0 && x < g.gx && y >= 0 && y < g.gy && z >= 0 && z < g.gz;
}
// ESDFMap::VoxInRange (ESDFMap.cpp:63-72)
__host__ __device__ __forceinline__ bool fb_in_range(const FbGeom &g, int x, int y, int z) {
  return x >= g.min_vec[0] && x <= g.max_vec[0] && y >= g.min_vec[1] && y <= g.max_vec[1] && z >= g.min_vec[2] && z <= g.max_vec[2];
}
__host__ __device__ __forceinline__ bool fb_in_last_range(const FbGeom &g, int x, int y, int z) {
  return x >= g.last_min_vec[0] && x <= g.last_max_vec[0] && y >= g.last_min_vec[1] && y <= g.last_max_vec[1] &&
         z >= g.last_min_vec[2] && z <= g.last_max_vec[2];
}

#ifdef __CUDACC__
// Warp-aggregated append: lanes with `pred` get consecutive slots from one atomicAdd per warp.
__device__ __forceinline__ unsigned fb_warp_append(unsigned *counter, bool pred) {
  unsigned mask = __ballot_sync(__activemask(), pred);
  unsigned slot = 0;
  if (mask) {
    int leader = __ffs(mask) - 1;
    unsigned lane = threadIdx.x & 31;
    unsigned base = 0;
    if ((int)lane == leader) base = atomicAdd(counter, (unsigned)__popc(mask));
    base = __shfl_sync(__activemask(), base, leader);
    slot = base + __popc(mask & ((1u << lane) - 1u));
  }
  return slot;
}
#endif

#ifdef __CUDACC__
struct FbTouch {
  unsigned long long *cnt;
  uint32_t *touch_flag, *touch_list;
  unsigned epoch;
  FbCounters *ctr;
  unsigned long long *tkey;   // exact mode only (else nullptr): per-voxel serial time of the first pending observation, epoch-coded
  unsigned long long key_hi;  // exact mode: integration epoch << FB_KEY_BITS
};
// Exact mode: tkey[v] = (epoch << 44) | (2^44-1 - t), t = serial time of an observation within the current integration epoch
// (the observations between two UpdateOccupancy calls).  atomicMax keeps the EARLIEST observation of the NEWEST epoch, so the
// array is never reset: entries of older epochs simply lose.
#define FB_KEY_BITS 44
#define FB_KEY_MASK ((1ull << FB_KEY_BITS) - 1ull)
// One observation of voxel ii (ESDFMap.cpp:424-435): num_miss_++, num_hit_ += occ; the first one since the last
// integration (num_miss_ == 1) queues the voxel.  The queue is kept per 8^3 tile: a tile is queued when it holds any pending
// observation, which is the same set as "some voxel of it saw its first observation" -- so the counter update needs no return
// value (a fire-and-forget RED instead of a round trip).  Exact mode additionally keeps the serial time `key` of the voxel's
// earliest pending observation (= its position in occupancy_queue_) with one more RED.
__device__ __forceinline__ void fb_touch(const FbGeom &g, const FbTouch &t, unsigned ii, unsigned occ, unsigned long long key) {
  atomicAdd(&t.cnt[ii], ((unsigned long long)occ << 32) | 1ull);
  if (t.tkey) atomicMax(&t.tkey[ii], t.key_hi | (FB_KEY_MASK - (key < FB_KEY_MASK ? key : FB_KEY_MASK)));
  const unsigned z = ii % (unsigned)g.pz, xy = ii / (unsigned)g.pz, y = xy % (unsigned)g.gy, x = xy / (unsigned)g.gy;
  const unsigned tile = ((x >> 3) * g.ty + (y >> 3)) * g.tz + (z >> 3);
  if (__ldcg(&t.touch_flag[tile]) != t.epoch && atomicExch(&t.touch_flag[tile], t.epoch) != t.epoch)
    t.touch_list[atomicAdd(&t.ctr->n_touch_tiles, 1u)] = tile;
}
#endif

// ---- host-side launch interface (defined in fb_esdf.cu / fb_raycast.cu) ----
struct FbEsdfArgs {
  uint32_t *cobs, *cobs_b;
  const double *occ;
  const uint32_t *occbits;
  uint32_t *tile_flag;   // generation stamp for which a tile is queued (dedupe)
  uint32_t *nb_flag;     // generation stamp for which a NEIGHBOUR (or a seed/reset) queued the tile: real work to do
  uint32_t *list[2];
  uint32_t *changed[2];
  uint32_t *changed_bbox[2];
  FbCounters *ctr;
  double l_occ;
  int tile_x_lo, tile_x_hi;  // tile columns [lo, hi) this map relaxes (x-slab sharding; whole grid when unsharded)
  unsigned long long *dbg;   // optional per-generation trace: {nwork, nchanged, t_phase1_ns, t_phase2_ns} x 256 (FIESTA_DEBUG_WF=1)
};

struct FbRayArgs {
  const float *xyz;       // n points
  long long n;
  double T[16];
  double org[3];          // raycast_origin_
  double start[3];        // org / res
  double bmin[3], bmax[3];  // l_cornor/res, r_cornor/res
  double min_len, max_len;
  int lattice_ok;         // host-verified: Pos2Vox((c+0.5)*res) == c - lattice_off for every DDA voxel c inside the box
  int lattice_off[3];
  unsigned long long *cnt;
  uint32_t *stamp[2];
  uint32_t *touch_flag, *touch_list;
  unsigned touch_epoch;
  unsigned long long *tkey;   // exact mode (else nullptr)
  unsigned long long key_hi;  // exact mode: integration epoch << FB_KEY_BITS
  unsigned long long key_base;  // serial time of this frame's first observation within the epoch
  uint32_t *ray_list;     // [n][cap] row-major, reversed (t = 0 is the voxel before the last emitted one)
  int *ray_len, *ray_reach;
  unsigned *ray_dirty;    // lowest list position a lower ray displaced this ray from since its last walk (FB_RAY_CLEAN: none)
  int cap;
  unsigned frame_tag;     // claim frame tag (1..3)
  unsigned owner_tag;     // endpoint-owner frame tag
  unsigned max_rounds;
  FbCounters *ctr;
  unsigned long long *dbg;  // FIESTA_DEBUG_RAY: per-round {work, check ns, walk ns}
};

cudaError_t fb_esdf_make_tensor_map(CUtensorMap *out, const FbGeom &g, uint32_t *cobs, char *err, int errlen);
cudaError_t fb_esdf_seed_inserts(const FbGeom &g, const FbEsdfArgs &a, const uint32_t *ins, unsigned n, cudaStream_t s);
cudaError_t fb_esdf_delete_scan(const FbGeom &g, const FbEsdfArgs &a, cudaStream_t s);
cudaError_t fb_esdf_wavefront(const FbGeom &g, const FbEsdfArgs &a, const CUtensorMap &tmap, int nblocks, cudaStream_t s);
int fb_esdf_wavefront_blocks(int device);
cudaError_t fb_esdf_halo_ingest(const FbGeom &g, const FbEsdfArgs &a, const uint32_t *recv, int x_first, int nlayers, int own_tile_x, unsigned *d_nchanged, cudaStream_t s);
cudaError_t fb_esdf_halo_retire(const FbGeom &g, uint32_t *cobs, int x_first, int nlayers, cudaStream_t s);
cudaError_t fb_ray_frame(const FbGeom &g, const FbRayArgs &a, int nblocks_resolve, cudaStream_t s, int *launches);
int fb_ray_resolve_blocks(int device);
cudaError_t fb_vis_point_cloud(const FbGeom &g, const double *occ, double l_occ, int zlo, int zhi, float *h_out, long long cap, long long *count, cudaStream_t s);
cudaError_t fb_vis_slice(const FbGeom &g, const uint32_t *cobs, int slice, double max_dist, double *h_xyz, float *h_rgba, long long cap, long long *count, cudaStream_t s);
struct FbDepthRel { double m[16]; };
struct fiesta_depth_params;
cudaError_t fb_depth_to_cloud(const uint16_t *d_img, const uint16_t *d_last, int rows, int cols, const fiesta_depth_params &p, int filter_on,
                              const FbDepthRel &rel, float *d_pts, uint8_t *d_flags, uint32_t *d_sel, float *d_cloud, unsigned *d_count,
                              FbDev<uint8_t> &tmp, unsigned *h_n, cudaStream_t s);
