// fiesta_b200 -- ORDER-EXACT mode of UpdateOccupancy / UpdateESDF (FIESTA_MODE_EXACT).
//
// The reference result is a function of its sequential FIFO order (/root/reference/src/ESDFMap.cpp:273-398): seeds in
// insert_queue_/delete_queue_ order, dependants of a deleted obstacle in LIFO list order (:301-334), neighbours in dirs_
// order, strict improvement, and every queue element seeing the writes of all earlier elements.  This file reproduces
// that order with data-parallel kernels (the CPU model of exactly this formulation is oracle/exact_model.c, which matches
// the sequential reference voxel for voxel):
//
//  * E3, the FIFO relaxation loop, is one persistent kernel (fb_xrelax.cu): every FIFO generation is one ordered list of
//    entries whose behaviours are resolved by a fixpoint over timestamped offers; see the header of that file.
//  * The doubly linked dependant lists are replaced by a per-voxel link time LS (time of the last relink; every accepted
//    write relinks at the list front, :24-42): dependants of deleted obstacles are found by a dense scan and ordered by
//    (position of the obstacle in delete_queue_, link time descending) = the order of the reference's list walk; their
//    re-seeding ("first valid neighbour in dirs_ order", :308-321, which sees earlier re-seeded dependants) is iterated to
//    its fixpoint the same way.
//  * occupancy_queue_ order = order of first observation: every observation carries its serial time (host event number,
//    or point index and position along the ray) and the per-voxel earliest one is kept (fb_touch).  The integration of a
//    voxel does not depend on its place in the queue, only the order of the insert_queue_ / delete_queue_ pushes does:
//    the tile-streamed k_integrate<true> (fb_map.cu) stages the threshold crossings with that time and
//    fb_exact_queue_crossings sorts just those, so the queues come out in the reference's order.
#include <cub/cub.cuh>
#include <stdio.h>
#include <stdlib.h>
#include <algorithm>
#include <chrono>
#include "fb_common.cuh"
#include "fb_exact.h"

#define XNONE 0xffffffffu
#define XMB_NONE 0xffffffffffffffffull

__device__ __forceinline__ void x_coords(const FbGeom &g, uint32_t ii, int &x, int &y, int &z) {
  z = ii % (unsigned)g.pz; const unsigned xy = ii / (unsigned)g.pz; y = xy % (unsigned)g.gy; x = xy / (unsigned)g.gy;
}
__device__ __forceinline__ unsigned x_d2(int x, int y, int z, uint32_t c) {
  int ox, oy, oz; fb_unpack(c, ox, oy, oz); ox -= x; oy -= y; oz -= z;
  return (unsigned)(ox * ox + oy * oy + oz * oz);
}
__device__ __forceinline__ unsigned x_dist_of(int x, int y, int z, uint32_t c) { return c < 2u ? 0xffffffffu : x_d2(x, y, z, c); }

// ------------------------------------------------------------------ E1: insert seeds
__global__ void k_x_flag_exist(const uint32_t *list, unsigned n, const double *occ, double l_occ, uint8_t *flags, int want) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = ((occ[list[i]] > l_occ) ? 1 : 0) == want;
}
__global__ void k_x_apply_seed(FbGeom g, const uint32_t *E, unsigned n, uint32_t *cobs, unsigned long long *LS, unsigned long long t0) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t ii = E[i];
  int x, y, z; x_coords(g, ii, x, y, z);
  cobs[ii] = fb_pack(x, y, z);                                 // closest_obstacle_ = self, distance_ = 0 (:286-287)
  LS[ii] = t0 + i;                                             // InsertIntoList(idx, idx) (:288)
}

// ------------------------------------------------------------------ E2: delete
__global__ void k_x_del_minpos(const uint32_t *del, unsigned n, const double *occ, double l_occ, uint32_t *scratch) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && !(occ[del[i]] > l_occ)) atomicMin(&scratch[del[i]], i);   // `if (!Exist(idx))` (:297); first occurrence wins
}
__global__ void k_x_del_flag(const uint32_t *del, unsigned n, const double *occ, double l_occ, const uint32_t *scratch, uint8_t *flags) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = (!(occ[del[i]] > l_occ) && scratch[del[i]] == i) ? 1 : 0;
}
__global__ void k_x_del_rank(const uint32_t *sel, unsigned n, uint32_t *scratch) {   // sel = deleted obstacles in queue order
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) scratch[sel[i]] = i;
}
// Dependants = voxels whose closest obstacle is a deleted one (the reference walks head_[idx] -> next_, :301).
// shift > 0: one combined sort key (rank << shift) | (low `shift` bits of ~LS); shift == 0: two keys for two stable sorts.
__global__ void k_x_scan_deps(FbGeom g, const uint32_t *cobs, const uint32_t *occbits, const uint32_t *rank, const unsigned long long *LS,
                              unsigned long long *k1, unsigned long long *k2, uint32_t *dv, unsigned *ndep, unsigned cap, int shift) {
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < g.ptotal; v += (long long)gridDim.x * blockDim.x) {
    const uint32_t c = cobs[v] & FB_CODE_MASK;
    bool dep = false;
    unsigned r = 0;
    if (c >= 2u) {
      int ox, oy, oz; fb_unpack(c, ox, oy, oz);
      const long long oi = fb_ii(g, ox, oy, oz);
      // a deleted obstacle is no longer occupied: the occupancy bitmap (1 bit per voxel, L2-resident) filters out the voxels
      // whose obstacle still stands before the random look-up into the per-voxel rank array
      if (!((__ldg(&occbits[oi >> 5]) >> (oi & 31)) & 1u)) { r = rank[oi]; dep = r != XNONE; }
    }
    const unsigned slot = fb_warp_append(ndep, dep);
    if (dep && slot < cap) {
      const unsigned long long inv = ~LS[v];                   // ~LS: most recently linked first
      if (shift) k1[slot] = ((unsigned long long)r << shift) | (inv & ((1ull << shift) - 1ull));
      else { k1[slot] = r; k2[slot] = inv; }
      dv[slot] = (uint32_t)v;
    }
  }
}
__global__ void k_x_unset(const uint32_t *list, unsigned n, uint32_t *scratch) {   // undo sparse writes: scratch stays all-XNONE between uses
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) scratch[list[i]] = XNONE;
}
__global__ void k_x_iota(uint32_t *a, unsigned n) { const unsigned i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) a[i] = i; }
__global__ void k_x_gather64(const unsigned long long *src, const uint32_t *idx, unsigned n, unsigned long long *dst) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) dst[i] = src[idx[i]];
}
__global__ void k_x_gather32(const uint32_t *src, const uint32_t *idx, unsigned n, uint32_t *dst) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) dst[i] = src[idx[i]];
}
__global__ void k_x_set_ord(const uint32_t *deps, unsigned n, uint32_t *ord, uint32_t *nc, uint8_t *nk) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { ord[deps[i]] = i; nc[i] = FB_INF; nk[i] = 24; }
}
__global__ void k_x_fill32(uint32_t *a, size_t n, uint32_t val) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) a[i] = val;
}
__global__ void k_x_fill64(unsigned long long *a, size_t n, unsigned long long val) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) a[i] = val;
}

// ================================================================== host side
#define XCK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { snprintf(X->err, sizeof(X->err), "%s: %s", #call, cudaGetErrorString(e__)); return e__; } } while (0)
static inline unsigned nblk(size_t n, unsigned t = 256) { return (unsigned)((n + t - 1) / t); }

// ordered compaction: out[0..count) = in[i] for flags[i] != 0, order kept
static cudaError_t x_select(FbExact *X, const uint32_t *in, const uint8_t *flags, uint32_t *out, unsigned n, unsigned *count, cudaStream_t s) {
  *count = 0;
  if (n == 0) return cudaSuccess;
  size_t bytes = 0;
  XCK(cub::DeviceSelect::Flagged(nullptr, bytes, in, flags, out, X->d_count.get(), (int)n, s));
  XCK(X->cub_tmp.reserve(bytes, s, false));
  XCK(cub::DeviceSelect::Flagged(X->cub_tmp.get(), bytes, in, flags, out, X->d_count.get(), (int)n, s));
  XCK(cudaMemcpyAsync(X->h_count, X->d_count, 4, cudaMemcpyDeviceToHost, s));
  XCK(cudaStreamSynchronize(s));
  *count = *X->h_count;
  return cudaSuccess;
}
static cudaError_t x_sort_pairs(FbExact *X, const unsigned long long *kin, unsigned long long *kout, const uint32_t *vin, uint32_t *vout, unsigned n, cudaStream_t s,
                                int key_bits = 64) {
  size_t bytes = 0;
  XCK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kin, kout, vin, vout, (int)n, 0, key_bits, s));
  XCK(X->cub_tmp.reserve(bytes, s, false));
  XCK(cub::DeviceRadixSort::SortPairs(X->cub_tmp.get(), bytes, kin, kout, vin, vout, (int)n, 0, key_bits, s));
  return cudaSuccess;
}
cudaError_t fb_exact_init(FbExact *X, const FbGeom &g, int device, cudaStream_t s) {
  const size_t P = (size_t)g.ptotal;
  XCK(fb_xrelax_init());
  X->relax_blocks = fb_xrelax_blocks(device);
  if (X->relax_blocks <= 0 || X->relax_blocks > FB_X_MAX_BLOCKS) { snprintf(X->err, sizeof(X->err), "k_x_relax does not fit on this device"); return cudaErrorInvalidConfiguration; }
  XCK(X->MB.alloc(P)); XCK(X->LS.alloc(P)); XCK(X->tkey.alloc(P));
  XCK(X->touched.alloc(P));
  XCK(X->SUM.alloc(P)); XCK(X->SUMg.alloc(P)); XCK(cudaMemsetAsync(X->SUMg, 0, P * 4, s));
  XCK(X->emask.alloc(P));
  XCK(X->wstamp.alloc(P)); XCK(cudaMemsetAsync(X->wstamp, 0, P * 4, s));
  for (int k = 0; k < 3; ++k) { XCK(X->W[k].alloc(P)); XCK(X->F[k].alloc(P)); }
  for (int k = 0; k < 2; ++k) XCK(X->E[k].alloc(P));
  X->dense_min = 16384u;
  if (const char *e = getenv("FIESTA_X_DENSE")) { long v = atol(e); if (v >= 0 && v <= (1 << 24)) X->dense_min = (unsigned)v; }
  X->small_max = FB_X_SMALL_DEFAULT;
  if (const char *e = getenv("FIESTA_X_SMALL")) { long v = atol(e); if (v >= 0 && v <= 65536) X->small_max = (unsigned)v; }
  XCK(X->slotc.alloc(((size_t)X->small_max + 1) * 32));
  // Per-frame work arrays (touched voxels, dependants of deleted obstacles, sort scratch) are sized up front for 1/8 of the
  // grid: growing them on demand puts an allocation and a free (device-wide synchronisations, milliseconds) inside UpdateESDF.
  const size_t c0 = P / 8 > (1u << 20) ? P / 8 : (1u << 20);
  for (FbDev<unsigned long long> *b : {&X->k1, &X->k2, &X->k1b, &X->k2b}) XCK(b->reserve(c0, s, false));
  for (FbDev<uint32_t> *b : {&X->dv, &X->idx[0], &X->idx[1], &X->deps, &X->nc[0], &X->nc[1], &X->sel}) XCK(b->reserve(c0, s, false));
  XCK(X->flags.reserve(c0, s, false)); XCK(X->flags2.reserve(c0, s, false));
  XCK(X->cub_tmp.reserve(c0 * 16 + (64u << 20), s, false));
  XCK(X->d_ctl.alloc(1)); XCK(cudaMemsetAsync(X->d_ctl, 0, sizeof(FbXCtl), s));
  XCK(X->h_ctl.alloc(1));
  XCK(X->d_count.alloc(4)); XCK(X->h_count.alloc(4));
  XCK(cudaMemsetAsync(X->d_count, 0, 16, s));
  k_x_fill64<<<148 * 8, 256, 0, s>>>(X->MB, P, XMB_NONE);
  XCK(cudaMemsetAsync(X->tkey, 0, P * 8, s));
  XCK(cudaMemsetAsync(X->LS, 0, P * 8, s));
  X->tclock = 1; X->key_base = 0; X->key_epoch = 1; X->key_hi = 1ull << FB_KEY_BITS; X->gen_id = 0; X->wclock = 0; X->sclock = 0;
  return cudaGetLastError();
}
// Second half of UpdateOccupancy (ESDFMap.cpp:263-267): k_integrate<true> (fb_map.cu) staged the voxels that crossed the
// occupancy threshold with the serial time of their first observation; sorted by that time they are appended to
// insert_queue_ / delete_queue_ in the order the reference's walk over occupancy_queue_ pushes them.
cudaError_t fb_exact_queue_crossings(FbExact *X, const unsigned long long *ins_key, const uint32_t *ins_vox, const unsigned long long *del_key,
                                     const uint32_t *del_vox, FbDev<uint32_t> &ins, unsigned *n_ins, FbDev<uint32_t> &del, unsigned *n_del,
                                     cudaStream_t s, int *launches) {
  cudaError_t e;
  XCK(cudaMemcpyAsync(X->h_count, X->d_count, 8, cudaMemcpyDeviceToHost, s));
  XCK(cudaStreamSynchronize(s));
  const unsigned ni = X->h_count[0], nd = X->h_count[1];
  XCK(ins.reserve((size_t)*n_ins + ni, s, true));             // the queues keep the pushes of an earlier UpdateOccupancy
  XCK(del.reserve((size_t)*n_del + nd, s, true));
  XCK(X->k1b.reserve(ni > nd ? ni : nd, s, false));
  if (ni) { if ((e = x_sort_pairs(X, ins_key, X->k1b, ins_vox, ins + *n_ins, ni, s, FB_KEY_BITS))) return e; *n_ins += ni; *launches += 1; }
  if (nd) { if ((e = x_sort_pairs(X, del_key, X->k1b, del_vox, del + *n_del, nd, s, FB_KEY_BITS))) return e; *n_del += nd; *launches += 1; }
  return cudaSuccess;
}
// A new integration epoch: later observations beat everything recorded so far in tkey (fb_touch), so nothing is reset.
cudaError_t fb_exact_next_epoch(FbExact *X, const FbGeom &g, cudaStream_t s) {
  X->key_base = 0;
  if (++X->key_epoch >= (1u << (64 - FB_KEY_BITS))) {          // epoch field exhausted (2^20 integrations): start over on a zeroed array
    XCK(cudaMemsetAsync(X->tkey, 0, (size_t)g.ptotal * 8, s));
    X->key_epoch = 1;
  }
  X->key_hi = (unsigned long long)X->key_epoch << FB_KEY_BITS;
  return cudaSuccess;
}

cudaError_t fb_exact_update_esdf(FbExact *X, const FbGeom &g, uint32_t *cobs, uint32_t *scratch, const double *occ, const uint32_t *occbits, double l_occ,
                                 const uint32_t *ins, unsigned n_ins, const uint32_t *del, unsigned n_del, cudaStream_t s, FbExactStats *st, int *launches) {
  cudaError_t e;
  const size_t P = (size_t)g.ptotal;
  memset(st, 0, sizeof(*st));
  XCK(X->flags.reserve((size_t)(n_ins > n_del ? n_ins : n_del) + 16, s, false));
  static const bool xdbg = getenv("FIESTA_DEBUG_X") != nullptr;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
  const auto t_begin = now();
  // ---- E1: insert seeds in insert_queue_ order (:278-291)
  unsigned nE = 0, ndep_run = 0;
  unsigned long long ls_deps = 0;
  bool scratch_ok = X->scratch_clean;
  if (n_ins) {
    k_x_flag_exist<<<nblk(n_ins), 256, 0, s>>>(ins, n_ins, occ, l_occ, X->flags, 1);
    if ((e = x_select(X, ins, X->flags, X->E[0], n_ins, &nE, s))) return e;
    if (nE) k_x_apply_seed<<<nblk(nE), 256, 0, s>>>(g, X->E[0], nE, cobs, X->LS, X->tclock);
    X->tclock += nE;
    *launches += 2;
  }
  // ---- E2: deletes (:292-337)
  if (n_del) {
    XCK(X->sel.reserve((size_t)n_del + 16, s, false));
    // `scratch` (one word per voxel) is all-XNONE between uses: every sparse use below undoes its own writes instead of
    // refilling 4 bytes per voxel of the grid three times per call
    if (!X->scratch_clean) { k_x_fill32<<<148 * 8, 256, 0, s>>>(scratch, P, XNONE); *launches += 1; }
    scratch_ok = true;
    X->scratch_clean = false;                                  // until the undo kernels below are queued (an error return leaves it false)
    k_x_del_minpos<<<nblk(n_del), 256, 0, s>>>(del, n_del, occ, l_occ, scratch);
    k_x_del_flag<<<nblk(n_del), 256, 0, s>>>(del, n_del, occ, l_occ, scratch, X->flags);
    unsigned nd = 0;
    if ((e = x_select(X, del, X->flags, X->sel, n_del, &nd, s))) return e;
    k_x_unset<<<nblk(n_del), 256, 0, s>>>(del, n_del, scratch);
    *launches += 3;
    if (nd) {
      k_x_del_rank<<<nblk(nd), 256, 0, s>>>(X->sel, nd, scratch);
      // order of the reference's list walk = (obstacle's position in delete_queue_, link time descending).  Both fit one
      // 64-bit key as long as (bits of the rank) + (bits of the relink clock) <= 64 -- one radix sort; else two stable sorts
      int rank_bits = 1; while ((1ull << rank_bits) < (unsigned long long)nd) ++rank_bits;
      int clock_bits = 1; while (clock_bits < 64 && (X->tclock >> clock_bits)) ++clock_bits;
      const bool two_sorts = getenv("FIESTA_X_TWO_SORTS") != nullptr;              // tests: force the fallback
      const int shift = (rank_bits + clock_bits <= 64 && !two_sorts) ? 64 - rank_bits : 0;
      // dependants: the list is sized by a first counting attempt, then (rarely) re-run with more room
      unsigned ndep = 0;
      for (int attempt = 0; attempt < 2; ++attempt) {
        const size_t cap = std::min({X->dv.size(), X->k1.size(), X->k2.size()});
        XCK(cudaMemsetAsync(X->d_count, 0, 4, s));
        k_x_scan_deps<<<148 * 16, 256, 0, s>>>(g, cobs, occbits, scratch, X->LS, X->k1, X->k2, X->dv, X->d_count, (unsigned)cap, shift);
        XCK(cudaMemcpyAsync(X->h_count, X->d_count, 4, cudaMemcpyDeviceToHost, s));
        XCK(cudaStreamSynchronize(s));
        ndep = *X->h_count;
        *launches += 1;
        if (ndep <= cap) break;
        XCK(X->dv.reserve(ndep, s, false)); XCK(X->k1.reserve(ndep, s, false)); XCK(X->k2.reserve(ndep, s, false));
      }
      st->dependants = ndep;
      k_x_unset<<<nblk(nd), 256, 0, s>>>(X->sel, nd, scratch);
      if (ndep) {
        for (FbDev<unsigned long long> *b : {&X->k1b, &X->k2b}) XCK(b->reserve(ndep, s, false));
        for (FbDev<uint32_t> *b : {&X->idx[0], &X->idx[1], &X->deps, &X->nc[0], &X->nc[1]}) XCK(b->reserve(ndep, s, false));
        XCK(X->flags.reserve(ndep, s, false));
        if (shift) {
          if ((e = x_sort_pairs(X, X->k1, X->k1b, X->dv, X->deps, ndep, s))) return e;
          *launches += 1;
        } else {
          k_x_iota<<<nblk(ndep), 256, 0, s>>>(X->idx[0], ndep);
          if ((e = x_sort_pairs(X, X->k2, X->k2b, X->idx[0], X->idx[1], ndep, s))) return e;
          k_x_gather64<<<nblk(ndep), 256, 0, s>>>(X->k1, X->idx[1], ndep, X->k1b);
          if ((e = x_sort_pairs(X, X->k1b, X->k2b, X->idx[1], X->idx[0], ndep, s))) return e;
          k_x_gather32<<<nblk(ndep), 256, 0, s>>>(X->dv, X->idx[0], ndep, X->deps);
          *launches += 5;
        }
        XCK(X->flags2.reserve(ndep, s, false));
        k_x_set_ord<<<nblk(ndep), 256, 0, s>>>(X->deps, ndep, scratch, X->nc[0], X->flags2);
        *launches += 1;
        ndep_run = ndep; ls_deps = X->tclock;                // the fixpoint and the hand-over to E[0] run inside k_x_relax
        X->tclock += ndep;
      }
    }
  }
  // ---- E3: relax (:338-392): one persistent kernel runs every generation
  st->generations = 0;
  if (xdbg) { cudaStreamSynchronize(s); fprintf(stderr, "[x] seeds+deletes %.2f ms (reseed rounds %u, dependants %u)\n", ms(t_begin, now()), st->reseed_rounds, st->dependants); }
  if (nE || ndep_run) {
    if (xdbg && !X->d_dbg) XCK(X->d_dbg.alloc(FB_X_DBG_WORDS));
    if (xdbg) XCK(cudaMemsetAsync(X->d_dbg, 0, FB_X_DBG_WORDS * 8, s));
    if (X->sclock > 0xf0000000u) { XCK(cudaMemsetAsync(X->SUMg, 0, P * 4, s)); X->sclock = 0; }       // stamp wrap-around
    if (X->gen_id > 0xf0000000u) X->gen_id = 0;
    if (X->wclock > 0xf0000000u) { XCK(cudaMemsetAsync(X->wstamp, 0, P * 4, s)); X->wclock = 0; }
    FbXCtl *h = X->h_ctl;
    memset(h, 0, sizeof(*h));
    h->gen_id = X->gen_id; h->wclock = X->wclock; h->tclock = X->tclock; h->sclock = X->sclock;
    XCK(cudaMemcpyAsync(X->d_ctl, h, sizeof(FbXCtl), cudaMemcpyHostToDevice, s));
    XCK(fb_xrelax_launch(X, g, cobs, nE, X->deps, ndep_run, scratch, X->nc[0], X->flags2, occbits, ls_deps, xdbg ? X->d_dbg.get() : nullptr, s));
    if (ndep_run) k_x_unset<<<nblk(ndep_run), 256, 0, s>>>(X->deps, ndep_run, scratch);
    XCK(cudaMemcpyAsync(h, X->d_ctl, sizeof(FbXCtl), cudaMemcpyDeviceToHost, s));
    XCK(cudaStreamSynchronize(s));
    *launches += 1;
    if (h->err) { snprintf(X->err, sizeof(X->err), h->err == 1u ? "exact mode: generation with more than 2^27 entries" : "exact mode: behaviour fixpoint did not converge"); return cudaErrorInvalidValue; }
    X->gen_id = h->gen_id; X->wclock = h->wclock; X->tclock = h->tclock; X->sclock = h->sclock;
    st->generations = h->generations; st->reseed_rounds = h->reseed_rounds; st->eval_rounds = h->rounds; st->dense_rounds = h->dense_rounds;
    st->voxels_changed = h->voxels_changed; st->expansions = h->expansions;
    if (xdbg) {
      static unsigned long long hd[FB_X_DBG_WORDS];
      XCK(cudaMemcpy(hd, X->d_dbg, sizeof(hd), cudaMemcpyDeviceToHost));
      static const char *cat[14] = {"S", "round1", "rounds", "dense", "commit", "apply", "s.round1", "s.rounds", "s.commit", "s.apply", "top", "empty-barrier", "reseed.rounds", "reseed.assemble"};
      fprintf(stderr, "[x] reseed rounds %u; phases (us, count):", st->reseed_rounds);
      for (int c = 0; c < 14; ++c) fprintf(stderr, " %s %.0f/%llu", cat[c], hd[3 * 1024 + 2 * c] / 1965.0, hd[3 * 1024 + 2 * c + 1]);
      fprintf(stderr, "\n");
      { double wm = 0; for (int q = 0; q < 4096; ++q) wm += hd[3 * 1024 + 32 + 1024 + q] / 1965.0; fprintf(stderr, "[x] sum over rounds of the longest per-CTA work time: %.0f us (the rest of round1+rounds+dense+s.round1+s.rounds is barrier + skew)\n", wm); }
      for (int gq = 0; gq < 2; ++gq) { fprintf(stderr, "[x] gen %d work lists:", gq); for (int r = 0; r < 512 && hd[3 * 1024 + 32 + gq * 512 + r]; ++r) fprintf(stderr, " %llu", hd[3 * 1024 + 32 + gq * 512 + r]); fprintf(stderr, "\n"); }
      fprintf(stderr, "[x] gens %u rounds %u dense %u deps %u nE0 %u |", st->generations, st->eval_rounds, st->dense_rounds, st->dependants, nE);
      for (unsigned q = 0; q < st->generations && q < 1024; ++q) fprintf(stderr, " %llu/%llu/%.1fus", hd[3 * q], hd[3 * q + 1], hd[3 * q + 2] / 1965.0);
      fprintf(stderr, "\n");
    }
  }
  X->scratch_clean = scratch_ok;                             // every sparse write above has its undo queued behind it
  return cudaSuccess;
}
