// fiesta_b200 -- host interface of the order-exact mode (fb_exact.cu: ordered UpdateOccupancy, insert / delete seeding;
// fb_xrelax.cu: the persistent relaxation kernel).
#pragma once
#include "fb_common.cuh"

#define FB_X_MAX_BLOCKS 256
#define FB_X_SMALL_DEFAULT 32768u   // (from a sweep on the 512^3 LIDAR frames; FIESTA_X_SMALL / FIESTA_X_DENSE override)
#define FB_X_DBG_WORDS (3 * 1024 + 32 + 2 * 512 + 4096)

struct FbExactStats {
  unsigned long long expansions;      // == the reference's "Expanding N nodes" (ESDFMap.cpp:347,394)
  unsigned long long voxels_changed;  // accepted final writes over all generations
  unsigned generations, eval_rounds, dense_rounds, reseed_rounds, dependants;
};

// Control block of k_x_relax (device memory; the host writes it before and reads it after every launch).
struct FbXCtl {
  unsigned bar, err;                  // grid barrier arrivals; 1 = a generation exceeded 2^27 entries
  unsigned sclock, pad1;              // stamp of the last summary pass (SUMg dedupe; persists across launches)
  unsigned nW[3], nF[3];              // work / flip list lengths, rotating per round
  unsigned gen_id, wclock;            // stamps for SUMg / wstamp dedupe (persist across launches)
  unsigned generations, rounds, dense_rounds, reseed_rounds;
  unsigned long long tclock, expansions, voxels_changed;
  unsigned partial[FB_X_MAX_BLOCKS];  // winners per CTA range (ordered hand-over)
};

struct FbExact {
  FbDev<unsigned long long> MB;   // per voxel: {parity | queue position | behaviour | code} of its live entry in the current generation
  FbDev<unsigned long long> LS;   // per voxel: time of the last relink into a dependant list
  FbDev<unsigned long long> tkey; // per voxel: epoch-coded serial time of the first pending observation (fb_touch, fb_common.cuh)
  FbDev<uint32_t> touched;     // [ptotal] staging of the voxels whose occupancy crossed the threshold (inserts; deletes use emask)
  unsigned long long tclock;   // relink clock
  unsigned long long key_base; // observation clock within the current integration epoch
  unsigned long long key_hi;   // key_epoch << FB_KEY_BITS
  unsigned key_epoch;          // integration epoch (one per UpdateOccupancy)
  FbDev<unsigned> d_count; FbPinned<unsigned> h_count;
  bool scratch_clean;           // the per-voxel scratch word array of UpdateESDF is all-XNONE
  FbDev<uint4> SUM;            // per voxel offer summary of the current generation: {first ts, best ts, best code, snapshot code}
  FbDev<uint32_t> SUMg;        // per voxel: summary pass for which SUM was computed (each target is claimed once per pass)
  unsigned gen_id, wclock, sclock;
  FbDev<uint32_t> emask;       // per entry: slots it owns in the next generation
  FbDev<uint32_t> W[3], F[3];  // work lists / flip lists, rotating per round
  FbDev<uint32_t> wstamp;      // per entry: round for which it is already in a work list
  FbDev<uint32_t> slotc;       // SMALL generations: codes of the owned slots
  unsigned dense_min;          // work lists longer than this are evaluated through refreshed summaries (one wave of warps)
  unsigned small_max;          // generations up to this many entries run without summaries
  FbDev<FbXCtl> d_ctl; FbPinned<FbXCtl> h_ctl;
  FbDev<unsigned long long> d_dbg;
  int relax_blocks;
  FbDev<uint32_t> E[2], sel;
  FbDev<unsigned long long> k1, k2, k1b, k2b;
  FbDev<uint32_t> dv, idx[2], deps, nc[2];
  FbDev<uint8_t> flags, flags2;
  FbDev<uint8_t> cub_tmp;
  char err[256];
};

cudaError_t fb_exact_init(FbExact *X, const FbGeom &g, int device, cudaStream_t s);
cudaError_t fb_exact_queue_crossings(FbExact *X, const unsigned long long *ins_key, const uint32_t *ins_vox, const unsigned long long *del_key,
                                     const uint32_t *del_vox, FbDev<uint32_t> &ins, unsigned *n_ins, FbDev<uint32_t> &del, unsigned *n_del,
                                     cudaStream_t s, int *launches);
cudaError_t fb_exact_next_epoch(FbExact *X, const FbGeom &g, cudaStream_t s);
cudaError_t fb_exact_update_esdf(FbExact *X, const FbGeom &g, uint32_t *cobs, uint32_t *scratch, const double *occ, const uint32_t *occbits, double l_occ,
                                 const uint32_t *ins, unsigned n_ins, const uint32_t *del, unsigned n_del, cudaStream_t s, FbExactStats *st, int *launches);
// fb_xrelax.cu
cudaError_t fb_xrelax_init();
int fb_xrelax_blocks(int device);
cudaError_t fb_xrelax_launch(FbExact *X, const FbGeom &g, uint32_t *cobs, unsigned nE0, const uint32_t *deps, unsigned ndep, uint32_t *ord, uint32_t *nc, uint8_t *nk,
                             const uint32_t *occbits, unsigned long long ls_deps, unsigned long long *dbg, cudaStream_t s);
