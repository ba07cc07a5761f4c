// nb_bank.cuh - device layout of a particle bank and the argument block of one timestep.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "nb_math.cuh"

namespace nb {

// Packed-pair SoA: every per-particle access is one 16-byte vector load/store that is
// coalesced across the warp (32 lanes x 16 B = 512 contiguous bytes per field pair).
// The fields are those of the reference's Particle (neutral_data.h:48-79):
//   pos  = (x, y)                      dir = (omega_x, omega_y)
//   ew   = (energy, weight)            tm  = (dt_to_census, mfp_to_collision)
//   meta = (cellx, celly, dead, origin)
// `origin` is the particle's index in injection order (global pid = pid0 + origin): the RNG
// key must follow a particle through any reordering of the bank (omp3/neutral.c:89,632-641).
struct BankView {
  double2* pos;
  double2* dir;
  double2* ew;
  double2* tm;
  int4* meta;
};

constexpr size_t kBankBytesPerParticle = 4 * sizeof(double2) + sizeof(int4);  // 80

// Plain 11-array SoA, the reference's -DSoA Particle (neutral_data.h:48-61). Used for
// import/export at the plugin boundary only.
struct SoaView {
  double* x;
  double* y;
  double* omega_x;
  double* omega_y;
  double* energy;
  double* weight;
  double* dt_to_census;
  double* mfp_to_collision;
  int* cellx;
  int* celly;
  int* dead;
};

// Step totals, one 64-bit counter each (device memory, zeroed by the host per step).
// kTotFault is raised by the staging kernels when what they find on the device contradicts
// what the host assumed (see stage.cu); the host turns it into a fatal error.
// kTotGridsDiffer counts the grid points at which the two cross-section tables' energy grids
// differ (stage.cu): whether "one search serves both tables" holds is decided where the data
// is, every timestep, never from a host-side cache of what some pointer once held.
// kTotGroupFault: a bounded wait of the tally collective expired (nb_group.cuh).
enum { kTotFacets = 0, kTotCollisions, kTotProcessed, kTotCensus, kTotDeaths,
       kTotGroupFault = 5, kTotGridsDiffer = 6, kTotFault = 7, kTotCount = 8 };

// Staged copy of one reference CrossSection (neutral_data.h:38-43), rebuilt from the caller's
// device arrays at the start of every timestep (stage.cu):
//   kv[i]      = {keys[i], values[i]}  - one 16-byte load fetches a grid point
//   bucket[b]  = number of keys whose bucket id is < b, with
//                bucket id(E) = clamp((bits(E) - bits0) >> shift, 0, nb - 1)
// The bracketing interval of an energy in bucket b lies in [bucket[b] - 1, bucket[b + 1]],
// so the lookup bisects a handful of entries instead of the whole grid. The map is
// monotone for ANY bits0/shift, so the index is exact whatever the keys are; bits0/shift
// only decide how evenly the keys spread over the buckets.
struct CsStage {
  const double2* kv;
  const int* bucket;
  unsigned long long bits0;
  int shift;
  int nb;
  int n;
};

// Density tile maps, rebuilt every timestep (stage.cu). fine[t] holds the density of the
// 16x16-cell tile t when all its cells carry the same bit pattern, else the kMixedTileBits
// marker; coarse[] is the same over 256x256-cell tiles (uniform iff its fine tiles are
// uniform and equal). A facet crossing inside a uniform coarse tile needs no memory access at
// all; the 2 KB coarse map stays L1-resident, the fine map L2-resident, and only mixed fine
// tiles read the density mesh itself.
constexpr int kTileShift = 4;
#ifndef NB_COARSE_SHIFT
#define NB_COARSE_SHIFT 8
#endif
constexpr int kCoarseShift = NB_COARSE_SHIFT;
constexpr unsigned long long kMixedTileBits = 0x7ff8b200dead0001ull;  // a NaN payload of ours
struct TileMap {
  const double* fine;
  const double* coarse;
  int fine_tx;    // fine tiles per mesh row
  int coarse_tx;  // coarse tiles per mesh row
};

struct StepArgs {
  int nx, ny;  // mesh cells (pad = 0, offsets = 0: the only configuration main.c produces)
  int n;       // bank slots to visit
  uint64_t master_key;
  uint64_t pid0;  // global pid of origin 0 (particle sharding across GPUs)
  double dt;
  double inv_ntotal;
  const double* density;
  const double* edgex;
  const double* edgey;
  const double* s_keys;
  const double* s_vals;
  const double* a_keys;
  const double* a_vals;
  int s_n, a_n;
  // Both tables have the same number of grid points: they MAY share one energy grid (then one
  // search serves both). Whether they do is totals[kTotGridsDiffer] == 0 - see same_grid().
  int same_keys;
  double* tally;
  // Per-particle cumulative event counters indexed by origin (the interface's three
  // uint64[nparticles] scratch arrays, neutral_interface.h:19); may be null.
  unsigned long long* p_facets;
  unsigned long long* p_collisions;
  unsigned long long* p_census;
  unsigned long long* totals;
  BankView bank;
  const LogTable* logt;
  // staged per-step copies (stage.cu); kernels that do not use them ignore the fields
  CsStage cs_s, cs_a;
  TileMap tiles;
  // Target edges of a facet crossing, restaged per step as four rows of `edge_stride` doubles:
  // row 0 = edgex, row 1 = edgey (the far edge of a cell for a direction component >= 0), rows
  // 2, 3 = the same minus OPEN_BOUND_CORRECTION (the near edge pulled in, omp3/neutral.c:443,
  // 449 - the subtraction is done once per edge instead of once per facet, same operands,
  // same bits). One base pointer and an integer row select replace two pointer selects and
  // the per-facet correction.
  const double* edges4;
  int edge_stride;
  // Staggered dispatch of the collision class (history.cu: dispatch_group): percent of the
  // streamer CTAs that go out in front of the delayed colliders (0: class order), percent of
  // the collider CTAs that are delayed, and the colliders' share of the live bank (per mille)
  // from which on it is done.
  int stagger_at, stagger_share, stagger_min;
};

// Option tally_batches (tally_batches.cu): with nbatches = B > 0 every deposit of the history
// kernel goes to the partial tally of the depositing particle's batch instead of
// StepArgs::tally; batch b is the contiguous pid range shard_split(n, b, B). A kernel
// parameter of its own behind the existing two: grown, StepArgs would move the offset of the
// parameter that follows it in every instantiation of k_history, batched or not.
struct BatchArgs {
  double* slab;
  int nbatches;
  int n;
};

// nb200_bank_set_group_flux_tally: with ngroups = G > 0 the flux deposits go to
// flux[g * ncells + cell], g the energy group with edges[g] <= e < edges[g + 1] (G + 1 edges in
// device memory); none outside [edges[0], edges[G]). A kernel parameter of its own behind the
// flux array, for the reason BatchArgs is one.
struct GroupArgs {
  const double* edges;
  int ngroups;
};

// Layout of the B partial tallies in the batch slab: batch-major [b][cell] (0) or cell-major
// [cell][b] (1). Both were built and measured (DESIGN.md 9); the product keeps batch-major.
// -DNB_TALLY_BATCH_CELL_MAJOR=1 builds the other one for tools/tally_batches_cost.py.
#ifndef NB_TALLY_BATCH_CELL_MAJOR
#define NB_TALLY_BATCH_CELL_MAJOR 0
#endif
__host__ __device__ __forceinline__ size_t batch_slot(int b, size_t cell, int B, size_t ncells) {
  return NB_TALLY_BATCH_CELL_MAJOR ? cell * (size_t)B + (size_t)b : (size_t)b * ncells + cell;
}

// Batch of global pid `pid` among the B contiguous ranges of shard_split(n, b, B) (capi.cu):
// batch b starts at b * (n / B) + min(b, n % B). The first n % B batches hold n / B + 1
// particles, the rest n / B. Requires 1 <= B <= n and pid < n.
__host__ __device__ __forceinline__ unsigned batch_of(unsigned pid, unsigned n, unsigned B) {
  const unsigned per = n / B, rem = n % B;
  const unsigned split = rem * (per + 1u);  // particles in the larger batches
  return pid < split ? pid / (per + 1u) : rem + (pid - split) / per;
}

// Scratch of the per-step counting sort (pipeline.cu).
struct SortArgs {
  unsigned* keys;        // [n] sort key of every slot in [0, n_upper)
  unsigned* bin_count;   // [nbins] histogram
  unsigned* bin_cursor;  // [nbins] running destination of every bin
  unsigned* chunk_sum;   // [ceil(nbins / 2048)] scratch of the histogram scan
  unsigned* n_live;      // device scalars: [0] slots in front of the dead bin after the sort,
                         // [1] slots of the collision class (the front of the sorted bank)
  int nbins;             // 3 classes x nq length bins x ntiles + 1 dead bin
  int nq;                // bins of expected history length (1: none)
  float q_scale;         // length bins per octave
  float inv_dx, inv_dy;  // cells per unit length (mean over the mesh)
  int ntiles;
  int tiles_x;
  int tile_shift;        // cells per tile edge = 1 << tile_shift; < 0: one tile
  int n_upper;           // host-known upper bound of the live prefix
  int n;                 // bank size
};

}  // namespace nb
