// engine.cuh - host-side state of libneutral_b200.so: per-device contexts, particle banks and
// their shards, the asynchronous timestep pipeline and the tally group of a particle-sharded
// run. Nothing here is exported; capi.cu is the C ABI on top of it.
//
// Ownership (SURVEY.md 8b): the kernel set owns the particle bank it hands out through
// inject_particles (omp3/neutral.c:570,629) and every piece of state the reference's single
// shared-memory kernel set does not need - per-GPU replicas of the read-only inputs, delta
// tallies, streams, the collective - lives here, created lazily, invisible to main.c.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <deque>
#include <string>
#include <utility>
#include <vector>

#include "../../include/neutral_b200.h"
#include "nb_group.cuh"
#include "nb_nccl_dyn.cuh"
#include "transport.cuh"

namespace nb {

constexpr uint64_t kBankMagic = 0x6e62323030424e4bull;  // "nb200BNK"
constexpr int kRing = 8;        // step-totals slots per device (steps in flight + being read)
constexpr int kMaxPending = 4;  // timesteps a bank may have enqueued and not yet collected
constexpr int kCsBuckets = 8192;
constexpr int kMaxDevices = 64;

// ------------------------------------------------------------------------------ options --
// Process-wide defaults (nb200_set_option) that a bank may override for itself
// (nb200_bank_set_option): two banks can run different kernel configurations side by side.
struct Options {
  int print = 1;
  int pipeline = 1;
  int fast_div = 1;
  int tile_shift = 8;
  int length_bins = 512;
  int tally_prereduce = 0;
  int l2_persist = 0;
  int defer_finish = 0;
  int device_inject = 1;
  int stage_overlap = 1;
  int history_smem_pad = 0;
  int ngpus = 0;         // GPUs the next inject_particles / nb200_bank_create shards over (0/1: one)
  int collective = 1;    // 1: the library's peer-memory reduce-scatter kernel; 0: NCCL
  int reduce_ctas = 592; // grid of the peer-memory reduce kernel
  int tally_reduce_every = 0;  // timesteps between reduce-scatters of a sharded tally; 0: on demand
  int host_mirror = 0;   // keep a host copy of the bank behind the handle's 11 pointers
  int headroom_pct = 0;  // extra bank capacity for produced particles (omp3/neutral.c:570: 100)
  int stagger_at = 0;      // percent of the streamer CTAs dispatched in front of the delayed colliders
  int stagger_share = 50;  // percent of the collider CTAs that are delayed
  int stagger_min = 35;    // colliders' share of the live bank (per mille) from which on it is done
  int step_graph = 1;    // submit a timestep as one CUDA graph launch instead of ~23 driver calls
  int tally_batches = 0; // batches of the next bank's tally statistics (0: none, else 2..64)
};
constexpr int kMaxTallyBatches = 64;

struct OptionSpec {
  const char* name;
  int Options::*slot;
  int lo, hi;
};
extern const OptionSpec kOptionSpecs[];
extern const int kNumOptionSpecs;

// ------------------------------------------------------------------------ device context --
struct CsParams {  // parameters of the bucket index of one table (CsStage in nb_bank.cuh)
  unsigned long long bits0 = 0;
  int shift = 63;
  int nb = 1;  // one bucket = plain bisection over the whole grid (always valid)
};

struct DeviceCtx {
  int device = -1;
  cudaStream_t stream = 0;  // every kernel of this device's banks (nb200_set_stream)
  cudaStream_t stage_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_tiles = nullptr;
  // option step_graph: a timestep's kernels are recorded on `capture` (never executed there),
  // the executable graph is updated in place with the step's parameters and launched on
  // `stream`. `work` is where the step's calls go: `stream`, or `capture` while recording.
  cudaStream_t capture = nullptr;
  cudaStream_t work = 0;
  cudaGraphExec_t step_exec = nullptr;
  uint64_t graph_updates = 0, graph_instantiations = 0;
  LogTable* d_logt = nullptr;
  SinCosTable* d_sct = nullptr;
  unsigned long long* d_totals = nullptr;
  // ring of step-total slots in mapped pinned memory: the device publishes a step's counts
  // itself (no copy engine involved), the host reads them when it collects the step
  unsigned long long* h_totals = nullptr;
  unsigned long long* h_totals_dev = nullptr;
  bool slot_busy[kRing] = {false};
  int next_slot = 0;
  cudaEvent_t ev_begin[kRing] = {nullptr}, ev_mid[kRing] = {nullptr}, ev_end[kRing] = {nullptr};
  cudaEvent_t ev_pub[kRing] = {nullptr};  // behind the kernel that publishes the slot
  int pending_steps = 0;
  // sort scratch
  unsigned* d_bins = nullptr;
  unsigned* d_n_live = nullptr;
  long long bins_capacity = 0;
  // per-step staging (stage.cu)
  char* d_cs_stage = nullptr;
  size_t cs_stage_bytes = 0;
  double* d_tile_rho = nullptr;
  int tile_capacity = 0;
  double* d_edges4 = nullptr;
  int edges_capacity = 0;
  // scheduling hints read back once per pointer (never a correctness input: a stale hint
  // spreads keys less evenly over buckets or bins, nothing else)
  struct MeshExtent { const double* ex; const double* ey; int nx, ny; double width, height; };
  std::vector<MeshExtent> mesh_cache;
  struct TableHint { const double* keys; int n; CsParams par; };
  std::vector<TableHint> table_cache;
  bool l2_limit_set = false;
  size_t l2_setaside = 0;
  uint64_t launches = 0;
};

// Replica of one of the caller's read-only inputs (which live on the bank's primary GPU) on
// another GPU of a single-process multi-GPU bank. Owned by the bank's shard: a new bank copies
// afresh, so an address the caller's allocator hands out twice cannot serve stale contents.
struct Replica {
  const void* src;
  size_t bytes;
  void* copy;
  uint64_t generation;
};

// ------------------------------------------------------------------------------- banks ----
struct Shard {
  int dev = 0;
  BankView cur{};
  BankView alt{};  // double buffer of the per-step sort (allocated on first use)
  bool has_alt = false;
  unsigned* keys = nullptr;
  int n = 0;          // particles
  int capacity = 0;   // slots allocated (>= n: head-room for produced particles)
  int n_upper = 0;    // slots [n_upper, n) are known to hold dead particles
  int first = 0;      // index of the shard's first particle in the bank's injection order
  uint64_t pid0 = 0;  // global particle index of origin 0 (the RNG key base)
  SoaView exported{};  // lazily allocated plain SoA view (11 device arrays)
  bool has_export = false;
  std::vector<Replica> replicas;  // secondary GPUs only
};

struct StepRequest {  // what solve_transport_2d was asked; pointers on the bank's primary GPU
  int nx = 0, ny = 0;
  uint64_t master_key = 0;
  double dt = 0.0;
  int ntotal = 0;
  const double *density = nullptr, *edgex = nullptr, *edgey = nullptr;
  const double *s_keys = nullptr, *s_vals = nullptr, *a_keys = nullptr, *a_vals = nullptr;
  int s_n = 0, a_n = 0;
  double* tally = nullptr;
  uint64_t *r0 = nullptr, *r1 = nullptr, *r2 = nullptr;
};

struct PendingStep {
  int slot[kMaxRanks];
  uint64_t launches0 = 0;
  uint64_t master_key = 0;
  bool pipeline = true;
  bool print = true;
};

struct GroupMember {
  int dev = -1;           // local CUDA ordinal; -1: the member lives in another process
  char* slab = nullptr;   // base of the member's slab as THIS process addresses it
  bool ipc_opened = false;
  SyncBlock* sync = nullptr;
  double* delta[kDeltaBuffers] = {nullptr};
  double* owned = nullptr;
  double* tmp = nullptr;       // NCCL flavour: reduce-scatter result (chunk)
  double* gathered = nullptr;  // NCCL flavour: all-gather result (nranks * chunk)
  // local members only
  cudaStream_t side = nullptr;
  cudaEvent_t ev_hist[kDeltaBuffers] = {nullptr};
  cudaEvent_t ev_zeroed[kDeltaBuffers] = {nullptr};
  bool zeroed_recorded[kDeltaBuffers] = {false};
  cudaEvent_t ev_side = nullptr;
  nccl_comm_t comm = nullptr;
};

// The ranks that share one tally (nb_group.cuh). Single-process: every member is local (one
// GPU each). Multi-process: exactly one member is local, the others are CUDA-IPC mappings.
struct TallyGroup {
  int nranks = 0;
  size_t ncells = 0, chunk = 0, padded = 0, slab_bytes = 0;
  int collective = 1;
  bool mp = false;
  int mp_rank = -1;
  int reduce_ctas = 592;
  int reduce_every = 0;      // timesteps deposited into one buffer before it is reduced (0: on demand)
  int steps_deposited = 0;   // timesteps in the current deposit buffer, not reduced yet
  int cur_k = 0;             // the deposit buffer in use
  GroupMember m[kMaxRanks];
  unsigned long long epoch = 0, flush_epoch = 0;  // reductions / flushes so far
  double* target = nullptr;  // the caller-visible tally the owned slices belong to
  int target_dev = -1;
  bool dirty = false;        // owned slices hold contributions the target has not received
};

struct HostMirror {  // pinned host copy of the bank in injection order (visit_dump decks)
  nb200_particle_soa a{};
  bool present = false;
};

// Option tally_batches of a single-GPU bank (tally_batches.cu): the history kernel deposits into
// B partial tallies; the caller's tally is brought up to date lazily, where a sharded run's
// would be (flush_groups_touching), by adding what the batches gained since the last flush.
struct TallyBatches {
  int B = 0;                 // 0: the bank deposits straight into the caller's tally
  double* slab = nullptr;    // B partial tallies (batch_slot layout), then F = their sum at the last flush
  size_t ncells = 0;
  double* target = nullptr;  // the caller-visible tally the batches belong to
  bool dirty = false;        // the batches hold deposits the target has not received
  bool deposited = false;    // a timestep has deposited into this slab
};

struct Bank {
  std::vector<Shard> shards;
  TallyBatches batches;
  // nb200_bank_set_flux_tally: the caller's track-length flux array (device memory on the
  // bank's GPU, flux_ncells doubles) every timestep also deposits into; null: none.
  double* flux = nullptr;
  size_t flux_ncells = 0;
  // nb200_bank_set_batched_flux_tally: B > 0 (the B of `batches`) when the flux deposits go to
  // B partial fluxes instead; their target is `flux`, their slab is allocated when it attaches.
  TallyBatches flux_batches;
  int n = 0;
  uint64_t pid0 = 0;
  int primary_dev = 0;
  std::vector<std::pair<int, int>> overrides;  // (option index, value)
  std::deque<PendingStep> pending;
  TallyGroup* group = nullptr;  // owned: single-process multi-GPU banks
  HostMirror mirror;
  struct BankHeader* header = nullptr;
};

// What inject_particles / nb200_bank_create hand out as `Particle*` points just behind this
// header, at `nviews` copies of the reference's -DSoA struct (neutral_data.h:48-61): one is
// all SoA-aware code needs; the reference's plot_particle_density (main.c:178-181) indexes
// `&local_particles[ii]` even under -DSoA, so a bank with a host mirror carries one copy per
// particle.
struct BankHeader {
  uint64_t magic;
  Bank* impl;
  uint64_t nviews;
  uint64_t reserved;
};

}  // namespace nb
