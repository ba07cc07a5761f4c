// capi.cu - the C ABI of libneutral_b200.so (declared in include/neutral_b200.h).
//
// Host-side glue only: argument checking, device memory, stream ordering, counters, the
// multi-GPU orchestration. The arithmetic of the hot path lives in the kernels (history.cu,
// pipeline.cu, stage.cu, transport.cu, group.cu). There is deliberately no CPU fallback:
// every compute entry point fails loudly when no CUDA device is usable.
#include <cuda_runtime.h>
#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <string>
#include <unordered_set>
#include <vector>

#include "engine.cuh"
#include "nb_sincos.cuh"

namespace nb {

// microbench.cu
int launch_red_rate(double* scratch, size_t cells, int nx, int iters, int pattern,
                    cudaEvent_t e0, cudaEvent_t e1, double* seconds, double* reductions,
                    cudaStream_t st);

const OptionSpec kOptionSpecs[] = {
    {"print", &Options::print, 0, 1},
    {"pipeline", &Options::pipeline, 0, 1},
    {"fast_div", &Options::fast_div, 0, 1},
    {"tile_shift", &Options::tile_shift, -1, 12},
    {"length_bins", &Options::length_bins, 0, 4096},
    {"tally_prereduce", &Options::tally_prereduce, 0, 1},
    {"l2_persist", &Options::l2_persist, 0, 2},
    {"defer_finish", &Options::defer_finish, 0, 1},
    {"device_inject", &Options::device_inject, 0, 1},
    {"stage_overlap", &Options::stage_overlap, 0, 1},
    {"history_smem_pad", &Options::history_smem_pad, 0, 200 * 1024},
    {"ngpus", &Options::ngpus, 0, kMaxRanks},
    {"collective", &Options::collective, 0, 1},
    {"reduce_ctas", &Options::reduce_ctas, 1, 8192},
    {"tally_reduce_every", &Options::tally_reduce_every, 0, 1000000},
    {"host_mirror", &Options::host_mirror, 0, 1},
    {"headroom_pct", &Options::headroom_pct, 0, 1000},
    {"step_graph", &Options::step_graph, 0, 1},
    {"stagger_at", &Options::stagger_at, 0, 95},
    {"stagger_share", &Options::stagger_share, 0, 100},
    {"stagger_min", &Options::stagger_min, 0, 1000},
    {"tally_batches", &Options::tally_batches, 0, kMaxTallyBatches},  // 1 is refused too
};
const int kNumOptionSpecs = (int)(sizeof(kOptionSpecs) / sizeof(kOptionSpecs[0]));

}  // namespace nb

namespace {

using namespace nb;

const SinCosTable kHostSinCosTable = {{
#include "glibc_sincos_table.inc"
}};

const LogTable kHostLogTable = {
#include "glibc_log_table.inc"
};

Options g_opt;                         // process-wide defaults
bool g_env_read = false;
DeviceCtx* g_ctx[kMaxDevices] = {nullptr};
std::string g_last_error;
Bank* g_last_deferred = nullptr;       // the bank nb200_solve_finish() refers to
TallyGroup* g_mp = nullptr;            // multi-process group of this process (one GPU)
std::vector<TallyGroup*> g_groups;     // every live group (tally-access hooks walk it)
uint64_t g_replica_generation = 1;     // bumped by nb200_update_replicas
int g_shard_first = 0, g_shard_count = -1;  // nb200_set_shard
std::unordered_set<const void*> g_handles;  // every live bank handle (what `Particle*` may be)
std::vector<Bank*> g_batched;          // every live bank with tally batches
std::vector<Bank*> g_flux;             // every live bank with a flux array attached

// What `validate` reports besides the reference's printed lines (SURVEY.md 8f 1).
struct StepLog {
  uint64_t master_key, facets, collisions, processed, census, deaths, history_ns, sort_ns;
  int ngpus;
};
std::vector<StepLog> g_step_log;
uint64_t g_last_stats[8] = {0};

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
}

[[noreturn]] void terminate(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  fprintf(stderr, "neutral_b200: fatal: %s\n", buf);
  fflush(stderr);
  exit(EXIT_FAILURE);
}

#define CU_FATAL(call)                                                              \
  do {                                                                              \
    cudaError_t err__ = (call);                                                     \
    if (err__ != cudaSuccess)                                                       \
      terminate("%s failed: %s [%s:%d]", #call, cudaGetErrorString(err__), __FILE__, \
                __LINE__);                                                          \
  } while (0)

#define CU_TRY(call)                                                                \
  do {                                                                              \
    cudaError_t err__ = (call);                                                     \
    if (err__ != cudaSuccess) {                                                     \
      set_error("%s failed: %s [%s:%d]", #call, cudaGetErrorString(err__), __FILE__, \
                __LINE__);                                                          \
      return -2;                                                                    \
    }                                                                               \
  } while (0)

#define NCCL_FATAL(api, call)                                                          \
  do {                                                                                 \
    int rc__ = (call);                                                                 \
    if (rc__ != kNcclSuccess)                                                          \
      terminate("%s failed: %s [%s:%d]", #call, (api)->GetErrorString(rc__), __FILE__, \
                __LINE__);                                                             \
  } while (0)

// Makes `dev` the current device for a scope.
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) {
      CU_FATAL(cudaSetDevice(dev));
      switched = true;
    }
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};

// Kernels are loaded when the CUDA context is created, not at their first launch: the first
// timestep is timed by the reference's driver like any other (main.c:99-116). Has to be in the
// environment before the process initialises CUDA; a host that already did keeps its own mode.
__attribute__((constructor)) void load_kernels_eagerly() { setenv("CUDA_MODULE_LOADING", "EAGER", 0); }

void read_environment() {
  if (g_env_read) return;
  g_env_read = true;
  // NB200_NGPUS: GPUs the drop-in binary shards its bank over (SURVEY.md 5 "config / flags").
  if (const char* s = getenv("NB200_NGPUS")) {
    int count = 0;
    if (strcmp(s, "all") == 0) {
      if (cudaGetDeviceCount(&count) != cudaSuccess) count = 0;
    } else {
      count = atoi(s);
    }
    g_opt.ngpus = std::max(0, std::min(count, kMaxRanks));
  }
  if (const char* s = getenv("NB200_COLLECTIVE")) g_opt.collective = strcmp(s, "nccl") == 0 ? 0 : 1;
  if (const char* s = getenv("NB200_HOST_MIRROR")) g_opt.host_mirror = atoi(s) != 0;
  if (const char* s = getenv("NB200_HEADROOM_PCT")) g_opt.headroom_pct = std::max(0, atoi(s));
  // NB200_TALLY_BATCHES: batches of the drop-in binary's tally statistics (option tally_batches)
  if (const char* s = getenv("NB200_TALLY_BATCHES")) {
    const int b = atoi(s);
    if (b == 0 || (b >= 2 && b <= kMaxTallyBatches))
      g_opt.tally_batches = b;
    else
      fprintf(stderr, "neutral_b200: NB200_TALLY_BATCHES=%s ignored (0 or 2..%d)\n", s,
              kMaxTallyBatches);
  }
}

// The context of CUDA device `dev`, initialised on first use (`dev` must be current).
// Returns nullptr with the error set.
DeviceCtx* ctx_create(int dev) {
  DeviceCtx* c = new DeviceCtx();
  c->device = dev;
#define CTX_TRY(call)                                                                    \
  do {                                                                                   \
    cudaError_t err__ = (call);                                                          \
    if (err__ != cudaSuccess) {                                                          \
      set_error("%s failed: %s [%s:%d]", #call, cudaGetErrorString(err__), __FILE__,     \
                __LINE__);                                                               \
      delete c;                                                                          \
      return nullptr;                                                                    \
    }                                                                                    \
  } while (0)
  CTX_TRY(cudaMalloc(&c->d_logt, sizeof(LogTable)));
  CTX_TRY(cudaMemcpy(c->d_logt, &kHostLogTable, sizeof(LogTable), cudaMemcpyHostToDevice));
  CTX_TRY(cudaMalloc(&c->d_sct, sizeof(SinCosTable)));
  CTX_TRY(cudaMemcpy(c->d_sct, &kHostSinCosTable, sizeof(SinCosTable), cudaMemcpyHostToDevice));
  CTX_TRY(cudaMalloc(&c->d_totals, sizeof(unsigned long long) * kTotCount));
  CTX_TRY(cudaHostAlloc(&c->h_totals, sizeof(unsigned long long) * kTotCount * kRing,
                        cudaHostAllocMapped | cudaHostAllocPortable));
  memset(c->h_totals, 0, sizeof(unsigned long long) * kTotCount * kRing);
  CTX_TRY(cudaHostGetDevicePointer(&c->h_totals_dev, c->h_totals, 0));
  for (int k = 0; k < kRing; ++k) {
    CTX_TRY(cudaEventCreate(&c->ev_begin[k]));
    CTX_TRY(cudaEventCreate(&c->ev_mid[k]));
    CTX_TRY(cudaEventCreate(&c->ev_end[k]));
    CTX_TRY(cudaEventCreateWithFlags(&c->ev_pub[k], cudaEventDisableTiming));
  }
  CTX_TRY(cudaStreamCreateWithFlags(&c->stage_stream, cudaStreamNonBlocking));
  CTX_TRY(cudaStreamCreateWithFlags(&c->capture, cudaStreamNonBlocking));
  CTX_TRY(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  CTX_TRY(cudaEventCreateWithFlags(&c->ev_tiles, cudaEventDisableTiming));
  CTX_TRY(cudaMalloc(&c->d_n_live, 2 * sizeof(unsigned)));
  CTX_TRY(cudaMemset(c->d_n_live, 0, 2 * sizeof(unsigned)));
#undef CTX_TRY
  return c;
}

// Context of the CURRENT device; nullptr (error set) when no device is usable.
DeviceCtx* ctx_current() {
  read_environment();
  int count = 0;
  cudaError_t err = cudaGetDeviceCount(&count);
  if (err != cudaSuccess || count <= 0) {
    set_error("no CUDA device available (%s): the b200 kernel set has no CPU fallback",
              err != cudaSuccess ? cudaGetErrorString(err) : "device count is 0");
    (void)cudaGetLastError();
    return nullptr;
  }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) {
    set_error("cudaGetDevice failed");
    return nullptr;
  }
  if (!g_ctx[dev]) g_ctx[dev] = ctx_create(dev);
  return g_ctx[dev];
}

DeviceCtx& ctx_required() {
  DeviceCtx* c = ctx_current();
  if (!c) terminate("%s", g_last_error.c_str());
  return *c;
}

// Context of device `dev` (made current for the call when it has to be created).
DeviceCtx& ctx_on(int dev) {
  if (dev < 0 || dev >= kMaxDevices) terminate("bad device ordinal %d", dev);
  if (!g_ctx[dev]) {
    DeviceGuard guard(dev);
    g_ctx[dev] = ctx_create(dev);
    if (!g_ctx[dev]) terminate("%s", g_last_error.c_str());
  }
  return *g_ctx[dev];
}

#define CTX_OR_RETURN(c)            \
  DeviceCtx* c##_ptr = ctx_current(); \
  if (!c##_ptr) return -1;           \
  DeviceCtx& c = *c##_ptr

// ------------------------------------------------------------------------------ options --
int option_index(const char* name) {
  for (int i = 0; i < kNumOptionSpecs; ++i)
    if (strcmp(kOptionSpecs[i].name, name) == 0) return i;
  return -1;
}

int opt_of(const Bank* bank, int Options::*slot) {
  if (bank)
    for (const auto& o : bank->overrides)
      if (kOptionSpecs[o.first].slot == slot) return o.second;
  return g_opt.*slot;
}

// A value the option's range admits but the option does not: one batch has no spread.
bool option_value_invalid(const OptionSpec& spec, int value) {
  return spec.slot == &Options::tally_batches && value == 1;
}

// --------------------------------------------------------------------------- allocation --
template <typename T>
size_t device_zalloc(DeviceCtx& c, T** buf, size_t len) {
  const size_t bytes = sizeof(T) * (len ? len : 1);
  CU_FATAL(cudaMalloc((void**)buf, bytes));
  CU_FATAL(cudaMemsetAsync(*buf, 0, bytes, c.stream));
  return sizeof(T) * len;
}

size_t bank_alloc(DeviceCtx& c, BankView& b, int n) {
  size_t bytes = 0;
  bytes += device_zalloc(c, &b.pos, (size_t)n);
  bytes += device_zalloc(c, &b.dir, (size_t)n);
  bytes += device_zalloc(c, &b.ew, (size_t)n);
  bytes += device_zalloc(c, &b.tm, (size_t)n);
  bytes += device_zalloc(c, &b.meta, (size_t)n);
  return bytes;
}

void bank_release(BankView& b) {
  cudaFree(b.pos);
  cudaFree(b.dir);
  cudaFree(b.ew);
  cudaFree(b.tm);
  cudaFree(b.meta);
  b = BankView{};
}

size_t soa_alloc(DeviceCtx& c, SoaView& s, int n) {
  size_t bytes = 0;
  double** d[] = {&s.x, &s.y, &s.omega_x, &s.omega_y, &s.energy, &s.weight,
                  &s.dt_to_census, &s.mfp_to_collision};
  for (double** p : d) bytes += device_zalloc(c, p, (size_t)n);
  int** i[] = {&s.cellx, &s.celly, &s.dead};
  for (int** p : i) bytes += device_zalloc(c, p, (size_t)n);
  return bytes;
}

void soa_release(SoaView& s) {
  void* p[] = {s.x, s.y, s.omega_x, s.omega_y, s.energy, s.weight, s.dt_to_census,
               s.mfp_to_collision, s.cellx, s.celly, s.dead};
  for (void* q : p) cudaFree(q);
  s = SoaView{};
}

SoaView as_soa_view(const nb200_particle_soa& p) {
  SoaView s;
  s.x = p.x; s.y = p.y; s.omega_x = p.omega_x; s.omega_y = p.omega_y;
  s.energy = p.energy; s.weight = p.weight; s.dt_to_census = p.dt_to_census;
  s.mfp_to_collision = p.mfp_to_collision;
  s.cellx = p.cellx; s.celly = p.celly; s.dead = p.dead;
  return s;
}

nb200_particle_soa as_public(const SoaView& s) {
  nb200_particle_soa p;
  p.x = s.x; p.y = s.y; p.omega_x = s.omega_x; p.omega_y = s.omega_y;
  p.energy = s.energy; p.weight = s.weight; p.dt_to_census = s.dt_to_census;
  p.mfp_to_collision = s.mfp_to_collision;
  p.cellx = s.cellx; p.celly = s.celly; p.dead = s.dead;
  return p;
}

// Element offset view of a host SoA (the slice that one shard covers).
SoaView soa_offset(const SoaView& s, size_t off) {
  SoaView o;
  o.x = s.x + off; o.y = s.y + off; o.omega_x = s.omega_x + off; o.omega_y = s.omega_y + off;
  o.energy = s.energy + off; o.weight = s.weight + off;
  o.dt_to_census = s.dt_to_census + off; o.mfp_to_collision = s.mfp_to_collision + off;
  o.cellx = s.cellx + off; o.celly = s.celly + off; o.dead = s.dead + off;
  return o;
}

nb200_particle_soa* views_of(BankHeader* h) { return reinterpret_cast<nb200_particle_soa*>(h + 1); }

void set_views(Bank* bank, const nb200_particle_soa& v) {
  nb200_particle_soa* views = views_of(bank->header);
  for (uint64_t i = 0; i < bank->header->nviews; ++i) views[i] = v;
}

// omp3's thread split (omp3/neutral.c:64-74) applied to GPUs: shard g of G.
void shard_split(int n, int g, int G, int* first, int* count) {
  const int per = n / G, rem = n % G;
  *first = g * per + std::min(g, rem);
  *count = per + (g < rem ? 1 : 0);
}

// A new bank of n particles holding global particles [pid0, pid0 + n), sharded over `ngpus`
// GPUs starting with the current one. Allocates the device arrays; fills nothing.
Bank* new_bank(int n, uint64_t pid0, int ngpus, int headroom_pct, bool mirror, size_t* bytes) {
  DeviceCtx& primary = ctx_required();
  int count = 1;
  CU_FATAL(cudaGetDeviceCount(&count));
  ngpus = std::max(1, ngpus);
  if (ngpus > count)
    terminate("ngpus=%d GPUs requested (NB200_NGPUS / option ngpus) but only %d visible", ngpus,
              count);
  if (ngpus > 1 && g_mp)
    terminate("a multi-process group is active on this process: banks are single-GPU");
  Bank* bank = new Bank();
  bank->n = n;
  bank->pid0 = pid0;
  bank->primary_dev = primary.device;
  size_t total = 0;
  for (int g = 0; g < ngpus; ++g) {
    Shard sh;
    sh.dev = (primary.device + g) % count;
    shard_split(n, g, ngpus, &sh.first, &sh.n);
    sh.pid0 = pid0 + (uint64_t)sh.first;
    sh.n_upper = sh.n;
    sh.capacity = sh.n + (int)(((long long)sh.n * headroom_pct + 99) / 100);
    DeviceGuard guard(sh.dev);
    DeviceCtx& c = ctx_on(sh.dev);
    total += bank_alloc(c, sh.cur, sh.capacity);
    // the double buffer of the per-step sort and its keys: allocated with the bank, so that the
    // first timestep (which main.c times like any other) does not pay for them
    total += bank_alloc(c, sh.alt, sh.capacity);
    total += device_zalloc(c, &sh.keys, (size_t)sh.capacity);
    sh.has_alt = true;
    bank->shards.push_back(sh);
  }
  const uint64_t nviews = mirror ? (uint64_t)std::max(n, 1) : 1;
  BankHeader* h = (BankHeader*)calloc(1, sizeof(BankHeader) + sizeof(nb200_particle_soa) * nviews);
  if (!h) terminate("out of host memory for a bank handle of %llu views", (unsigned long long)nviews);
  h->magic = kBankMagic;
  h->impl = bank;
  h->nviews = nviews;
  bank->header = h;
  g_handles.insert(views_of(h));
  if (mirror) {
    const size_t m = (size_t)std::max(n, 1);
    nb200_particle_soa& a = bank->mirror.a;
    double** d[] = {&a.x, &a.y, &a.omega_x, &a.omega_y, &a.energy, &a.weight, &a.dt_to_census,
                    &a.mfp_to_collision};
    for (double** p : d) CU_FATAL(cudaHostAlloc((void**)p, sizeof(double) * m, cudaHostAllocPortable));
    int** i[] = {&a.cellx, &a.celly, &a.dead};
    for (int** p : i) CU_FATAL(cudaHostAlloc((void**)p, sizeof(int) * m, cudaHostAllocPortable));
    bank->mirror.present = true;
    set_views(bank, a);
  }
  if (bytes) *bytes = total;
  return bank;
}

Bank* bank_of(nb200_particle_soa* particles) {
  // only pointers this library handed out are looked behind (the header sits in front of them)
  if (!particles || !g_handles.count(particles)) return nullptr;
  BankHeader* h = reinterpret_cast<BankHeader*>(particles) - 1;
  if (h->magic != kBankMagic || !h->impl) return nullptr;
  return h->impl;
}

nb200_particle_soa* handle_of(Bank* bank) { return views_of(bank->header); }

bool single_shard(const Bank* bank) { return bank->shards.size() == 1; }

// ------------------------------------------------------------------------ tally batches --
// Why a bank of n particles with global pids [pid0, pid0 + n) cannot have B tally batches under
// the current defaults, or nullptr. The batches are ranges of the whole run's pids: the bank
// must hold all of them, on one GPU, and be stepped by the batched history kernel.
const char* why_no_batches(int B, int n, uint64_t pid0, int ngpus) {
  static char why[256];
  if (B <= 0) return nullptr;
  if (ngpus > 1 || g_mp)
    return "tally_batches: a bank sharded over several GPUs or in a multi-process group has no "
           "batched tally";
  if (pid0 != 0) {
    snprintf(why, sizeof(why), "tally_batches: the bank starts at particle %llu; batches need "
             "the whole run's particles from 0", (unsigned long long)pid0);
    return why;
  }
  if (B > n) {
    snprintf(why, sizeof(why), "tally_batches=%d exceeds the bank's %d particles", B, n);
    return why;
  }
  if (!g_opt.pipeline) return "tally_batches: needs option pipeline=1 (the direct kernel has no batches)";
  if (g_opt.tally_prereduce) return "tally_batches: cannot be combined with tally_prereduce=1";
  return nullptr;
}

void batches_attach(Bank* bank, int B) {
  if (B <= 0) return;
  bank->batches.B = B;
  g_batched.push_back(bank);
}

// Brings the target of `tb` up to date (the caller's tally for bank->batches, the attached flux
// array for bank->flux_batches): target += sum_b S_b - F, F = sum_b S_b. Synchronous.
void batches_flush(Bank* bank, TallyBatches& tb) {
  if (!tb.dirty || !tb.target) return;
  const Shard& sh = bank->shards[0];
  DeviceGuard guard(sh.dev);
  DeviceCtx& c = ctx_on(sh.dev);
  c.launches += launch_batch_flush(tb.slab, tb.B, tb.ncells, tb.target, c.stream);
  CU_FATAL(cudaGetLastError());
  CU_FATAL(cudaStreamSynchronize(c.stream));
  tb.dirty = false;
}

// Flushes `tb` into its target (if it still has one), frees its slab and clears it.
void batches_release(Bank* bank, TallyBatches& tb) {
  if (tb.B <= 0) return;
  batches_flush(bank, tb);
  if (tb.slab) {
    DeviceGuard guard(bank->shards[0].dev);
    cudaFree(tb.slab);
  }
  tb = TallyBatches{};
}

// Binds the batches to the tally and mesh of a timestep (before it is enqueued): another tally
// or mesh flushes into the old target and starts over, as enqueue_step does for a group.
// Terminates on a step the batches cannot serve.
void batches_bind(Bank* bank, const StepRequest& rq) {
  TallyBatches& tb = bank->batches;
  const size_t ncells = (size_t)rq.nx * (size_t)rq.ny;
  if (!single_shard(bank) || bank->pid0 != 0 || rq.ntotal != bank->n)
    terminate("solve_transport_2d: a bank with tally_batches must hold the whole run on one GPU "
              "(bank: %d particles from %llu on %zu GPU(s); ntotal_particles = %d)", bank->n,
              (unsigned long long)bank->pid0, bank->shards.size(), rq.ntotal);
  if (g_mp) terminate("solve_transport_2d: tally_batches in a multi-process group");
  if (!opt_of(bank, &Options::pipeline) || opt_of(bank, &Options::tally_prereduce))
    terminate("solve_transport_2d: tally_batches needs pipeline=1 and tally_prereduce=0");
  if ((unsigned long long)ncells * (unsigned long long)tb.B >= (1ull << 31))
    terminate("solve_transport_2d: tally_batches=%d over %zu cells needs 2^31 or more tally "
              "slots (the history kernel indexes them with 32 bits)", tb.B, ncells);
  if (tb.target == rq.tally && tb.ncells == ncells) return;
  batches_flush(bank, tb);
  const Shard& sh = bank->shards[0];
  DeviceGuard guard(sh.dev);
  DeviceCtx& c = ctx_on(sh.dev);
  const size_t bytes = sizeof(double) * (size_t)(tb.B + 1) * ncells;
  if (tb.ncells != ncells || !tb.slab) {
    if (tb.slab) {
      CU_FATAL(cudaStreamSynchronize(c.stream));
      cudaFree(tb.slab);
    }
    CU_FATAL(cudaMalloc(&tb.slab, bytes));
    tb.ncells = ncells;
  }
  CU_FATAL(cudaMemsetAsync(tb.slab, 0, bytes, c.stream));
  tb.target = rq.tally;
}

// R of the total of `tb` (tally or flux): the B batch totals through a fixed-order device
// reduction, then the estimator in FP64 on the host.
double batches_total_relerr(Bank* bank, const TallyBatches& tb) {
  const Shard& sh = bank->shards[0];
  DeviceGuard guard(sh.dev);
  DeviceCtx& c = ctx_on(sh.dev);
  const size_t np = (size_t)tb.B * kBatchSumBlocks;
  double* d_partial = nullptr;
  CU_FATAL(cudaMalloc(&d_partial, sizeof(double) * np));
  c.launches += launch_batch_sums(tb.slab, tb.B, tb.ncells, d_partial, c.stream);
  std::vector<double> h(np);
  CU_FATAL(cudaMemcpyAsync(h.data(), d_partial, sizeof(double) * np, cudaMemcpyDeviceToHost,
                           c.stream));
  CU_FATAL(cudaStreamSynchronize(c.stream));
  cudaFree(d_partial);
  std::vector<double> x(tb.B);
  double sum = 0.0;
  for (int b = 0; b < tb.B; ++b) {
    double t = 0.0;
    for (int k = 0; k < kBatchSumBlocks; ++k) t += h[(size_t)b * kBatchSumBlocks + k];
    const int nb = bank->n / tb.B + (b < bank->n % tb.B ? 1 : 0);
    x[b] = t * (double)bank->n / (double)nb;
    sum += x[b];
  }
  const double m = sum / (double)tb.B;
  double ss = 0.0;
  for (int b = 0; b < tb.B; ++b) ss += (x[b] - m) * (x[b] - m);
  const double var = ss / (double)(tb.B - 1);
  return m == 0.0 ? 0.0 : sqrt(var / (double)tb.B) / fabs(m);
}

Bank* batched_bank_of_tally(const double* tally) {
  for (Bank* b : g_batched)
    if (b->batches.target == tally && b->batches.slab) return b;
  return nullptr;
}

// ------------------------------------------------------------------------- flux tally --
// `flux` null detaches. The attachment is the bank's own: nb200_bank_copy does not move it.
// A batched flux of the old attachment is flushed into the old array and its slab freed first.
// B > 0 attaches a batched flux: deposits go to a zeroed slab of B partial fluxes on the bank's
// GPU, allocated here. Returns 0, or -2 (error set) when the slab cannot be had.
int flux_attach(Bank* bank, double* flux, size_t ncells, int B = 0) {
  batches_release(bank, bank->flux_batches);
  g_flux.erase(std::remove(g_flux.begin(), g_flux.end(), bank), g_flux.end());
  bank->flux = nullptr;
  bank->flux_ncells = 0;
  if (!flux) return 0;
  if (B > 0) {
    DeviceGuard guard(bank->shards[0].dev);
    DeviceCtx& c = ctx_on(bank->shards[0].dev);
    const size_t bytes = sizeof(double) * (size_t)(B + 1) * ncells;
    double* slab = nullptr;
    CU_TRY(cudaMalloc(&slab, bytes));
    if (cudaError_t err = cudaMemsetAsync(slab, 0, bytes, c.stream)) {
      cudaFree(slab);
      set_error("cudaMemsetAsync of the flux batch slab failed: %s", cudaGetErrorString(err));
      return -2;
    }
    // the bank has a batched flux only once its slab is whole
    TallyBatches& tb = bank->flux_batches;
    tb.slab = slab;
    tb.B = B;
    tb.ncells = ncells;
    tb.target = flux;
  }
  bank->flux = flux;
  bank->flux_ncells = ncells;
  g_flux.push_back(bank);
  return 0;
}

// deallocate_data of an attached array: no later timestep may write into the freed memory, and
// nothing is flushed into it.
void flux_detach_array(const double* buf) {
  std::vector<Bank*> attached;
  for (Bank* b : g_flux)
    if (b->flux == buf) attached.push_back(b);
  for (Bank* b : attached) {
    b->flux_batches.target = nullptr;
    flux_attach(b, nullptr, 0);
  }
}

// Terminates on a timestep the flux kernel cannot serve (before it is enqueued): another mesh,
// or options changed since the array was attached.
void flux_check(Bank* bank, const StepRequest& rq, bool grouped) {
  const size_t ncells = (size_t)rq.nx * (size_t)rq.ny;
  if (ncells != bank->flux_ncells)
    terminate("solve_transport_2d: the bank's flux tally has %zu cells, the mesh has %d x %d = "
              "%zu", bank->flux_ncells, rq.nx, rq.ny, ncells);
  if (grouped || !single_shard(bank))
    terminate("solve_transport_2d: a flux tally in a sharded or multi-process run");
  if (!opt_of(bank, &Options::pipeline) || opt_of(bank, &Options::tally_prereduce))
    terminate("solve_transport_2d: a flux tally needs pipeline=1 and tally_prereduce=0");
}

// Uploads host SoA slices into the shards of `bank` (origins from 0 within each shard).
void upload_host_soa(Bank* bank, const SoaView& host) {
  for (Shard& sh : bank->shards) {
    if (sh.n <= 0) continue;
    DeviceGuard guard(sh.dev);
    DeviceCtx& c = ctx_on(sh.dev);
    SoaView staging{};
    soa_alloc(c, staging, sh.n);
    const SoaView h = soa_offset(host, (size_t)sh.first);
    const double* hd[] = {h.x, h.y, h.omega_x, h.omega_y, h.energy, h.weight, h.dt_to_census,
                          h.mfp_to_collision};
    double* dd[] = {staging.x, staging.y, staging.omega_x, staging.omega_y, staging.energy,
                    staging.weight, staging.dt_to_census, staging.mfp_to_collision};
    for (int k = 0; k < 8; ++k)
      CU_FATAL(cudaMemcpyAsync(dd[k], hd[k], sizeof(double) * sh.n, cudaMemcpyHostToDevice,
                               c.stream));
    const int* hi[] = {h.cellx, h.celly, h.dead};
    int* di[] = {staging.cellx, staging.celly, staging.dead};
    for (int k = 0; k < 3; ++k)
      CU_FATAL(cudaMemcpyAsync(di[k], hi[k], sizeof(int) * sh.n, cudaMemcpyHostToDevice,
                               c.stream));
    c.launches += launch_import_soa(sh.cur, staging, sh.n, 0, c.stream);
    CU_FATAL(cudaStreamSynchronize(c.stream));
    soa_release(staging);
    sh.n_upper = sh.n;
  }
}

void ensure_export(DeviceCtx& c, Shard& sh) {
  if (sh.has_export) return;
  soa_alloc(c, sh.exported, sh.capacity);
  sh.has_export = true;
}

// Copies the bank to host SoA arrays in injection order (synchronous).
void download_to_host(Bank* bank, const SoaView& host) {
  for (Shard& sh : bank->shards) {
    if (sh.n <= 0) continue;
    DeviceGuard guard(sh.dev);
    DeviceCtx& c = ctx_on(sh.dev);
    ensure_export(c, sh);
    c.launches += launch_export_soa(sh.cur, sh.exported, sh.n, c.stream);
    const SoaView& s = sh.exported;
    const SoaView h = soa_offset(host, (size_t)sh.first);
    const double* dd[] = {s.x, s.y, s.omega_x, s.omega_y, s.energy, s.weight, s.dt_to_census,
                          s.mfp_to_collision};
    double* hd[] = {h.x, h.y, h.omega_x, h.omega_y, h.energy, h.weight, h.dt_to_census,
                    h.mfp_to_collision};
    for (int k = 0; k < 8; ++k)
      CU_FATAL(cudaMemcpyAsync(hd[k], dd[k], sizeof(double) * sh.n, cudaMemcpyDeviceToHost,
                               c.stream));
    const int* di[] = {s.cellx, s.celly, s.dead};
    int* hi[] = {h.cellx, h.celly, h.dead};
    for (int k = 0; k < 3; ++k)
      CU_FATAL(cudaMemcpyAsync(hi[k], di[k], sizeof(int) * sh.n, cudaMemcpyDeviceToHost,
                               c.stream));
  }
  for (Shard& sh : bank->shards) {
    DeviceGuard guard(sh.dev);
    CU_FATAL(cudaStreamSynchronize(ctx_on(sh.dev).stream));
  }
}

void refresh_mirror(Bank* bank) {
  if (bank->mirror.present) download_to_host(bank, as_soa_view(bank->mirror.a));
}

// --------------------------------------------------------------------- scheduling hints --
CsParams cs_params_from_ends(double k_first, double k_last, int n) {
  CsParams p;
  if (n >= 2 && k_first > 0.0 && k_last > k_first) {
    unsigned long long lo, hi;
    memcpy(&lo, &k_first, 8);
    memcpy(&hi, &k_last, 8);
    p.bits0 = lo;
    p.nb = kCsBuckets;
    p.shift = 0;
    while (((hi - lo) >> p.shift) >= (unsigned long long)p.nb) p.shift++;
  }
  return p;
}

// Which leading bits spread a table's keys over its bucket index: read off the first and the
// last key once per (pointer, size). A hint, not an input: the index is exact for any
// parameters (nb_bank.cuh: CsStage), stale ones only fill the buckets less evenly. Cached so
// that no timestep of a known table issues a device-to-host copy, which would queue behind
// whatever bulk download the caller has in flight on the same copy engine.
CsParams table_hint(DeviceCtx& c, const double* keys, int n) {
  for (const auto& t : c.table_cache)
    if (t.keys == keys && t.n == n) return t.par;
  double ends[2] = {0.0, 0.0};
  if (n >= 2) {
    CU_FATAL(cudaMemcpyAsync(&ends[0], keys, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    CU_FATAL(cudaMemcpyAsync(&ends[1], keys + n - 1, sizeof(double), cudaMemcpyDeviceToHost,
                             c.stream));
    CU_FATAL(cudaStreamSynchronize(c.stream));
  }
  const CsParams par = cs_params_from_ends(ends[0], ends[1], n);
  if (c.table_cache.size() >= 16) c.table_cache.erase(c.table_cache.begin());
  c.table_cache.push_back({keys, n, par});
  return par;
}

// Extent of the mesh, for the sort's history-length estimate (a scheduling hint only).
void mesh_hint(DeviceCtx& c, const double* edgex, const double* edgey, int nx, int ny,
               double* width, double* height) {
  for (const auto& m : c.mesh_cache)
    if (m.ex == edgex && m.ey == edgey && m.nx == nx && m.ny == ny) {
      *width = m.width;
      *height = m.height;
      return;
    }
  double ex[2], ey[2];
  CU_FATAL(cudaMemcpyAsync(&ex[0], edgex, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  CU_FATAL(cudaMemcpyAsync(&ex[1], edgex + nx, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  CU_FATAL(cudaMemcpyAsync(&ey[0], edgey, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  CU_FATAL(cudaMemcpyAsync(&ey[1], edgey + ny, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  CU_FATAL(cudaStreamSynchronize(c.stream));
  *width = ex[1] > ex[0] ? ex[1] - ex[0] : 1.0;
  *height = ey[1] > ey[0] ? ey[1] - ey[0] : 1.0;
  if (c.mesh_cache.size() >= 16) c.mesh_cache.erase(c.mesh_cache.begin());
  c.mesh_cache.push_back({edgex, edgey, nx, ny, *width, *height});
}

// The step totals reach the host through mapped pinned memory, written by the device itself:
// a cudaMemcpyAsync would wait its turn on the device-to-host copy engine behind any bulk
// download the caller has in flight (measured: 3.4 ms per deck run in bench.py's e2e loop).
// In a sharded run the same kernel raises the rank's `ready` flag: the history kernel in front
// of it in stream order has deposited the whole delta (nb_group.cuh).
__global__ void k_publish_totals(const unsigned long long* __restrict__ totals,
                                 volatile unsigned long long* host_totals, SyncBlock* sync,
                                 unsigned long long epoch) {
  if (threadIdx.x < kTotCount) {
    unsigned long long v = totals[threadIdx.x];
    if (sync && threadIdx.x == kTotGroupFault) v = sync->fault;
    host_totals[threadIdx.x] = v;
  }
  __threadfence_system();
  if (sync && threadIdx.x == 0)
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(&sync->ready), "l"(epoch) : "memory");
}

// Restages both tables into the device's own block (stage.cu) and fills the views. With
// `reserve_only` nothing is launched: the hints are fetched and the block sized (what has to
// happen before a timestep is recorded into a graph).
void stage_tables(DeviceCtx& c, StepArgs& a, bool reserve_only = false) {
  const CsParams ps = table_hint(c, a.s_keys, a.s_n), pa = table_hint(c, a.a_keys, a.a_n);
  auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t kv_s = align(sizeof(double2) * a.s_n), kv_a = align(sizeof(double2) * a.a_n);
  const size_t bk_s = align(sizeof(int) * (ps.nb + 1));
  const size_t bk_a = align(sizeof(int) * (pa.nb + 1));
  const size_t need = kv_s + kv_a + bk_s + bk_a;
  if (c.cs_stage_bytes < need) {
    // the block may still be read by a timestep in flight: freeing synchronises the device
    cudaFree(c.d_cs_stage);
    CU_FATAL(cudaMalloc(&c.d_cs_stage, need));
    c.cs_stage_bytes = need;
  }
  if (reserve_only) return;
  char* p = c.d_cs_stage;
  double2* d_kv_s = (double2*)p; p += kv_s;
  double2* d_kv_a = (double2*)p; p += kv_a;
  int* d_bk_s = (int*)p; p += bk_s;
  int* d_bk_a = (int*)p;
  c.launches += launch_stage_cs(a.s_keys, a.s_vals, a.s_n, d_kv_s, d_bk_s, ps.bits0, ps.shift,
                                ps.nb, a.same_keys ? a.a_keys : nullptr, a.totals, c.work);
  c.launches += launch_stage_cs(a.a_keys, a.a_vals, a.a_n, d_kv_a, d_bk_a, pa.bits0, pa.shift,
                                pa.nb, nullptr, a.totals, c.work);
  a.cs_s = CsStage{d_kv_s, d_bk_s, ps.bits0, ps.shift, ps.nb, a.s_n};
  a.cs_a = CsStage{d_kv_a, d_bk_a, pa.bits0, pa.shift, pa.nb, a.a_n};
}

// Per-mesh staging blocks of a device (tile maps, target-edge rows) and the sort's histogram
// for the default key space. Sized when a bank is created for a mesh (inject_particles knows
// nx and ny), so that the first timestep - which the driver times like any other - finds them.
void reserve_mesh_scratch(DeviceCtx& c, int nx, int ny, long long nbins) {
  const int nfine = (((nx - 1) >> kTileShift) + 1) * (((ny - 1) >> kTileShift) + 1);
  const int ncoarse = (((nx - 1) >> kCoarseShift) + 1) * (((ny - 1) >> kCoarseShift) + 1);
  if (c.tile_capacity < nfine + ncoarse) {
    cudaFree(c.d_tile_rho);
    CU_FATAL(cudaMalloc(&c.d_tile_rho, sizeof(double) * (nfine + ncoarse)));
    c.tile_capacity = nfine + ncoarse;
  }
  const int stride = ((std::max(nx, ny) + 1 + 31) / 32) * 32;
  if (c.edges_capacity < 4 * stride) {
    cudaFree(c.d_edges4);
    CU_FATAL(cudaMalloc(&c.d_edges4, sizeof(double) * 4 * (size_t)stride));
    c.edges_capacity = 4 * stride;
  }
  if (c.bins_capacity < nbins) {
    cudaFree(c.d_bins);
    // histogram, cursors, and one scan partial per 2048 bins
    CU_FATAL(cudaMalloc(&c.d_bins, sizeof(unsigned) * (2 * (size_t)nbins + nbins / 2048 + 1)));
    c.bins_capacity = nbins;
  }
  // the staged cross-section block for two tables of the reference's size (grown on demand)
  const size_t cs_guess = 2 * (((sizeof(double2) * 32768) + 255) & ~(size_t)255) +
                          2 * (((sizeof(int) * (kCsBuckets + 1)) + 255) & ~(size_t)255);
  if (c.cs_stage_bytes < cs_guess) {
    cudaFree(c.d_cs_stage);
    CU_FATAL(cudaMalloc(&c.d_cs_stage, cs_guess));
    c.cs_stage_bytes = cs_guess;
  }
}

// The sort's key space for a mesh under the given options: 3 classes x length bins x tiles + the
// dead bin, in 64 bits; a combination that asks for more bins than the scratch is worth gets
// coarser tiles (a scheduling key, nothing else).
long long sort_key_space(int nx, int ny, int length_bins, int* tile_shift, int* tiles_x,
                         int* ntiles) {
  const long long nq = std::max(length_bins, 1);
  long long nt = 1, tx = 1;
  for (;; ++*tile_shift) {
    tx = *tile_shift >= 0 ? ((nx - 1) >> *tile_shift) + 1 : 1;
    nt = *tile_shift >= 0 ? tx * (((ny - 1) >> *tile_shift) + 1) : 1;
    if (*tile_shift < 0 || 3ll * nq * nt + 1 <= (1ll << 24)) break;
  }
  *tiles_x = (int)tx;
  *ntiles = (int)nt;
  return 3ll * nq * nt + 1;
}

void stage_tiles(DeviceCtx& c, StepArgs& a, cudaStream_t st) {
  const int nfine = (((a.nx - 1) >> kTileShift) + 1) * (((a.ny - 1) >> kTileShift) + 1);
  reserve_mesh_scratch(c, a.nx, a.ny, 0);
  c.launches += launch_stage_tiles(a.density, a.nx, a.ny, c.d_tile_rho, c.d_tile_rho + nfine,
                                   &a.tiles, st);
  // ... and the target-edge rows (same consumer: the event loop only)
  const int stride = ((std::max(a.nx, a.ny) + 1 + 31) / 32) * 32;
  c.launches += launch_stage_edges(a.edgex, a.nx, a.edgey, a.ny, stride, c.d_edges4, st);
  a.edges4 = c.d_edges4;
  a.edge_stride = stride;
}

int take_slot(DeviceCtx& c) {
  for (int tries = 0; tries < kRing; ++tries) {
    const int s = (c.next_slot + tries) % kRing;
    if (!c.slot_busy[s]) {
      c.slot_busy[s] = true;
      c.next_slot = (s + 1) % kRing;
      return s;
    }
  }
  terminate("more than %d timesteps in flight on GPU %d: collect them with nb200_solve_finish",
            kRing, c.device);
}

// What one shard's timestep reads and writes, as pointers on the shard's own GPU.
struct ShardIO {
  const double *density, *edgex, *edgey, *s_keys, *s_vals, *a_keys, *a_vals;
  double* tally;
  uint64_t *r0, *r1, *r2;
  BatchArgs batches;
  double* flux;  // track-length flux array, or null
};

// An event the host will wait on or read a time from. While a timestep is being recorded into
// a graph it has to become an event-record NODE (cudaEventRecordExternal); a plain record
// inside a capture is only an edge between the captured streams.
void record_external(DeviceCtx& c, cudaEvent_t ev) {
  if (c.work == c.capture)
    CU_FATAL(cudaEventRecordWithFlags(ev, c.work, cudaEventRecordExternal));
  else
    CU_FATAL(cudaEventRecord(ev, c.work));
}

// Everything a timestep of this shard may have to allocate or read back (hints), done ahead of
// the timestep's own calls - nothing of this kind may happen while a graph is being recorded.
void prepare_shard_step(DeviceCtx& c, const Bank* bank, Shard& sh, const StepRequest& rq,
                        const ShardIO& io) {
  if (!opt_of(bank, &Options::pipeline)) return;
  double w, h;
  mesh_hint(c, io.edgex, io.edgey, rq.nx, rq.ny, &w, &h);
  StepArgs a{};
  a.s_keys = io.s_keys;
  a.s_n = rq.s_n;
  a.a_keys = io.a_keys;
  a.a_n = rq.a_n;
  stage_tables(c, a, true);
  int shift = opt_of(bank, &Options::tile_shift), tx = 1, nt = 1;
  const long long nbins = sort_key_space(rq.nx, rq.ny, opt_of(bank, &Options::length_bins), &shift,
                                         &tx, &nt);
  reserve_mesh_scratch(c, rq.nx, rq.ny, nbins);
  if (!sh.has_alt) {
    bank_alloc(c, sh.alt, sh.capacity);
    device_zalloc(c, &sh.keys, (size_t)sh.capacity);
    sh.has_alt = true;
  }
}

// The calls of one timestep of one shard, issued on c.work (the device is current): the
// device's stream, or its capture stream while the timestep is being recorded into a graph.
void record_shard_step(DeviceCtx& c, const Bank* bank, Shard& sh, const StepRequest& rq,
                       const ShardIO& io, int slot, SyncBlock* sync, unsigned long long epoch) {
  StepArgs a{};
  a.nx = rq.nx;
  a.ny = rq.ny;
  a.n = sh.n;
  a.master_key = rq.master_key;
  a.pid0 = sh.pid0;
  a.dt = rq.dt;
  a.inv_ntotal = 1.0 / (double)rq.ntotal;  // omp3/neutral.c:120
  a.density = io.density;
  a.edgex = io.edgex;
  a.edgey = io.edgey;
  a.s_keys = io.s_keys;
  a.s_vals = io.s_vals;
  a.s_n = rq.s_n;
  a.a_keys = io.a_keys;
  a.a_vals = io.a_vals;
  a.a_n = rq.a_n;
  a.same_keys = rq.s_n == rq.a_n;  // necessary; the staging kernel decides (same_grid())
  a.tally = io.tally;
  a.p_facets = (unsigned long long*)io.r0;
  a.p_collisions = (unsigned long long*)io.r1;
  a.p_census = (unsigned long long*)io.r2;
  a.totals = c.d_totals;
  a.bank = sh.cur;
  a.logt = c.d_logt;

  const int opt_l2 = opt_of(bank, &Options::l2_persist);
  CU_FATAL(cudaMemsetAsync(c.d_totals, 0, sizeof(unsigned long long) * kTotCount, c.work));
  record_external(c, c.ev_begin[slot]);
  if (opt_of(bank, &Options::pipeline)) {
    double mesh_w = 1.0, mesh_h = 1.0;
    mesh_hint(c, io.edgex, io.edgey, rq.nx, rq.ny, &mesh_w, &mesh_h);
    if (opt_l2 && !c.l2_limit_set) {  // set-aside for the persisting window
      size_t want = 4u << 20;
      if (opt_l2 == 2) {  // experiment: persist (part of) the tally instead
        int max_bytes = 0;
        CU_FATAL(cudaDeviceGetAttribute(&max_bytes, cudaDevAttrMaxPersistingL2CacheSize, c.device));
        want = (size_t)max_bytes;
      }
      CU_FATAL(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want));
      CU_FATAL(cudaDeviceGetLimit(&c.l2_setaside, cudaLimitPersistingL2CacheSize));
      c.l2_limit_set = true;
    }
    // P0: restage the read-only inputs (cross-section tables, density tile map)
    const bool overlap = opt_of(bank, &Options::stage_overlap) != 0;
    if (overlap) {
      CU_FATAL(cudaEventRecord(c.ev_fork, c.work));
      CU_FATAL(cudaStreamWaitEvent(c.stage_stream, c.ev_fork, 0));
      stage_tiles(c, a, c.stage_stream);
      CU_FATAL(cudaEventRecord(c.ev_tiles, c.stage_stream));
    }
    stage_tables(c, a);
    if (!overlap) stage_tiles(c, a, c.work);
    // P1-P3: begin-step set-up, classification and counting sort into the double buffer
    SortArgs s{};
    s.nq = std::max(opt_of(bank, &Options::length_bins), 1);
    s.tile_shift = opt_of(bank, &Options::tile_shift);
    s.nbins = (int)sort_key_space(rq.nx, rq.ny, s.nq, &s.tile_shift, &s.tiles_x, &s.ntiles);
    s.q_scale = 24.0f;  // 12 bins across the sqrt(2) spread of facet counts with direction
    s.inv_dx = (float)((double)rq.nx / mesh_w);
    s.inv_dy = (float)((double)rq.ny / mesh_h);
    s.n_upper = sh.n_upper;
    s.n = sh.n;
    if (!sh.has_alt) {
      bank_alloc(c, sh.alt, sh.capacity);
      device_zalloc(c, &sh.keys, (size_t)sh.capacity);
      sh.has_alt = true;
    }
    reserve_mesh_scratch(c, rq.nx, rq.ny, s.nbins);
    s.keys = sh.keys;
    s.bin_count = c.d_bins;
    s.bin_cursor = c.d_bins + s.nbins;
    s.chunk_sum = c.d_bins + 2 * (size_t)s.nbins;
    s.n_live = c.d_n_live;
    c.launches += launch_sort_phase(a, s, sh.alt, c.work);
    if (s.n_upper > 0) {  // the sort ran: the double buffer now holds the bank
      std::swap(sh.cur, sh.alt);
      a.bank = sh.cur;
    }
    if (overlap) CU_FATAL(cudaStreamWaitEvent(c.work, c.ev_tiles, 0));
    record_external(c, c.ev_mid[slot]);
    // P4: event loop over the sorted live prefix
    a.stagger_at = opt_of(bank, &Options::stagger_at);
    a.stagger_share = opt_of(bank, &Options::stagger_share);
    a.stagger_min = opt_of(bank, &Options::stagger_min);
    const bool fast_div = opt_of(bank, &Options::fast_div) != 0;
    c.launches += launch_history(a, io.batches, io.flux, c.d_n_live, s.n_upper, fast_div,
                                 opt_of(bank, &Options::tally_prereduce) != 0,
                                 opt_l2 == 2 ? (const void*)io.tally
                                 : opt_l2    ? (const void*)c.d_cs_stage : nullptr,
                                 opt_l2 == 2 ? sizeof(double) * (size_t)rq.nx * rq.ny
                                             : c.cs_stage_bytes,
                                 opt_l2 == 2 ? c.l2_setaside : 0,
                                 opt_of(bank, &Options::history_smem_pad), c.work);
  } else {
    if (a.same_keys)
      c.launches += launch_compare_grids(a.s_keys, a.a_keys, a.s_n, a.totals, c.work);
    record_external(c, c.ev_mid[slot]);
    c.launches += launch_history_direct(a, c.work);
  }
  CU_FATAL(cudaGetLastError());
  record_external(c, c.ev_end[slot]);
  k_publish_totals<<<1, 32, 0, c.work>>>(c.d_totals, c.h_totals_dev + (size_t)slot * kTotCount,
                                           sync, epoch);
  record_external(c, c.ev_pub[slot]);
  c.launches += 1;
}

// Enqueues one timestep of one shard on its device's stream (the device is current): call by
// call, or - option step_graph - recorded into a graph on the capture stream, which then
// updates the device's executable graph in place (same topology every timestep; only the
// parameters move) and goes out as ONE launch. A topology change (an option flipped, an empty
// bank) re-instantiates.
void enqueue_shard_step(DeviceCtx& c, const Bank* bank, Shard& sh, const StepRequest& rq,
                        const ShardIO& io, int slot, SyncBlock* sync, unsigned long long epoch) {
  prepare_shard_step(c, bank, sh, rq, io);
  const bool graph = opt_of(bank, &Options::step_graph) && opt_of(bank, &Options::pipeline) &&
                     !opt_of(bank, &Options::l2_persist) &&
                     !opt_of(bank, &Options::history_smem_pad);
  if (!graph) {
    c.work = c.stream;
    record_shard_step(c, bank, sh, rq, io, slot, sync, epoch);
    c.pending_steps++;
    return;
  }
  CU_FATAL(cudaStreamBeginCapture(c.capture, cudaStreamCaptureModeRelaxed));
  c.work = c.capture;
  record_shard_step(c, bank, sh, rq, io, slot, sync, epoch);
  c.work = c.stream;
  cudaGraph_t recorded = nullptr;
  CU_FATAL(cudaStreamEndCapture(c.capture, &recorded));
  bool fresh = c.step_exec == nullptr;
  if (!fresh) {
    cudaGraphExecUpdateResultInfo info{};
    if (cudaGraphExecUpdate(c.step_exec, recorded, &info) != cudaSuccess) {
      (void)cudaGetLastError();
      cudaGraphExecDestroy(c.step_exec);
      c.step_exec = nullptr;
      fresh = true;
    } else {
      c.graph_updates++;
    }
  }
  if (fresh) {
    CU_FATAL(cudaGraphInstantiate(&c.step_exec, recorded, 0));
    c.graph_instantiations++;
  }
  CU_FATAL(cudaGraphDestroy(recorded));
  CU_FATAL(cudaGraphLaunch(c.step_exec, c.stream));
  c.pending_steps++;
}

// ------------------------------------------------------------------------- tally groups --
size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Slab of one rank: SyncBlock | delta x 3 | owned | (NCCL flavour: tmp | gathered).
void group_layout(TallyGroup& g) {
  g.chunk = (g.ncells + g.nranks - 1) / g.nranks;
  g.chunk = (g.chunk + 1) & ~(size_t)1;  // even: 16-byte vector accesses never straddle slices
  g.padded = g.chunk * g.nranks;
  g.slab_bytes = align256(sizeof(SyncBlock)) + kDeltaBuffers * align256(g.padded * 8) +
                 align256(g.chunk * 8);
  if (!g.collective) g.slab_bytes += align256(g.chunk * 8) + align256(g.padded * 8);
}

void group_bind(TallyGroup& g, GroupMember& m, char* base) {
  m.slab = base;
  char* p = base;
  m.sync = (SyncBlock*)p; p += align256(sizeof(SyncBlock));
  for (int k = 0; k < kDeltaBuffers; ++k) { m.delta[k] = (double*)p; p += align256(g.padded * 8); }
  m.owned = (double*)p; p += align256(g.chunk * 8);
  if (!g.collective) {
    m.tmp = (double*)p; p += align256(g.chunk * 8);
    m.gathered = (double*)p;
  }
}

// Allocates the local member `rank` on device `dev` (made current by the caller).
void group_alloc_member(TallyGroup& g, int rank, int dev) {
  GroupMember& m = g.m[rank];
  m.dev = dev;
  char* base = nullptr;
  CU_FATAL(cudaMalloc(&base, g.slab_bytes));
  CU_FATAL(cudaMemset(base, 0, g.slab_bytes));
  group_bind(g, m, base);
  int lo = 0, hi = 0;
  CU_FATAL(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  // the collective of timestep t runs beside the transport of timestep t+1: let its (few,
  // small) CTAs in whenever an SM has room
  const char* prio = getenv("NB200_SIDE_PRIORITY");  // measurement knob: 0 = default priority
  CU_FATAL(cudaStreamCreateWithPriority(&m.side, cudaStreamNonBlocking,
                                        prio && atoi(prio) == 0 ? lo : hi));
  for (int k = 0; k < kDeltaBuffers; ++k) {
    CU_FATAL(cudaEventCreateWithFlags(&m.ev_hist[k], cudaEventDisableTiming));
    CU_FATAL(cudaEventCreateWithFlags(&m.ev_zeroed[k], cudaEventDisableTiming));
  }
  CU_FATAL(cudaEventCreateWithFlags(&m.ev_side, cudaEventDisableTiming));
}

void group_free(TallyGroup* g) {
  if (!g) return;
  g_groups.erase(std::remove(g_groups.begin(), g_groups.end(), g), g_groups.end());
  const NcclApi* api = g->collective ? nullptr : nccl_api(nullptr);
  for (int r = 0; r < g->nranks; ++r) {
    GroupMember& m = g->m[r];
    if (m.dev >= 0) {
      DeviceGuard guard(m.dev);
      cudaDeviceSynchronize();
      if (m.comm && api) api->CommDestroy(m.comm);
      if (m.side) cudaStreamDestroy(m.side);
      for (int k = 0; k < kDeltaBuffers; ++k) {
        if (m.ev_hist[k]) cudaEventDestroy(m.ev_hist[k]);
        if (m.ev_zeroed[k]) cudaEventDestroy(m.ev_zeroed[k]);
      }
      if (m.ev_side) cudaEventDestroy(m.ev_side);
      cudaFree(m.slab);
    } else if (m.ipc_opened) {
      cudaIpcCloseMemHandle(m.slab);
    }
  }
  delete g;
}

// Single-process group over the shards' devices: slabs, peer access, (optionally) NCCL.
TallyGroup* group_create_local(const Bank* bank, size_t ncells) {
  TallyGroup* g = new TallyGroup();
  g->nranks = (int)bank->shards.size();
  g->ncells = ncells;
  g->collective = opt_of(bank, &Options::collective);
  g->reduce_ctas = opt_of(bank, &Options::reduce_ctas);
  g->reduce_every = opt_of(bank, &Options::tally_reduce_every);
  if (g->collective) {  // the peer-memory kernel needs every pair of GPUs peer-mapped
    for (const Shard& a : bank->shards)
      for (const Shard& b : bank->shards) {
        if (a.dev == b.dev) continue;
        int can = 0;
        CU_FATAL(cudaDeviceCanAccessPeer(&can, a.dev, b.dev));
        if (!can) g->collective = 0;
      }
    if (!g->collective)
      fprintf(stderr, "neutral_b200: GPUs are not all peer-accessible: the tally collective "
                      "falls back to NCCL\n");
  }
  group_layout(*g);
  for (int r = 0; r < g->nranks; ++r) {
    DeviceGuard guard(bank->shards[r].dev);
    ctx_on(bank->shards[r].dev);
    group_alloc_member(*g, r, bank->shards[r].dev);
  }
  if (g->collective) {
    for (int r = 0; r < g->nranks; ++r) {
      DeviceGuard guard(g->m[r].dev);
      for (int q = 0; q < g->nranks; ++q) {
        if (q == r) continue;
        static bool enabled[kMaxDevices][kMaxDevices] = {{false}};  // once per pair and process
        if (enabled[g->m[r].dev][g->m[q].dev]) continue;
        const cudaError_t err = cudaDeviceEnablePeerAccess(g->m[q].dev, 0);
        if (err != cudaSuccess && err != cudaErrorPeerAccessAlreadyEnabled)
          terminate("cudaDeviceEnablePeerAccess(%d -> %d) failed: %s", g->m[r].dev, g->m[q].dev,
                    cudaGetErrorString(err));
        if (err != cudaSuccess) (void)cudaGetLastError();  // somebody else had enabled it
        enabled[g->m[r].dev][g->m[q].dev] = true;
      }
    }
  } else {
    std::string why;
    const NcclApi* api = nccl_api(&why);
    if (!api) terminate("the NCCL flavour of the tally collective was asked for, but %s", why.c_str());
    nccl_comm_t comms[kMaxRanks];
    int devs[kMaxRanks];
    for (int r = 0; r < g->nranks; ++r) devs[r] = g->m[r].dev;
    NCCL_FATAL(api, api->CommInitAll(comms, g->nranks, devs));
    for (int r = 0; r < g->nranks; ++r) g->m[r].comm = comms[r];
  }
  g_groups.push_back(g);
  return g;
}

// What rank `rank` waits for: 0 = every rank's `ready`, 1 = the `consumed` flags in its own
// block, 2 = every rank's `flush_ready`, 3 = the `flush_consumed` flags in its own block.
WaitList wait_list(const TallyGroup& g, int rank, int what) {
  WaitList w{};
  w.n = g.nranks;
  w.fault = &g.m[rank].sync->fault;
  for (int d = 0; d < g.nranks; ++d)
    w.flag[d] = what == 0   ? &g.m[d].sync->ready
                : what == 1 ? &g.m[rank].sync->consumed[d]
                : what == 2 ? &g.m[d].sync->flush_ready
                            : &g.m[rank].sync->flush_consumed[d];
  return w;
}

GroupView group_view(const TallyGroup& g, int rank, int k, bool owned_slices) {
  GroupView v{};
  v.nranks = g.nranks;
  v.rank = rank;
  v.chunk = g.chunk;
  v.ncells = g.ncells;
  for (int d = 0; d < g.nranks; ++d) {
    v.src[d] = owned_slices ? g.m[d].owned : g.m[d].delta[k];
    v.sync[d] = g.m[d].sync;
  }
  return v;
}

// Reduction number `g.epoch + 1` of the deposit buffer in use, for every LOCAL member, queued
// on the members' side streams behind the last history kernel that deposited into it (ev_hist):
// reduce-scatter of the buffer fused with the fold into the owned slice, then the buffer is
// cleared for its next turn and the ranks move on to the next of the three buffers.
// `signalled`: the last timestep's publish kernel already raised `ready` to this epoch (a
// reduction that was known when the timestep was enqueued); otherwise it is raised here.
void group_reduce(TallyGroup& g, bool signalled) {
  if (g.steps_deposited == 0) return;
  const unsigned long long epoch = ++g.epoch;
  const int k = g.cur_k;
  const NcclApi* api = g.collective ? nullptr : nccl_api(nullptr);
  for (int r = 0; r < g.nranks; ++r) {
    GroupMember& m = g.m[r];
    if (m.dev < 0) continue;
    DeviceGuard guard(m.dev);
    if (!signalled && g.collective) {
      DeviceCtx& c = ctx_on(m.dev);
      c.launches += launch_signal(m.sync, 0, epoch, c.stream);
      CU_FATAL(cudaEventRecord(m.ev_hist[k], c.stream));
    }
    CU_FATAL(cudaStreamWaitEvent(m.side, m.ev_hist[k], 0));
  }
  if (g.collective) {
    for (int r = 0; r < g.nranks; ++r) {
      GroupMember& m = g.m[r];
      if (m.dev < 0) continue;
      DeviceGuard guard(m.dev);
      DeviceCtx& c = ctx_on(m.dev);
      c.launches += launch_wait_flags(wait_list(g, r, 0), epoch, m.side);
      c.launches += launch_reduce_fold(group_view(g, r, k, false), m.owned, epoch, g.reduce_ctas,
                                       m.side);
      // every rank has read its slice of this delta: clear it for its reuse in three epochs
      c.launches += launch_wait_flags(wait_list(g, r, 1), epoch, m.side);
      CU_FATAL(cudaMemsetAsync(m.delta[k], 0, g.padded * 8, m.side));
      CU_FATAL(cudaGetLastError());
    }
  } else {
    NCCL_FATAL(api, api->GroupStart());
    for (int r = 0; r < g.nranks; ++r) {
      GroupMember& m = g.m[r];
      if (m.dev < 0) continue;
      DeviceGuard guard(m.dev);
      NCCL_FATAL(api, api->ReduceScatter(m.delta[k], m.tmp, g.chunk, kNcclDouble, kNcclSum, m.comm,
                                         m.side));
    }
    NCCL_FATAL(api, api->GroupEnd());
    for (int r = 0; r < g.nranks; ++r) {
      GroupMember& m = g.m[r];
      if (m.dev < 0) continue;
      DeviceGuard guard(m.dev);
      DeviceCtx& c = ctx_on(m.dev);
      c.launches += launch_fold_plain(m.owned, m.tmp, g.chunk, m.side);
      // the send buffer is free as soon as the collective has completed on this stream
      CU_FATAL(cudaMemsetAsync(m.delta[k], 0, g.padded * 8, m.side));
    }
  }
  for (int r = 0; r < g.nranks; ++r) {
    GroupMember& m = g.m[r];
    if (m.dev < 0) continue;
    DeviceGuard guard(m.dev);
    CU_FATAL(cudaEventRecord(m.ev_zeroed[k], m.side));
    m.zeroed_recorded[k] = true;
  }
  g.cur_k = (k + 1) % kDeltaBuffers;
  g.steps_deposited = 0;
  g.dirty = true;
}

void group_check_fault(TallyGroup& g) {
  for (int r = 0; r < g.nranks; ++r) {
    GroupMember& m = g.m[r];
    if (m.dev < 0) continue;
    DeviceGuard guard(m.dev);
    SyncBlock sb;
    CU_FATAL(cudaMemcpy(&sb, m.sync, sizeof(SyncBlock), cudaMemcpyDeviceToHost));
    if (sb.fault)
      terminate("tally collective: rank %d waited more than %llu s for a peer (every rank must "
                "run the same timesteps and tally syncs)", r, kWaitTimeoutNs / 1000000000ull);
  }
}

// Brings the caller-visible tally up to date: target[i] += owned slices, owned = 0
// (an all-gather fused with the accumulation). Synchronous. In a multi-process group it is a
// collective: every rank must call it the same number of times.
void group_flush(TallyGroup& g) {
  if (!g.dirty || !g.target) return;
  group_reduce(g, false);  // whatever has been deposited since the last reduction
  const NcclApi* api = g.collective ? nullptr : nccl_api(nullptr);
  const unsigned long long fe = ++g.flush_epoch;
  const int primary = g.mp ? g.mp_rank : 0;
  // everything deposited so far must be in the owned slices
  for (int r = 0; r < g.nranks; ++r) {
    GroupMember& m = g.m[r];
    if (m.dev < 0) continue;
    DeviceGuard guard(m.dev);
    if (g.mp && g.collective) ctx_on(m.dev).launches += launch_signal(m.sync, 1, fe, m.side);
    CU_FATAL(cudaStreamSynchronize(m.side));
  }
  if (g.collective) {
    GroupMember& m = g.m[primary];
    DeviceGuard guard(m.dev);
    DeviceCtx& c = ctx_on(m.dev);
    if (g.mp) c.launches += launch_wait_flags(wait_list(g, primary, 2), fe, m.side);
    c.launches += launch_gather_owned(group_view(g, primary, 0, true), g.target, g.mp ? fe : 0,
                                      m.side);
    if (g.mp) {
      c.launches += launch_wait_flags(wait_list(g, primary, 3), fe, m.side);
      CU_FATAL(cudaMemsetAsync(m.owned, 0, g.chunk * 8, m.side));
      CU_FATAL(cudaStreamSynchronize(m.side));
    } else {
      CU_FATAL(cudaStreamSynchronize(m.side));
      for (int r = 0; r < g.nranks; ++r) {
        DeviceGuard gr(g.m[r].dev);
        CU_FATAL(cudaMemsetAsync(g.m[r].owned, 0, g.chunk * 8, g.m[r].side));
        CU_FATAL(cudaStreamSynchronize(g.m[r].side));
      }
    }
  } else {
    NCCL_FATAL(api, api->GroupStart());
    for (int r = 0; r < g.nranks; ++r) {
      GroupMember& m = g.m[r];
      if (m.dev < 0) continue;
      DeviceGuard guard(m.dev);
      NCCL_FATAL(api, api->AllGather(m.owned, m.gathered, g.chunk, kNcclDouble, m.comm, m.side));
    }
    NCCL_FATAL(api, api->GroupEnd());
    for (int r = 0; r < g.nranks; ++r) {
      GroupMember& m = g.m[r];
      if (m.dev < 0) continue;
      DeviceGuard guard(m.dev);
      if (r == primary) ctx_on(m.dev).launches += launch_fold_plain(g.target, m.gathered, g.ncells, m.side);
      CU_FATAL(cudaMemsetAsync(m.owned, 0, g.chunk * 8, m.side));
      CU_FATAL(cudaStreamSynchronize(m.side));
    }
  }
  g.dirty = false;
  group_check_fault(g);
}

// Any library-mediated look at memory that a group's unflushed contributions belong to
// flushes first (validate, copy_buffer, the nb200_memcpy / memset helpers).
void flush_groups_touching(const void* ptr, size_t bytes) {
  auto touches = [ptr, bytes](const TallyBatches& tb) {
    if (!tb.dirty || !tb.target) return false;
    const char* lo = (const char*)tb.target;
    const char* hi = lo + tb.ncells * 8;
    const char* p = (const char*)ptr;
    return p < hi && p + bytes > lo;
  };
  for (Bank* b : g_batched)
    if (touches(b->batches)) batches_flush(b, b->batches);
  for (Bank* b : g_flux)
    if (touches(b->flux_batches)) batches_flush(b, b->flux_batches);
  for (TallyGroup* g : g_groups) {
    if (!g->dirty || !g->target) continue;
    const char* lo = (const char*)g->target;
    const char* hi = lo + g->ncells * 8;
    const char* p = (const char*)ptr;
    if (p < hi && p + bytes > lo) group_flush(*g);
  }
}

// Replica of a read-only input that lives on `primary_dev`, for shard sh on device c (current).
const double* replica_of(DeviceCtx& c, Shard& sh, int primary_dev, const double* src,
                         size_t count) {
  if (c.device == primary_dev || !src) return src;
  const size_t bytes = count * sizeof(double);
  for (auto& r : sh.replicas)
    if (r.src == src && r.bytes == bytes) {
      if (r.generation != g_replica_generation) {
        CU_FATAL(cudaMemcpyPeerAsync(r.copy, c.device, src, primary_dev, bytes, c.stream));
        r.generation = g_replica_generation;
      }
      return (const double*)r.copy;
    }
  void* copy = nullptr;
  for (auto& r : sh.replicas)  // a buffer of this size reserved when the bank was created?
    if (!r.src && r.bytes == bytes) {
      copy = r.copy;
      r = sh.replicas.back();
      sh.replicas.pop_back();
      break;
    }
  if (!copy) CU_FATAL(cudaMalloc(&copy, bytes ? bytes : 8));
  // the primary's uploads went through its own stream: make sure they have landed
  {
    DeviceGuard guard(primary_dev);
    CU_FATAL(cudaStreamSynchronize(ctx_on(primary_dev).stream));
  }
  CU_FATAL(cudaMemcpyPeerAsync(copy, c.device, src, primary_dev, bytes, c.stream));
  sh.replicas.push_back({src, bytes, copy, g_replica_generation});
  return (const double*)copy;
}

// --------------------------------------------------------------------- timestep pipeline --
void finish_oldest(Bank* bank, uint64_t* facet_events, uint64_t* collision_events);

// First half of a timestep: everything is enqueued, nothing is waited for.
void enqueue_step(Bank* bank, const StepRequest& rq) {
  if ((int)bank->pending.size() >= kMaxPending)
    terminate("solve_transport_2d: %d timesteps of this bank are enqueued and not collected "
              "(defer_finish=1): call nb200_solve_finish", kMaxPending);
  const size_t ncells = (size_t)rq.nx * rq.ny;
  TallyGroup* group = nullptr;
  if (!single_shard(bank)) {
    if (bank->group && bank->group->ncells != ncells) {  // another mesh: start over
      group_flush(*bank->group);
      group_free(bank->group);
      bank->group = nullptr;
    }
    if (!bank->group) bank->group = group_create_local(bank, ncells);
    group = bank->group;
  } else if (g_mp && g_mp->m[g_mp->mp_rank].dev == bank->shards[0].dev) {
    group = g_mp;
    if (group->ncells != ncells)
      terminate("solve_transport_2d: the multi-process group was created for %zu cells, the "
                "mesh has %zu", group->ncells, ncells);
  }
  // In a group every rank deposits into a private buffer; the buffers are reduce-scattered into
  // the owned slices every `reduce_every` timesteps, or - the default - only when somebody looks
  // at the tally: nothing on this path reads the tally between timesteps (main.c touches it in
  // validate and in VisIt dumps only), and a collective that is not run costs nothing.
  unsigned long long epoch = 0;
  int k = 0;
  bool closes = false;
  if (group) {
    if (group->target != rq.tally) {  // a different caller tally: settle the old one first
      group_flush(*group);
      group->target = rq.tally;
      group->target_dev = bank->primary_dev;
    }
    k = group->cur_k;
    closes = group->reduce_every > 0 && group->steps_deposited + 1 >= group->reduce_every;
    epoch = group->epoch + 1;
  }
  if (bank->batches.B > 0) batches_bind(bank, rq);
  if (bank->flux) flux_check(bank, rq, group != nullptr);
  PendingStep ps;
  ps.pipeline = opt_of(bank, &Options::pipeline) != 0;
  ps.print = opt_of(bank, &Options::print) != 0;
  ps.master_key = rq.master_key;
  uint64_t launches0 = 0;
  for (const Shard& sh : bank->shards) launches0 += ctx_on(sh.dev).launches;
  ps.launches0 = launches0;
  for (size_t si = 0; si < bank->shards.size(); ++si) {
    Shard& sh = bank->shards[si];
    DeviceGuard guard(sh.dev);
    DeviceCtx& c = ctx_on(sh.dev);
    const int slot = take_slot(c);
    ps.slot[si] = slot;
    ShardIO io;
    const int pd = bank->primary_dev;
    io.density = replica_of(c, sh, pd, rq.density, ncells);
    io.edgex = replica_of(c, sh, pd, rq.edgex, (size_t)rq.nx + 1);
    io.edgey = replica_of(c, sh, pd, rq.edgey, (size_t)rq.ny + 1);
    io.s_keys = replica_of(c, sh, pd, rq.s_keys, (size_t)rq.s_n);
    io.s_vals = replica_of(c, sh, pd, rq.s_vals, (size_t)rq.s_n);
    io.a_keys = replica_of(c, sh, pd, rq.a_keys, (size_t)rq.a_n);
    io.a_vals = replica_of(c, sh, pd, rq.a_vals, (size_t)rq.a_n);
    io.tally = rq.tally;
    io.batches = BatchArgs{bank->batches.slab, bank->batches.B, bank->n};
    io.flux = bank->flux_batches.B > 0 ? bank->flux_batches.slab : bank->flux;
    // per-particle counters live on the primary GPU, indexed in injection order: a secondary
    // shard reaches its part of them through peer access (one 8-byte update per particle-step)
    const bool counters_ok = sh.dev == pd || (group && group->collective);
    io.r0 = rq.r0 && counters_ok ? rq.r0 + sh.first : nullptr;
    io.r1 = rq.r1 && counters_ok ? rq.r1 + sh.first : nullptr;
    io.r2 = rq.r2 && counters_ok ? rq.r2 + sh.first : nullptr;
    SyncBlock* sync = nullptr;
    if (group) {
      const int rank = group->mp ? group->mp_rank : (int)si;
      GroupMember& m = group->m[rank];
      io.tally = m.delta[k];
      if (group->collective && closes) sync = m.sync;  // this timestep's publish raises `ready`
      // the buffer was cleared behind its last reduction, on the side stream
      if (m.zeroed_recorded[k]) CU_FATAL(cudaStreamWaitEvent(c.stream, m.ev_zeroed[k], 0));
      enqueue_shard_step(c, bank, sh, rq, io, slot, sync, epoch);
      CU_FATAL(cudaEventRecord(m.ev_hist[k], c.stream));
    } else {
      enqueue_shard_step(c, bank, sh, rq, io, slot, nullptr, 0);
    }
  }
  if (bank->batches.B > 0) bank->batches.dirty = true;
  if (bank->flux_batches.B > 0) bank->flux_batches.dirty = bank->flux_batches.deposited = true;
  if (group) {
    group->steps_deposited++;
    group->dirty = true;
    if (closes) group_reduce(*group, true);
  }
  bank->pending.push_back(ps);
  g_last_deferred = bank;
}

// Second half of a timestep: waits for the streams, checks the device-side faults, updates
// the live-prefix bounds and hands the counts to the caller (omp3/neutral.c:202-205).
void finish_oldest(Bank* bank, uint64_t* facet_events, uint64_t* collision_events) {
  if (bank->pending.empty()) return;
  const PendingStep ps = bank->pending.front();
  bank->pending.pop_front();
  uint64_t tot[kTotCount] = {0};
  uint64_t launches1 = 0;
  double hist_ms = 0.0, sort_ms = 0.0;
  for (size_t si = 0; si < bank->shards.size(); ++si) {
    Shard& sh = bank->shards[si];
    DeviceGuard guard(sh.dev);
    DeviceCtx& c = ctx_on(sh.dev);
    const int slot = ps.slot[si];
    // wait for THIS step's totals only: later timesteps may already be queued behind it
    CU_FATAL(cudaEventSynchronize(c.ev_pub[slot]));
    const volatile unsigned long long* h = c.h_totals + (size_t)slot * kTotCount;
    if (h[kTotFault])
      terminate("solve_transport_2d: a cross-section table's energy grid is not strictly "
                "increasing (omp3/neutral.c:506-511 assumes it is)");
    if (h[kTotGroupFault])
      terminate("solve_transport_2d: the tally collective timed out waiting for a peer GPU");
    // The sort compacted every particle that was dead at the start of this step behind the
    // live prefix; particles that died DURING the step still sit inside the prefix (the next
    // sort moves them out), so the prefix to visit next is this step's live count.
    if (ps.pipeline) sh.n_upper = std::min(sh.n_upper, (int)h[kTotProcessed]);
    for (int t = 0; t <= kTotDeaths; ++t) tot[t] += h[t];
    float ms = 0.0f;
    CU_FATAL(cudaEventElapsedTime(&ms, c.ev_mid[slot], c.ev_end[slot]));
    hist_ms = std::max(hist_ms, (double)ms);
    CU_FATAL(cudaEventElapsedTime(&ms, c.ev_begin[slot], c.ev_mid[slot]));
    sort_ms = std::max(sort_ms, (double)ms);
    memset((void*)(c.h_totals + (size_t)slot * kTotCount), 0, sizeof(unsigned long long) * kTotCount);
    c.slot_busy[slot] = false;
    c.pending_steps--;
    launches1 += c.launches;
  }
  for (int t = 0; t <= kTotDeaths; ++t) g_last_stats[t] = tot[t];
  g_last_stats[5] = launches1 - ps.launches0;
  g_last_stats[6] = (uint64_t)(hist_ms * 1.0e6);  // history kernel, ns on the stream (max over GPUs)
  g_last_stats[7] = (uint64_t)(sort_ms * 1.0e6);  // sort phase, ns
  if (g_step_log.size() < 100000)
    g_step_log.push_back({ps.master_key, tot[kTotFacets], tot[kTotCollisions], tot[kTotProcessed],
                          tot[kTotCensus], tot[kTotDeaths], g_last_stats[6], g_last_stats[7],
                          (int)bank->shards.size()});
  if (facet_events) *facet_events += tot[kTotFacets];            // omp3/neutral.c:202
  if (collision_events) *collision_events += tot[kTotCollisions];  // omp3/neutral.c:203
  if (ps.print) printf("Particles  %llu\n", (unsigned long long)tot[kTotProcessed]);  // :205
  if (bank->pending.empty()) refresh_mirror(bank);
}

void finish_all(Bank* bank) {
  while (!bank->pending.empty()) finish_oldest(bank, nullptr, nullptr);
}

void check_boundary_args(const char* who, int nx, int ny, int global_nx, int global_ny,
                         int pad, int x_off, int y_off) {
  if (pad != 0 || x_off != 0 || y_off != 0 || nx != global_nx || ny != global_ny) {
    terminate("%s: only the single-rank mesh of main.c:34,42-43 is supported "
              "(pad=%d x_off=%d y_off=%d nx=%d/%d ny=%d/%d)",
              who, pad, x_off, y_off, nx, global_nx, ny, global_ny);
  }
}

// problems/neutral.tests lookup: "<params_filename> result=<value>"
bool find_expected(const char* tests_file, const char* key, double* value) {
  FILE* fp = fopen(tests_file, "r");
  if (!fp) return false;
  char line[4096];
  bool found = false;
  while (fgets(line, sizeof(line), fp)) {
    char name[2048];
    int off = 0;
    if (sscanf(line, "%2047s%n", name, &off) != 1 || name[0] == '#') continue;
    if (strcmp(name, key) != 0) continue;
    const char* eq = strchr(line + off, '=');
    if (!eq) continue;
    *value = strtod(eq + 1, nullptr);
    found = true;
    break;
  }
  fclose(fp);
  return found;
}

__global__ void k_partial_sums(const double* __restrict__ v, size_t n, double* partial) {
  double s = 0.0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    s += v[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __shared__ double warp_part[32];
  if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = threadIdx.x < (blockDim.x >> 5) ? warp_part[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
  }
}

double device_sum(DeviceCtx& c, const double* v, size_t n) {
  const int blocks = 592, threads = 256;
  double* d_partial = nullptr;
  CU_FATAL(cudaMalloc(&d_partial, sizeof(double) * blocks));
  k_partial_sums<<<blocks, threads, 0, c.stream>>>(v, n, d_partial);
  c.launches++;
  std::vector<double> h(blocks);
  CU_FATAL(cudaMemcpyAsync(h.data(), d_partial, sizeof(double) * blocks,
                           cudaMemcpyDeviceToHost, c.stream));
  CU_FATAL(cudaStreamSynchronize(c.stream));
  cudaFree(d_partial);
  double s = 0.0;
  for (double x : h) s += x;
  return s;
}

// The machine-readable side of `validate` (SURVEY.md 8f 1): written when NB200_RESULTS_JSON
// names a file. Same verdict as the printed lines, plus what the library saw of the run.
// `batches` > 0: the tally came from a bank with tally batches, whose total has relative error
// `total_relerr`.
void write_results_json(const char* path, const char* deck, int nx, int ny, double total,
                        bool have_expected, double expected, const char* verdict, int batches,
                        double total_relerr) {
  FILE* fp = fopen(path, "w");
  if (!fp) {
    fprintf(stderr, "neutral_b200: cannot write %s\n", path);
    return;
  }
  cudaDeviceProp prop{};
  int dev = 0;
  cudaGetDevice(&dev);
  cudaGetDeviceProperties(&prop, dev);
  fprintf(fp, "{\"deck\": \"%s\", \"nx\": %d, \"ny\": %d, \"device\": \"%s\",\n", deck, nx, ny,
          prop.name);
  fprintf(fp, " \"tally_total\": %.17e, ", total);
  if (batches > 0)
    fprintf(fp, "\"tally_batches\": %d, \"tally_total_relative_error\": %.17e, ", batches,
            total_relerr);
  if (have_expected)
    fprintf(fp, "\"expected\": %.17e, \"relative_error\": %.6e, \"tolerance\": 1e-3, ", expected,
            fabs(expected - total) / (fabs(expected) > 0.0 ? fabs(expected) : 1.0));
  else
    fprintf(fp, "\"expected\": null, ");
  fprintf(fp, "\"verdict\": \"%s\",\n \"steps\": [", verdict);
  for (size_t i = 0; i < g_step_log.size(); ++i) {
    const StepLog& s = g_step_log[i];
    fprintf(fp, "%s\n  {\"facets\": %llu, \"collisions\": %llu, \"particles\": %llu, \"census\": %llu, "
                "\"deaths\": %llu, \"history_kernel_ns\": %llu, \"sort_phase_ns\": %llu, \"gpus\": %d}",
            i ? "," : "", (unsigned long long)s.facets, (unsigned long long)s.collisions,
            (unsigned long long)s.processed, (unsigned long long)s.census,
            (unsigned long long)s.deaths, (unsigned long long)s.history_ns,
            (unsigned long long)s.sort_ns, s.ngpus);
  }
  fprintf(fp, "\n ]}\n");
  fclose(fp);
}

}  // namespace

// ======================================================================================
// 1. plugin boundary, device-resident flavour
// ======================================================================================
extern "C" void solve_transport_2d(
    const int nx, const int ny, const int global_nx, const int global_ny,
    const uint64_t master_key, const int pad, const int x_off, const int y_off,
    const double dt, const int ntotal_particles, int* nlocal_particles,
    const int* neighbours, nb200_particle_soa* particles, const double* density,
    const double* edgex, const double* edgey, const double* edgedx, const double* edgedy,
    nb200_cross_section* cs_scatter_table, nb200_cross_section* cs_absorb_table,
    double* energy_deposition_tally, uint64_t* reduce_array0, uint64_t* reduce_array1,
    uint64_t* reduce_array2, uint64_t* facet_events, uint64_t* collision_events) {
  (void)neighbours; (void)edgedx; (void)edgedy;
  if (!(*nlocal_particles)) {  // omp3/neutral.c:30-33
    printf("Out of particles\n");
    return;
  }
  ctx_required();
  check_boundary_args("solve_transport_2d", nx, ny, global_nx, global_ny, pad, x_off, y_off);
  Bank* bank = bank_of(particles);
  if (!bank) terminate("solve_transport_2d: `particles` is not a bank created by this "
                       "kernel set's inject_particles / nb200_bank_create");
  const bool defer = opt_of(bank, &Options::defer_finish) != 0;
  if (!defer && !bank->pending.empty())
    terminate("solve_transport_2d: earlier timesteps of this bank were enqueued with "
              "defer_finish=1 and nb200_solve_finish has not collected them");
  StepRequest rq;
  rq.nx = nx;
  rq.ny = ny;
  rq.master_key = master_key;
  rq.dt = dt;
  rq.ntotal = ntotal_particles;
  rq.density = density;
  rq.edgex = edgex;
  rq.edgey = edgey;
  rq.s_keys = cs_scatter_table->keys;
  rq.s_vals = cs_scatter_table->values;
  rq.s_n = cs_scatter_table->nentries;
  rq.a_keys = cs_absorb_table->keys;
  rq.a_vals = cs_absorb_table->values;
  rq.a_n = cs_absorb_table->nentries;
  rq.tally = energy_deposition_tally;
  rq.r0 = reduce_array0;
  rq.r1 = reduce_array1;
  rq.r2 = reduce_array2;
  enqueue_step(bank, rq);
  // "defer_finish": the caller keeps the GPU fed (the next timestep, its own host work) and
  // collects the counts later with nb200_solve_finish
  if (!defer) finish_oldest(bank, facet_events, collision_events);
}

extern "C" size_t inject_particles(
    const int nparticles, const int global_nx, const int local_nx, const int local_ny,
    const int pad, const double local_particle_left_off,
    const double local_particle_bottom_off, const double local_particle_width,
    const double local_particle_height, const int x_off, const int y_off, const double dt,
    const double* edgex, const double* edgey, const double initial_energy,
    nb200_particle_soa** particles) {
  DeviceCtx& primary = ctx_required();
  check_boundary_args("inject_particles", local_nx, local_ny, global_nx, local_ny, pad, x_off,
                      y_off);
  const int first = g_shard_count >= 0 ? g_shard_first : 0;
  const int count = g_shard_count >= 0 ? g_shard_count : nparticles;
  if (first < 0 || first + count > nparticles)
    terminate("inject_particles: shard [%d, %d) outside [0, %d)", first, first + count,
              nparticles);

  if (const char* why = why_no_batches(g_opt.tally_batches, count, (uint64_t)first, g_opt.ngpus))
    terminate("inject_particles: %s", why);
  size_t bytes = 0;
  Bank* bank = new_bank(count, (uint64_t)first, g_opt.ngpus, g_opt.headroom_pct,
                        g_opt.host_mirror != 0, &bytes);
  batches_attach(bank, g_opt.tally_batches);
  for (Shard& sh : bank->shards) {  // per-mesh scratch of every GPU involved, ahead of timestep 1
    DeviceGuard guard(sh.dev);
    int shift = g_opt.tile_shift, tx = 1, nt = 1;
    const long long nbins = sort_key_space(local_nx, local_ny, g_opt.length_bins, &shift, &tx, &nt);
    reserve_mesh_scratch(ctx_on(sh.dev), local_nx, local_ny, nbins);
  }
  if (g_opt.device_inject) {
    // The bank is generated where it lives: no host loop, no 80-byte-per-particle upload.
    for (Shard& sh : bank->shards) {
      DeviceGuard guard(sh.dev);
      DeviceCtx& c = ctx_on(sh.dev);
      InjectArgs ia{replica_of(c, sh, primary.device, edgex, (size_t)local_nx + 1),
                    replica_of(c, sh, primary.device, edgey, (size_t)local_ny + 1), local_nx,
                    local_ny, local_particle_left_off, local_particle_bottom_off,
                    local_particle_width, local_particle_height, dt, initial_energy};
      c.launches += launch_inject(sh.cur, sh.n, sh.pid0, ia, c.d_sct, c.stream);
      CU_FATAL(cudaGetLastError());
    }
    for (Shard& sh : bank->shards) {
      DeviceGuard guard(sh.dev);
      CU_FATAL(cudaStreamSynchronize(ctx_on(sh.dev).stream));
    }
    // the tally group of a sharded bank (slabs, peer mappings) and the buffer its secondary GPUs
    // will hold their replica of the density mesh in: built here, outside the timesteps
    if (!single_shard(bank)) {
      bank->group = group_create_local(bank, (size_t)local_nx * (size_t)local_ny);
      for (Shard& sh : bank->shards) {
        if (sh.dev == bank->primary_dev) continue;
        DeviceGuard guard(sh.dev);
        const size_t bytes = sizeof(double) * (size_t)local_nx * (size_t)local_ny;
        void* reserved = nullptr;
        CU_FATAL(cudaMalloc(&reserved, bytes));
        sh.replicas.push_back({nullptr, bytes, reserved, 0});
      }
    }
    refresh_mirror(bank);
    *particles = handle_of(bank);
    return bytes;
  }

  // Host flavour ("device_inject" = 0): the same arithmetic with the host's libm.
  // The mesh edges live in kernel-set (device) memory.
  std::vector<double> ex(local_nx + 1), ey(local_ny + 1);
  CU_FATAL(cudaMemcpy(ex.data(), edgex, sizeof(double) * (local_nx + 1),
                      cudaMemcpyDeviceToHost));
  CU_FATAL(cudaMemcpy(ey.data(), edgey, sizeof(double) * (local_ny + 1),
                      cudaMemcpyDeviceToHost));

  const size_t n = (size_t)std::max(count, 1);
  std::vector<double> x(n), y(n), ox(n), oy(n), en(n), wt(n), dtc(n), mfp(n);
  std::vector<int> cx(n), cy(n), dead(n);

  // First cell whose half-open interval holds v; 0 when there is none - what the
  // reference's linear scan returns (omp3/neutral.c:590-603), found by bisection.
  auto locate = [](const std::vector<double>& edge, int ncells, double v) {
    int lo = 0, hi = ncells;
    if (!(v >= edge[0])) return 0;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (v >= edge[mid]) lo = mid; else hi = mid;
    }
    return (v >= edge[lo] && v < edge[lo + 1]) ? lo : 0;
  };

#pragma omp parallel for schedule(static)
  for (int s = 0; s < count; ++s) {
    const uint64_t kk = (uint64_t)(first + s);
    double r0, r1;
    random_pair(kk, 0, 0, r0, r1);  // omp3/neutral.c:581
    x[s] = local_particle_left_off + r0 * local_particle_width;
    y[s] = local_particle_bottom_off + r1 * local_particle_height;
    cx[s] = locate(ex, local_nx, x[s]);
    cy[s] = locate(ey, local_ny, y[s]);
    random_pair(kk, 0, 1, r0, r1);  // omp3/neutral.c:611
    const double theta = 2.0 * M_PI * r0;
    ox[s] = cos(theta);
    oy[s] = sin(theta);
    en[s] = initial_energy;
    wt[s] = 1.0;
    dtc[s] = dt;
    mfp[s] = 0.0;
    dead[s] = 0;
  }

  SoaView host{x.data(), y.data(), ox.data(), oy.data(), en.data(), wt.data(), dtc.data(),
               mfp.data(), cx.data(), cy.data(), dead.data()};
  upload_host_soa(bank, host);
  refresh_mirror(bank);
  *particles = handle_of(bank);
  return bytes;
}

extern "C" void validate(const int nx, const int ny, const char* params_filename,
                         const int rank, double* energy_tally) {
  DeviceCtx& c = ctx_required();
  flush_groups_touching(energy_tally, sizeof(double) * (size_t)nx * ny);
  const double total = device_sum(c, energy_tally, (size_t)nx * ny);
  if (rank != 0) return;
  const char* json = getenv("NB200_RESULTS_JSON");
  int batches = 0;
  double total_relerr = 0.0;
  if (json && *json) {
    if (Bank* b = batched_bank_of_tally(energy_tally)) {
      batches = b->batches.B;
      total_relerr = batches_total_relerr(b, b->batches);
    }
  }
  printf("\nFinal global_energy_tally %.15e\n", total);
  double expected = 0.0;
  if (!find_expected("problems/neutral.tests", params_filename, &expected)) {
    printf("Warning. Test entry was not found, could NOT validate.\n");
    if (json && *json)
      write_results_json(json, params_filename, nx, ny, total, false, 0.0, "NOT_VALIDATED",
                         batches, total_relerr);
    return;
  }
  printf("Expected %.12e, result was %.12e.\n", expected, total);
  // arch's within_tolerance is not in the reference tree; archlite's (and this) reading of it
  // is the relative difference against VALIDATE_TOLERANCE (neutral_data.h:27)
  const double scale = fabs(expected) > 0.0 ? fabs(expected) : 1.0;
  const bool pass = fabs(expected - total) / scale < 1.0e-3;
  printf(pass ? "PASSED validation.\n" : "FAILED validation.\n");
  if (json && *json)
    write_results_json(json, params_filename, nx, ny, total, true, expected,
                       pass ? "PASSED" : "FAILED", batches, total_relerr);
}

// ======================================================================================
// 2. allocation layer
// ======================================================================================
extern "C" size_t allocate_data(double** buf, size_t len) { return device_zalloc(ctx_required(), buf, len); }
extern "C" size_t allocate_float_data(float** buf, size_t len) { return device_zalloc(ctx_required(), buf, len); }
extern "C" size_t allocate_int_data(int** buf, size_t len) { return device_zalloc(ctx_required(), buf, len); }
extern "C" size_t allocate_uint64_data(uint64_t** buf, size_t len) {
  return device_zalloc(ctx_required(), buf, len);
}

extern "C" void allocate_host_data(double** buf, size_t len) {
  ctx_required();
  CU_FATAL(cudaMallocHost((void**)buf, sizeof(double) * (len ? len : 1)));
  memset(*buf, 0, sizeof(double) * len);
}

extern "C" void allocate_host_float_data(float** buf, size_t len) {
  ctx_required();
  CU_FATAL(cudaMallocHost((void**)buf, sizeof(float) * (len ? len : 1)));
  memset(*buf, 0, sizeof(float) * len);
}

extern "C" void deallocate_data(double* buf) {
  // a tally that a sharded run still owes contributions to is completed before it goes away,
  // and no group keeps pointing at freed memory
  if (buf) {
    flux_detach_array(buf);
    flush_groups_touching(buf, sizeof(double));
    for (TallyGroup* g : g_groups)
      if (g->target == buf) g->target = nullptr;
    for (Bank* b : g_batched)
      if (b->batches.target == buf) b->batches.target = nullptr;
  }
  cudaFree(buf);
}
extern "C" void deallocate_host_data(double* buf) { cudaFreeHost(buf); }

extern "C" void copy_buffer(const size_t len, double** src, double** dst, int send) {
  DeviceCtx& c = ctx_required();
  if (!send) flush_groups_touching(*src, sizeof(double) * len);
  // cudaMemcpyDefault: the direction follows from the pointers, so a RECV of a buffer that
  // happens to be host memory (main.c:169-200 hands its own malloc to the VisIt writer) works
  (void)send;
  CU_FATAL(cudaMemcpyAsync(*dst, *src, sizeof(double) * len, cudaMemcpyDefault, c.stream));
  CU_FATAL(cudaStreamSynchronize(c.stream));
}

extern "C" void move_host_buffer_to_device(const size_t len, double** src, double** dst) {
  DeviceCtx& c = ctx_required();
  device_zalloc(c, dst, len);
  CU_FATAL(cudaMemcpyAsync(*dst, *src, sizeof(double) * len, cudaMemcpyHostToDevice, c.stream));
  CU_FATAL(cudaStreamSynchronize(c.stream));
  cudaPointerAttributes attr{};
  if (cudaPointerGetAttributes(&attr, *src) == cudaSuccess && attr.type == cudaMemoryTypeHost) {
    cudaFreeHost(*src);
  } else {
    (void)cudaGetLastError();
    free(*src);
  }
  *src = nullptr;
}

extern "C" void initialise_devices(int rank) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0)
    terminate("no CUDA device available: the b200 kernel set has no CPU fallback");
  CU_FATAL(cudaSetDevice(rank % count));
  ctx_required();
  cudaDeviceProp prop{};
  CU_FATAL(cudaGetDeviceProperties(&prop, rank % count));
  printf("Rank %d using GPU %d: %s (sm_%d%d, %d SMs, %.0f GB)\n", rank, rank % count, prop.name,
         prop.major, prop.minor, prop.multiProcessorCount,
         (double)prop.totalGlobalMem / (1024.0 * 1024.0 * 1024.0));
  if (g_opt.ngpus > 1)
    printf("Particle bank sharded over %d GPUs (NB200_NGPUS), tally combined by the %s\n",
           g_opt.ngpus, g_opt.collective ? "library's peer-memory reduce-scatter kernel"
                                         : "NCCL reduce-scatter");
}

// ======================================================================================
// 3. host-buffer flavour
// ======================================================================================
extern "C" void nb200_solve_transport_2d_host(
    const int nx, const int ny, const int global_nx, const int global_ny,
    const uint64_t master_key, const int pad, const int x_off, const int y_off,
    const double dt, const int ntotal_particles, int* nlocal_particles,
    const int* neighbours, nb200_particle_aos* particles, const double* density,
    const double* edgex, const double* edgey, const double* edgedx, const double* edgedy,
    nb200_cross_section* cs_scatter_table, nb200_cross_section* cs_absorb_table,
    double* energy_deposition_tally, uint64_t* reduce_array0, uint64_t* reduce_array1,
    uint64_t* reduce_array2, uint64_t* facet_events, uint64_t* collision_events) {
  (void)neighbours; (void)edgedx; (void)edgedy;
  static_assert(sizeof(nb200_particle_aos) == 80, "AoS particle must be 80 bytes");
  const int n = *nlocal_particles;
  if (!n) {
    printf("Out of particles\n");
    return;
  }
  DeviceCtx& c = ctx_required();
  check_boundary_args("nb200_solve_transport_2d_host", nx, ny, global_nx, global_ny, pad,
                      x_off, y_off);
  const size_t ncells = (size_t)nx * ny;
  const int s_n = cs_scatter_table->nentries, a_n = cs_absorb_table->nentries;

  auto upload = [&](const void* host, size_t bytes) {
    void* d = nullptr;
    CU_FATAL(cudaMalloc(&d, bytes ? bytes : 1));
    CU_FATAL(cudaMemcpyAsync(d, host, bytes, cudaMemcpyHostToDevice, c.stream));
    return d;
  };
  double* d_density = (double*)upload(density, sizeof(double) * ncells);
  double* d_edgex = (double*)upload(edgex, sizeof(double) * (nx + 1));
  double* d_edgey = (double*)upload(edgey, sizeof(double) * (ny + 1));
  double* d_sk = (double*)upload(cs_scatter_table->keys, sizeof(double) * s_n);
  double* d_sv = (double*)upload(cs_scatter_table->values, sizeof(double) * s_n);
  double* d_ak = (double*)upload(cs_absorb_table->keys, sizeof(double) * a_n);
  double* d_av = (double*)upload(cs_absorb_table->values, sizeof(double) * a_n);
  double* d_tally = (double*)upload(energy_deposition_tally, sizeof(double) * ncells);
  void* d_aos = upload(particles, sizeof(nb200_particle_aos) * (size_t)n);
  uint64_t* d_r[3] = {nullptr, nullptr, nullptr};
  uint64_t* h_r[3] = {reduce_array0, reduce_array1, reduce_array2};
  for (int k = 0; k < 3; ++k)
    if (h_r[k]) d_r[k] = (uint64_t*)upload(h_r[k], sizeof(uint64_t) * (size_t)n);

  // fresh device addresses every call: the per-pointer scheduling hints must not go stale on
  // recycled addresses (they would still be harmless, but they would be worthless)
  c.table_cache.clear();
  c.mesh_cache.clear();
  Bank bank;
  bank.n = n;
  bank.pid0 = 0;
  bank.primary_dev = c.device;
  bank.overrides.push_back({option_index("defer_finish"), 0});  // the host flavour never defers
  Shard sh;
  sh.dev = c.device;
  sh.n = sh.capacity = sh.n_upper = n;
  bank_alloc(c, sh.cur, n);
  bank.shards.push_back(sh);
  c.launches += launch_import_aos(bank.shards[0].cur, d_aos, n, c.stream);
  StepRequest rq;
  rq.nx = nx; rq.ny = ny; rq.master_key = master_key; rq.dt = dt; rq.ntotal = ntotal_particles;
  rq.density = d_density; rq.edgex = d_edgex; rq.edgey = d_edgey;
  rq.s_keys = d_sk; rq.s_vals = d_sv; rq.s_n = s_n;
  rq.a_keys = d_ak; rq.a_vals = d_av; rq.a_n = a_n;
  rq.tally = d_tally; rq.r0 = d_r[0]; rq.r1 = d_r[1]; rq.r2 = d_r[2];
  Bank* const was_deferred = g_last_deferred;
  enqueue_step(&bank, rq);
  finish_oldest(&bank, facet_events, collision_events);
  g_last_deferred = was_deferred;
  Shard& s0 = bank.shards[0];
  c.launches += launch_export_aos(s0.cur, d_aos, n, c.stream);
  CU_FATAL(cudaMemcpyAsync(particles, d_aos, sizeof(nb200_particle_aos) * (size_t)n,
                           cudaMemcpyDeviceToHost, c.stream));
  CU_FATAL(cudaMemcpyAsync(energy_deposition_tally, d_tally, sizeof(double) * ncells,
                           cudaMemcpyDeviceToHost, c.stream));
  for (int k = 0; k < 3; ++k)
    if (h_r[k])
      CU_FATAL(cudaMemcpyAsync(h_r[k], d_r[k], sizeof(uint64_t) * (size_t)n,
                               cudaMemcpyDeviceToHost, c.stream));
  CU_FATAL(cudaStreamSynchronize(c.stream));
  bank_release(s0.cur);
  if (s0.has_alt) {
    bank_release(s0.alt);
    cudaFree(s0.keys);
  }
  void* to_free[] = {d_density, d_edgex, d_edgey, d_sk, d_sv, d_ak, d_av, d_tally, d_aos,
                     d_r[0], d_r[1], d_r[2]};
  for (void* p : to_free) cudaFree(p);
  c.table_cache.clear();
  c.mesh_cache.clear();
}

// ======================================================================================
// 4. extensions
// ======================================================================================
extern "C" int nb200_abi_version(void) { return NB200_ABI_VERSION; }
extern "C" const char* nb200_last_error(void) { return g_last_error.c_str(); }

extern "C" int nb200_device_count(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return count;
}

extern "C" int nb200_set_stream(void* cuda_stream) {
  CTX_OR_RETURN(c);
  if (c.pending_steps > 0) {
    set_error("nb200_set_stream: %d timestep(s) are still enqueued on the current stream; "
              "collect them with nb200_solve_finish first", c.pending_steps);
    return -4;
  }
  c.stream = (cudaStream_t)cuda_stream;
  return 0;
}

extern "C" int nb200_set_shard(int first, int count) {
  g_shard_first = first;
  g_shard_count = count;
  return 0;
}

// A bank operation that rewrites or releases the bank must not race a timestep in flight.
static int refuse_if_pending(Bank* bank, const char* who) {
  if (bank->pending.empty()) return 0;
  set_error("%s: %d timestep(s) of this bank are enqueued and not collected; call "
            "nb200_solve_finish first", who, (int)bank->pending.size());
  return -4;
}

extern "C" int nb200_bank_create(const nb200_particle_soa* host, int count, int pid_first,
                                 nb200_particle_soa** particles) {
  CTX_OR_RETURN(c);
  (void)c;
  if (!host || !particles || count < 0) {
    set_error("nb200_bank_create: bad arguments");
    return -3;
  }
  if (const char* why = why_no_batches(g_opt.tally_batches, count, (uint64_t)pid_first,
                                     g_opt.ngpus)) {
    set_error("nb200_bank_create: %s", why);
    return -3;
  }
  Bank* bank = new_bank(count, (uint64_t)pid_first, g_opt.ngpus, g_opt.headroom_pct,
                        g_opt.host_mirror != 0, nullptr);
  batches_attach(bank, g_opt.tally_batches);
  if (count > 0) upload_host_soa(bank, as_soa_view(*host));
  refresh_mirror(bank);
  *particles = handle_of(bank);
  return 0;
}

extern "C" int nb200_bank_upload(nb200_particle_soa* particles, const nb200_particle_soa* host) {
  CTX_OR_RETURN(c0);
  (void)c0;
  Bank* bank = bank_of(particles);
  if (!bank || !host) {
    set_error("nb200_bank_upload: not a bank handle");
    return -3;
  }
  if (int rc = refuse_if_pending(bank, "nb200_bank_upload")) return rc;
  for (Shard& sh : bank->shards) {
    DeviceGuard guard(sh.dev);
    DeviceCtx& c = ctx_on(sh.dev);
    ensure_export(c, sh);
    // The plain SoA view doubles as the staging area: H2D per field, then one repack kernel.
    const SoaView& s = sh.exported;
    const SoaView h = soa_offset(as_soa_view(*host), (size_t)sh.first);
    const size_t n = (size_t)sh.n;
    const double* hd[] = {h.x, h.y, h.omega_x, h.omega_y, h.energy, h.weight, h.dt_to_census,
                          h.mfp_to_collision};
    double* dd[] = {s.x, s.y, s.omega_x, s.omega_y, s.energy, s.weight, s.dt_to_census,
                    s.mfp_to_collision};
    for (int k = 0; k < 8; ++k)
      CU_TRY(cudaMemcpyAsync(dd[k], hd[k], sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
    const int* hi[] = {h.cellx, h.celly, h.dead};
    int* di[] = {s.cellx, s.celly, s.dead};
    for (int k = 0; k < 3; ++k)
      CU_TRY(cudaMemcpyAsync(di[k], hi[k], sizeof(int) * n, cudaMemcpyHostToDevice, c.stream));
    c.launches += launch_import_soa(sh.cur, s, sh.n, 0, c.stream);
    sh.n_upper = sh.n;
  }
  if (single_shard(bank) && !bank->mirror.present)
    set_views(bank, as_public(bank->shards[0].exported));
  return 0;
}

// The plain device SoA view behind the handle (allocated on first use). Together with
// nb200_bank_import / nb200_bank_export it lets a host move banks with its own asynchronous
// copies: fill the view, then import; export, then read the view. Single-GPU banks only.
extern "C" int nb200_bank_view(nb200_particle_soa* particles, nb200_particle_soa* view_out) {
  CTX_OR_RETURN(c0);
  (void)c0;
  Bank* bank = bank_of(particles);
  if (!bank || !view_out || !single_shard(bank)) {
    set_error("nb200_bank_view: not a (single-GPU) bank handle");
    return -3;
  }
  Shard& sh = bank->shards[0];
  DeviceGuard guard(sh.dev);
  ensure_export(ctx_on(sh.dev), sh);
  if (!bank->mirror.present) set_views(bank, as_public(sh.exported));
  *view_out = as_public(sh.exported);
  return 0;
}

// Rebuilds the bank from its plain SoA view (asynchronous on the library's stream).
extern "C" int nb200_bank_import(nb200_particle_soa* particles) {
  CTX_OR_RETURN(c0);
  (void)c0;
  Bank* bank = bank_of(particles);
  if (!bank || !single_shard(bank) || !bank->shards[0].has_export) {
    set_error("nb200_bank_import: not a (single-GPU) bank handle, or its view was never requested");
    return -3;
  }
  if (int rc = refuse_if_pending(bank, "nb200_bank_import")) return rc;
  Shard& sh = bank->shards[0];
  DeviceGuard guard(sh.dev);
  DeviceCtx& c = ctx_on(sh.dev);
  c.launches += launch_import_soa(sh.cur, sh.exported, sh.n, 0, c.stream);
  sh.n_upper = sh.n;
  return 0;
}

extern "C" int nb200_accumulate(double* dst_device, const double* src_device, size_t n) {
  CTX_OR_RETURN(c);
  c.launches += launch_accumulate(dst_device, src_device, n, c.stream);
  return 0;
}

extern "C" int nb200_accumulate_clear(double* dst_device, double* src_device, size_t n) {
  CTX_OR_RETURN(c);
  c.launches += launch_accumulate_clear(dst_device, src_device, n, c.stream);
  return 0;
}

extern "C" int nb200_accumulate_clear_async(double* dst_device, double* src_device, size_t n,
                                            void* cuda_stream) {
  CTX_OR_RETURN(c);
  c.launches += launch_accumulate_clear(dst_device, src_device, n, (cudaStream_t)cuda_stream);
  return 0;
}

extern "C" int nb200_bank_export(nb200_particle_soa* particles) {
  CTX_OR_RETURN(c0);
  (void)c0;
  Bank* bank = bank_of(particles);
  if (!bank || !single_shard(bank)) {
    set_error("nb200_bank_export: not a (single-GPU) bank handle");
    return -3;
  }
  if (int rc = refuse_if_pending(bank, "nb200_bank_export")) return rc;
  Shard& sh = bank->shards[0];
  DeviceGuard guard(sh.dev);
  DeviceCtx& c = ctx_on(sh.dev);
  ensure_export(c, sh);
  if (!bank->mirror.present) set_views(bank, as_public(sh.exported));
  c.launches += launch_export_soa(sh.cur, sh.exported, sh.n, c.stream);
  CU_TRY(cudaStreamSynchronize(c.stream));
  return 0;
}

extern "C" int nb200_bank_download(nb200_particle_soa* particles, nb200_particle_soa* host) {
  CTX_OR_RETURN(c0);
  (void)c0;
  Bank* bank = bank_of(particles);
  if (!bank || !host) {
    set_error("nb200_bank_download: not a bank handle");
    return -3;
  }
  if (int rc = refuse_if_pending(bank, "nb200_bank_download")) return rc;
  download_to_host(bank, as_soa_view(*host));
  return 0;
}

extern "C" int nb200_bank_copy(nb200_particle_soa* dst, nb200_particle_soa* src) {
  CTX_OR_RETURN(c0);
  (void)c0;
  Bank* d = bank_of(dst);
  Bank* s = bank_of(src);
  if (!d || !s || d->n != s->n || d->shards.size() != s->shards.size()) {
    set_error("nb200_bank_copy: handles must be banks of the same size and sharding");
    return -3;
  }
  if (int rc = refuse_if_pending(d, "nb200_bank_copy")) return rc;
  if (int rc = refuse_if_pending(s, "nb200_bank_copy")) return rc;
  for (size_t si = 0; si < d->shards.size(); ++si) {
    Shard& ds = d->shards[si];
    Shard& ss = s->shards[si];
    if (ds.dev != ss.dev || ds.n != ss.n) {
      set_error("nb200_bank_copy: shard %zu differs in device or size", si);
      return -3;
    }
    DeviceGuard guard(ds.dev);
    DeviceCtx& c = ctx_on(ds.dev);
    const size_t n = (size_t)ss.n;
    CU_TRY(cudaMemcpyAsync(ds.cur.pos, ss.cur.pos, sizeof(double2) * n, cudaMemcpyDeviceToDevice, c.stream));
    CU_TRY(cudaMemcpyAsync(ds.cur.dir, ss.cur.dir, sizeof(double2) * n, cudaMemcpyDeviceToDevice, c.stream));
    CU_TRY(cudaMemcpyAsync(ds.cur.ew, ss.cur.ew, sizeof(double2) * n, cudaMemcpyDeviceToDevice, c.stream));
    CU_TRY(cudaMemcpyAsync(ds.cur.tm, ss.cur.tm, sizeof(double2) * n, cudaMemcpyDeviceToDevice, c.stream));
    CU_TRY(cudaMemcpyAsync(ds.cur.meta, ss.cur.meta, sizeof(int4) * n, cudaMemcpyDeviceToDevice, c.stream));
    ds.pid0 = ss.pid0;
    ds.n_upper = ss.n_upper;
  }
  d->pid0 = s->pid0;
  return 0;
}

extern "C" int nb200_bank_size(nb200_particle_soa* particles) {
  Bank* bank = bank_of(particles);
  return bank ? bank->n : -3;
}

extern "C" int nb200_bank_capacity(nb200_particle_soa* particles) {
  Bank* bank = bank_of(particles);
  if (!bank) return -3;
  long long cap = 0;
  for (const Shard& sh : bank->shards) cap += sh.capacity;
  return (int)std::min<long long>(cap, INT_MAX);
}

extern "C" int nb200_bank_gpus(nb200_particle_soa* particles) {
  Bank* bank = bank_of(particles);
  return bank ? (int)bank->shards.size() : -3;
}

// Appends `count` particles (host SoA arrays) into the bank's head-room: they become
// particles [n, n + count) in injection order, global index pid0 + n + i (single-GPU banks).
extern "C" int nb200_bank_append(nb200_particle_soa* particles, const nb200_particle_soa* host,
                                 int count) {
  CTX_OR_RETURN(c0);
  (void)c0;
  Bank* bank = bank_of(particles);
  if (!bank || !host || count < 0 || !single_shard(bank)) {
    set_error("nb200_bank_append: not a (single-GPU) bank handle");
    return -3;
  }
  if (int rc = refuse_if_pending(bank, "nb200_bank_append")) return rc;
  Shard& sh = bank->shards[0];
  if (bank->mirror.present) {
    set_error("nb200_bank_append: banks with a host mirror cannot grow");
    return -3;
  }
  if (bank->batches.B > 0) {
    set_error("nb200_bank_append: a bank with tally_batches cannot grow (its batches are ranges "
              "of the particles it was created with)");
    return -3;
  }
  if (sh.n + count > sh.capacity) {
    set_error("nb200_bank_append: %d particles do not fit the head-room (%d of %d slots used; "
              "option headroom_pct)", count, sh.n, sh.capacity);
    return -5;
  }
  if (count == 0) return 0;
  DeviceGuard guard(sh.dev);
  DeviceCtx& c = ctx_on(sh.dev);
  SoaView staging{};
  soa_alloc(c, staging, count);
  const SoaView h = as_soa_view(*host);
  const double* hd[] = {h.x, h.y, h.omega_x, h.omega_y, h.energy, h.weight, h.dt_to_census,
                        h.mfp_to_collision};
  double* dd[] = {staging.x, staging.y, staging.omega_x, staging.omega_y, staging.energy,
                  staging.weight, staging.dt_to_census, staging.mfp_to_collision};
  for (int k = 0; k < 8; ++k)
    CU_TRY(cudaMemcpyAsync(dd[k], hd[k], sizeof(double) * count, cudaMemcpyHostToDevice, c.stream));
  const int* hi[] = {h.cellx, h.celly, h.dead};
  int* di[] = {staging.cellx, staging.celly, staging.dead};
  for (int k = 0; k < 3; ++k)
    CU_TRY(cudaMemcpyAsync(di[k], hi[k], sizeof(int) * count, cudaMemcpyHostToDevice, c.stream));
  // the new records go behind the last slot, with the next origins
  BankView tail = sh.cur;
  tail.pos += sh.n; tail.dir += sh.n; tail.ew += sh.n; tail.tm += sh.n; tail.meta += sh.n;
  c.launches += launch_import_soa(tail, staging, count, sh.n, c.stream);
  CU_TRY(cudaStreamSynchronize(c.stream));
  soa_release(staging);
  sh.n += count;
  sh.n_upper = sh.n;  // the live prefix is unknown again: the next sort visits every slot
  bank->n += count;
  if (sh.has_export) {  // the plain view was sized for the old bank only if capacity == n
    // (it is allocated with `capacity` slots, so nothing to do)
  }
  return 0;
}

extern "C" int nb200_bank_free(nb200_particle_soa* particles) {
  Bank* bank = bank_of(particles);
  if (!bank) return -3;
  finish_all(bank);
  batches_release(bank, bank->batches);
  g_batched.erase(std::remove(g_batched.begin(), g_batched.end(), bank), g_batched.end());
  flux_attach(bank, nullptr, 0);
  if (bank->group) {
    group_flush(*bank->group);
    group_free(bank->group);
  }
  for (Shard& sh : bank->shards) {
    DeviceGuard guard(sh.dev);
    bank_release(sh.cur);
    if (sh.has_alt) {
      bank_release(sh.alt);
      cudaFree(sh.keys);
    }
    if (sh.has_export) soa_release(sh.exported);
    for (Replica& r : sh.replicas) cudaFree(r.copy);
  }
  if (bank->mirror.present) {
    nb200_particle_soa& a = bank->mirror.a;
    void* p[] = {a.x, a.y, a.omega_x, a.omega_y, a.energy, a.weight, a.dt_to_census,
                 a.mfp_to_collision, a.cellx, a.celly, a.dead};
    for (void* q : p) cudaFreeHost(q);
  }
  if (g_last_deferred == bank) g_last_deferred = nullptr;
  BankHeader* h = bank->header;
  g_handles.erase(views_of(h));
  h->magic = 0;
  delete bank;
  free(h);
  return 0;
}

extern "C" int nb200_memcpy_h2d(void* dst_device, const void* src_host, size_t bytes) {
  CTX_OR_RETURN(c);
  flush_groups_touching(dst_device, bytes);
  CU_TRY(cudaMemcpyAsync(dst_device, src_host, bytes, cudaMemcpyHostToDevice, c.stream));
  CU_TRY(cudaStreamSynchronize(c.stream));
  return 0;
}

extern "C" int nb200_memcpy_d2h(void* dst_host, const void* src_device, size_t bytes) {
  CTX_OR_RETURN(c);
  flush_groups_touching(src_device, bytes);
  CU_TRY(cudaMemcpyAsync(dst_host, src_device, bytes, cudaMemcpyDeviceToHost, c.stream));
  CU_TRY(cudaStreamSynchronize(c.stream));
  return 0;
}

extern "C" int nb200_memcpy_h2d_async(void* dst_device, const void* src_host, size_t bytes,
                                      void* cuda_stream) {
  CTX_OR_RETURN(c);
  (void)c;
  CU_TRY(cudaMemcpyAsync(dst_device, src_host, bytes, cudaMemcpyHostToDevice,
                         (cudaStream_t)cuda_stream));
  return 0;
}

extern "C" int nb200_memcpy_d2h_async(void* dst_host, const void* src_device, size_t bytes,
                                      void* cuda_stream) {
  CTX_OR_RETURN(c);
  (void)c;
  flush_groups_touching(src_device, bytes);
  CU_TRY(cudaMemcpyAsync(dst_host, src_device, bytes, cudaMemcpyDeviceToHost,
                         (cudaStream_t)cuda_stream));
  return 0;
}

extern "C" int nb200_memset_d(void* dst_device, int value, size_t bytes) {
  CTX_OR_RETURN(c);
  flush_groups_touching(dst_device, bytes);
  CU_TRY(cudaMemsetAsync(dst_device, value, bytes, c.stream));
  return 0;
}

extern "C" int nb200_synchronize(void) {
  CTX_OR_RETURN(c);
  CU_TRY(cudaStreamSynchronize(c.stream));
  return 0;
}

extern "C" int nb200_set_option(const char* name, int value) {
  read_environment();
  const int i = option_index(name);
  if (i < 0) {
    set_error("nb200_set_option: unknown option '%s'", name);
    return NB200_BAD_OPTION;
  }
  const OptionSpec& spec = kOptionSpecs[i];
  if (value < spec.lo || value > spec.hi || option_value_invalid(spec, value)) {
    set_error("nb200_set_option: %s=%d is outside [%d, %d]%s", name, value, spec.lo, spec.hi,
              option_value_invalid(spec, value) ? " (1: one batch has no spread)" : "");
    return NB200_BAD_OPTION;
  }
  const int prev = g_opt.*(spec.slot);
  g_opt.*(spec.slot) = value;
  return prev;
}

extern "C" int nb200_get_option(const char* name) {
  read_environment();
  const int i = option_index(name);
  if (i < 0) {
    set_error("nb200_get_option: unknown option '%s'", name);
    return NB200_BAD_OPTION;
  }
  return g_opt.*(kOptionSpecs[i].slot);
}

extern "C" int nb200_bank_set_option(nb200_particle_soa* particles, const char* name, int value) {
  Bank* bank = bank_of(particles);
  const int i = option_index(name);
  if (!bank || i < 0) {
    set_error("nb200_bank_set_option: not a bank handle, or unknown option '%s'", name);
    return NB200_BAD_OPTION;
  }
  const OptionSpec& spec = kOptionSpecs[i];
  if (value < spec.lo || value > spec.hi) {
    set_error("nb200_bank_set_option: %s=%d is outside [%d, %d]", name, value, spec.lo, spec.hi);
    return NB200_BAD_OPTION;
  }
  if (spec.slot == &Options::tally_batches) {
    set_error("nb200_bank_set_option: tally_batches is fixed when the bank is created "
              "(nb200_set_option before inject_particles / nb200_bank_create)");
    return NB200_BAD_OPTION;
  }
  if (bank->batches.B > 0 && ((spec.slot == &Options::pipeline && value == 0) ||
                              (spec.slot == &Options::tally_prereduce && value != 0))) {
    set_error("nb200_bank_set_option: %s=%d on a bank with tally_batches (only the pipelined "
              "kernel without tally_prereduce has batches)", name, value);
    return NB200_BAD_OPTION;
  }
  if (bank->flux && ((spec.slot == &Options::pipeline && value == 0) ||
                     (spec.slot == &Options::tally_prereduce && value != 0))) {
    set_error("nb200_bank_set_option: %s=%d on a bank with a flux tally attached (only the "
              "pipelined kernel without tally_prereduce has the flux)", name, value);
    return NB200_BAD_OPTION;
  }
  const int prev = opt_of(bank, spec.slot);
  for (auto& o : bank->overrides)
    if (o.first == i) {
      o.second = value;
      return prev;
    }
  bank->overrides.push_back({i, value});
  return prev;
}

extern "C" int nb200_solve_finish(uint64_t* facet_events, uint64_t* collision_events) {
  if (!g_last_deferred || g_last_deferred->pending.empty()) {
    set_error("nb200_solve_finish: no timestep is pending");
    return -3;
  }
  finish_oldest(g_last_deferred, facet_events, collision_events);
  return 0;
}

extern "C" int nb200_bank_solve_finish(nb200_particle_soa* particles, uint64_t* facet_events,
                                       uint64_t* collision_events) {
  Bank* bank = bank_of(particles);
  if (!bank || bank->pending.empty()) {
    set_error("nb200_bank_solve_finish: not a bank handle, or no timestep is pending");
    return -3;
  }
  finish_oldest(bank, facet_events, collision_events);
  return 0;
}

extern "C" int nb200_bank_pending(nb200_particle_soa* particles) {
  Bank* bank = bank_of(particles);
  return bank ? (int)bank->pending.size() : -3;
}

extern "C" int nb200_last_step_stats(uint64_t out[8]) {
  for (int k = 0; k < 8; ++k) out[k] = g_last_stats[k];
  return 0;
}

extern "C" uint64_t nb200_kernel_launches(void) {
  uint64_t total = 0;
  for (DeviceCtx* c : g_ctx)
    if (c) total += c->launches;
  return total;
}

// ----------------------------------------------------------------- sharded runs: tally --
extern "C" int nb200_tally_sync(double* tally_device) {
  CTX_OR_RETURN(c);
  (void)c;
  for (Bank* b : g_batched)
    if (!tally_device || b->batches.target == tally_device) batches_flush(b, b->batches);
  for (Bank* b : g_flux)
    if (!tally_device || b->flux == tally_device) batches_flush(b, b->flux_batches);
  for (TallyGroup* g : g_groups)
    if (!tally_device || g->target == tally_device) group_flush(*g);
  return 0;
}

// ------------------------------------------------------------------------ tally batches --
// The bank's batched state, flushed into the caller's tally; nullptr (error set) if there is none.
static Bank* flushed_batches(nb200_particle_soa* particles, const char* who) {
  Bank* bank = bank_of(particles);
  if (!bank || bank->batches.B <= 0) {
    set_error("%s: not a bank handle created with tally_batches", who);
    return nullptr;
  }
  if (!bank->batches.slab) {
    set_error("%s: no timestep of this bank has deposited into its batches yet", who);
    return nullptr;
  }
  batches_flush(bank, bank->batches);
  return bank;
}

extern "C" int nb200_bank_tally_batches(nb200_particle_soa* particles, double* out_device,
                                        size_t ncells) {
  CTX_OR_RETURN(c0);
  (void)c0;
  Bank* bank = flushed_batches(particles, "nb200_bank_tally_batches");
  if (!bank) return -3;
  const TallyBatches& tb = bank->batches;
  if (!out_device || ncells != tb.ncells) {
    set_error("nb200_bank_tally_batches: the batches cover %zu cells, %zu were asked for",
              tb.ncells, ncells);
    return -3;
  }
  DeviceGuard guard(bank->shards[0].dev);
  DeviceCtx& c = ctx_on(bank->shards[0].dev);
  c.launches += launch_batch_export(tb.slab, tb.B, tb.ncells, out_device, c.stream);
  CU_TRY(cudaGetLastError());
  CU_TRY(cudaStreamSynchronize(c.stream));
  return tb.B;
}

extern "C" int nb200_bank_tally_relerr(nb200_particle_soa* particles, double* relerr_device,
                                       double* total_relerr_host) {
  CTX_OR_RETURN(c0);
  (void)c0;
  Bank* bank = flushed_batches(particles, "nb200_bank_tally_relerr");
  if (!bank) return -3;
  const TallyBatches& tb = bank->batches;
  DeviceGuard guard(bank->shards[0].dev);
  DeviceCtx& c = ctx_on(bank->shards[0].dev);
  if (relerr_device) {
    c.launches += launch_batch_relerr(tb.slab, tb.B, tb.ncells, bank->n, relerr_device, c.stream);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(c.stream));
  }
  if (total_relerr_host) *total_relerr_host = batches_total_relerr(bank, tb);
  return 0;
}

// Host-side evaluation of the history kernel's pid -> batch map (pure integer arithmetic), for
// the tests: it has to reproduce shard_split's ranges for any n and B.
extern "C" unsigned nb200_selftest_batch_of(uint64_t pid, uint64_t n, int nbatches) {
  if (nbatches < 1 || n > 0x7fffffffull || (uint64_t)nbatches > n || pid >= n) return UINT_MAX;
  return batch_of((unsigned)pid, (unsigned)n, (unsigned)nbatches);
}

// ------------------------------------------------------------------------- flux tally --
// Why flux_device cannot be attached to the bank (plain, or batched with the bank's B), as an
// error code with the message set; 0 if it can. Both attach functions check the same things.
static int refuse_flux_array(Bank* bank, double* flux_device, size_t ncells, bool batched,
                             const char* who) {
  if (!single_shard(bank) || g_mp) {
    set_error("%s: a bank sharded over several GPUs or in a multi-process group has no flux "
              "tally", who);
    return -3;
  }
  if (!batched && bank->batches.B > 0) {
    set_error("%s: a bank with tally_batches has no flux tally (nb200_bank_set_batched_flux_tally "
              "attaches a batched one)", who);
    return -3;
  }
  if (batched && bank->batches.B <= 0) {
    set_error("%s: the bank has no tally_batches (a batched flux has the bank's batches)", who);
    return -3;
  }
  if (!opt_of(bank, &Options::pipeline) || opt_of(bank, &Options::tally_prereduce)) {
    set_error("%s: needs pipeline=1 and tally_prereduce=0 (only the pipelined kernel without "
              "tally_prereduce has the flux)", who);
    return -3;
  }
  if (ncells == 0 || ncells >= (1ull << 31)) {
    set_error("%s: %zu cells (1 .. 2^31 - 1)", who, ncells);
    return -3;
  }
  if (batched && (unsigned long long)ncells * (unsigned long long)bank->batches.B >= (1ull << 31)) {
    set_error("%s: tally_batches=%d over %zu cells needs 2^31 or more flux slots (the history "
              "kernel indexes them with 32 bits)", who, bank->batches.B, ncells);
    return -3;
  }
  cudaPointerAttributes attr{};
  if (cudaPointerGetAttributes(&attr, flux_device) != cudaSuccess ||
      (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) ||
      attr.device != bank->shards[0].dev) {
    (void)cudaGetLastError();
    set_error("%s: the flux array is not device memory on the bank's GPU %d", who,
              bank->shards[0].dev);
    return -3;
  }
  return 0;
}

extern "C" int nb200_bank_set_flux_tally(nb200_particle_soa* particles, double* flux_device,
                                         size_t ncells) {
  const char* who = "nb200_bank_set_flux_tally";
  Bank* bank = bank_of(particles);
  if (!bank) {
    set_error("%s: not a bank handle", who);
    return -3;
  }
  if (int rc = refuse_if_pending(bank, who)) return rc;
  if (!flux_device) return flux_attach(bank, nullptr, 0);
  if (int rc = refuse_flux_array(bank, flux_device, ncells, false, who)) return rc;
  return flux_attach(bank, flux_device, ncells);
}

extern "C" int nb200_bank_set_batched_flux_tally(nb200_particle_soa* particles,
                                                 double* flux_device, size_t ncells) {
  const char* who = "nb200_bank_set_batched_flux_tally";
  Bank* bank = bank_of(particles);
  if (!bank) {
    set_error("%s: not a bank handle", who);
    return -3;
  }
  if (int rc = refuse_if_pending(bank, who)) return rc;
  if (!flux_device) return flux_attach(bank, nullptr, 0);
  if (int rc = refuse_flux_array(bank, flux_device, ncells, true, who)) return rc;
  return flux_attach(bank, flux_device, ncells, bank->batches.B);
}

// The bank's flux batches, flushed into the attached array; nullptr (error set) if there are none.
static Bank* flushed_flux_batches(nb200_particle_soa* particles, const char* who) {
  Bank* bank = bank_of(particles);
  if (!bank || bank->flux_batches.B <= 0) {
    set_error("%s: not a bank handle with a batched flux tally attached", who);
    return nullptr;
  }
  if (!bank->flux_batches.deposited) {
    set_error("%s: no timestep of this bank has deposited into its flux batches yet", who);
    return nullptr;
  }
  batches_flush(bank, bank->flux_batches);
  return bank;
}

extern "C" int nb200_bank_flux_batches(nb200_particle_soa* particles, double* out_device,
                                       size_t ncells) {
  Bank* bank = flushed_flux_batches(particles, "nb200_bank_flux_batches");
  if (!bank) return -3;
  const TallyBatches& tb = bank->flux_batches;
  if (!out_device || ncells != tb.ncells) {
    set_error("nb200_bank_flux_batches: the flux batches cover %zu cells, %zu were asked for",
              tb.ncells, ncells);
    return -3;
  }
  DeviceGuard guard(bank->shards[0].dev);
  DeviceCtx& c = ctx_on(bank->shards[0].dev);
  c.launches += launch_batch_export(tb.slab, tb.B, tb.ncells, out_device, c.stream);
  CU_TRY(cudaGetLastError());
  CU_TRY(cudaStreamSynchronize(c.stream));
  return tb.B;
}

extern "C" int nb200_bank_flux_relerr(nb200_particle_soa* particles, double* relerr_device,
                                      double* total_relerr_host) {
  Bank* bank = flushed_flux_batches(particles, "nb200_bank_flux_relerr");
  if (!bank) return -3;
  const TallyBatches& tb = bank->flux_batches;
  DeviceGuard guard(bank->shards[0].dev);
  DeviceCtx& c = ctx_on(bank->shards[0].dev);
  if (relerr_device) {
    c.launches += launch_batch_relerr(tb.slab, tb.B, tb.ncells, bank->n, relerr_device, c.stream);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(c.stream));
  }
  if (total_relerr_host) *total_relerr_host = batches_total_relerr(bank, tb);
  return 0;
}

extern "C" int nb200_update_replicas(void) {
  g_replica_generation++;
  return 0;
}

// Multi-process sharding (one process per GPU): this process's member of the group, and the
// blob its peers need to map it.
extern "C" int nb200_mp_init(int nranks, int rank, size_t ncells, void* blob_out) {
  CTX_OR_RETURN(c);
  if (nranks < 1 || nranks > kMaxRanks || rank < 0 || rank >= nranks || !ncells || !blob_out) {
    set_error("nb200_mp_init: bad arguments (nranks=%d rank=%d ncells=%zu)", nranks, rank, ncells);
    return -3;
  }
  if (g_mp) {
    set_error("nb200_mp_init: a multi-process group already exists (nb200_mp_finalize first)");
    return -3;
  }
  TallyGroup* g = new TallyGroup();
  g->nranks = nranks;
  g->ncells = ncells;
  g->collective = g_opt.collective;
  g->reduce_ctas = g_opt.reduce_ctas;
  g->reduce_every = g_opt.tally_reduce_every;
  g->mp = true;
  g->mp_rank = rank;
  group_layout(*g);
  group_alloc_member(*g, rank, c.device);
  memset(blob_out, 0, NB200_MP_BLOB_BYTES);
  char* blob = (char*)blob_out;
  if (g->collective) {
    cudaIpcMemHandle_t h;
    CU_TRY(cudaIpcGetMemHandle(&h, g->m[rank].slab));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(blob, &h, 64);
  } else if (rank == 0) {
    std::string why;
    const NcclApi* api = nccl_api(&why);
    if (!api) {
      set_error("nb200_mp_init: %s", why.c_str());
      return -6;
    }
    NcclUniqueId id;
    if (api->GetUniqueId(&id) != kNcclSuccess) {
      set_error("nb200_mp_init: ncclGetUniqueId failed");
      return -6;
    }
    memcpy(blob + 64, &id, 128);
  }
  g_mp = g;
  return 0;
}

extern "C" int nb200_mp_connect(const void* blobs) {
  CTX_OR_RETURN(c);
  (void)c;
  if (!g_mp || !blobs) {
    set_error("nb200_mp_connect: nb200_mp_init has not been called");
    return -3;
  }
  TallyGroup& g = *g_mp;
  const char* all = (const char*)blobs;
  if (g.collective && getenv("NB200_TEST_IPC_FAIL")) {  // test hook: exercise the host's fallback
    set_error("nb200_mp_connect: peer mapping refused (NB200_TEST_IPC_FAIL is set)");
    return -7;
  }
  if (g.collective) {
    for (int r = 0; r < g.nranks; ++r) {
      if (r == g.mp_rank) continue;
      cudaIpcMemHandle_t h;
      memcpy(&h, all + (size_t)r * NB200_MP_BLOB_BYTES, 64);
      void* base = nullptr;
      const cudaError_t err = cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess);
      if (err != cudaSuccess) {
        set_error("nb200_mp_connect: cannot map rank %d's tally slab over CUDA IPC: %s", r,
                  cudaGetErrorString(err));
        (void)cudaGetLastError();
        return -7;
      }
      group_bind(g, g.m[r], (char*)base);
      g.m[r].ipc_opened = true;
    }
  } else {
    std::string why;
    const NcclApi* api = nccl_api(&why);
    if (!api) {
      set_error("nb200_mp_connect: %s", why.c_str());
      return -6;
    }
    NcclUniqueId id;
    memcpy(&id, all + 64, 128);  // rank 0's blob carries the id
    const int rc = api->CommInitRank(&g.m[g.mp_rank].comm, g.nranks, id, g.mp_rank);
    if (rc != kNcclSuccess) {
      set_error("nb200_mp_connect: ncclCommInitRank failed: %s", api->GetErrorString(rc));
      return -6;
    }
  }
  g_groups.push_back(g_mp);
  return 0;
}

extern "C" int nb200_mp_finalize(void) {
  if (!g_mp) return 0;
  group_free(g_mp);
  g_mp = nullptr;
  return 0;
}

// ------------------------------------------------------------------------- microbench --
extern "C" int nb200_microbench_red(int pattern, size_t footprint_bytes, int iters,
                                    double* reductions_per_s) {
  CTX_OR_RETURN(c);
  size_t cells = 1;
  while (cells * 2 * sizeof(double) <= footprint_bytes) cells *= 2;  // power of two
  if (cells < 1024 || iters < 1 || !reductions_per_s) {
    set_error("nb200_microbench_red: bad arguments");
    return -3;
  }
  double* scratch = nullptr;
  CU_TRY(cudaMalloc(&scratch, cells * sizeof(double)));
  CU_TRY(cudaMemsetAsync(scratch, 0, cells * sizeof(double), c.stream));
  double seconds = 0.0, reds = 0.0;
  c.launches += launch_red_rate(scratch, cells, 4000, iters, pattern, c.ev_begin[0], c.ev_end[0],
                                &seconds, &reds, c.stream);
  cudaFree(scratch);
  CU_TRY(cudaGetLastError());
  *reductions_per_s = seconds > 0.0 ? reds / seconds : 0.0;
  return 0;
}

// ---------------------------------------------------------------------- self-test hooks --
extern "C" int nb200_selftest_rng_log(uint64_t pkey0, uint64_t master_key, uint64_t counter,
                                      int n, uint64_t* raw_host, double* unit_host,
                                      double* neglog_host) {
  CTX_OR_RETURN(c);
  uint64_t* d_raw = nullptr;
  double *d_unit = nullptr, *d_nl = nullptr;
  CU_TRY(cudaMalloc(&d_raw, sizeof(uint64_t) * 2 * n));
  CU_TRY(cudaMalloc(&d_unit, sizeof(double) * 2 * n));
  CU_TRY(cudaMalloc(&d_nl, sizeof(double) * 2 * n));
  c.launches += launch_selftest_rng_log(pkey0, master_key, counter, n, c.d_logt, d_raw, d_unit,
                                        d_nl, c.stream);
  CU_TRY(cudaMemcpyAsync(raw_host, d_raw, sizeof(uint64_t) * 2 * n, cudaMemcpyDeviceToHost, c.stream));
  CU_TRY(cudaMemcpyAsync(unit_host, d_unit, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, c.stream));
  CU_TRY(cudaMemcpyAsync(neglog_host, d_nl, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, c.stream));
  CU_TRY(cudaStreamSynchronize(c.stream));
  cudaFree(d_raw);
  cudaFree(d_unit);
  cudaFree(d_nl);
  return 0;
}

extern "C" int nb200_selftest_log(const double* x_host, double* y_host, int n) {
  CTX_OR_RETURN(c);
  double *d_x = nullptr, *d_y = nullptr;
  CU_TRY(cudaMalloc(&d_x, sizeof(double) * n));
  CU_TRY(cudaMalloc(&d_y, sizeof(double) * n));
  CU_TRY(cudaMemcpyAsync(d_x, x_host, sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
  c.launches += launch_selftest_log(d_x, d_y, n, c.d_logt, c.stream);
  CU_TRY(cudaMemcpyAsync(y_host, d_y, sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
  CU_TRY(cudaStreamSynchronize(c.stream));
  cudaFree(d_x);
  cudaFree(d_y);
  return 0;
}

extern "C" int nb200_selftest_cs(const double* keys_host, const double* values_host,
                                 int nentries, const double* energies_host, int n,
                                 int* index_host, double* value_host) {
  CTX_OR_RETURN(c);
  double *d_k = nullptr, *d_v = nullptr, *d_e = nullptr, *d_o = nullptr;
  int* d_i = nullptr;
  CU_TRY(cudaMalloc(&d_k, sizeof(double) * nentries));
  CU_TRY(cudaMalloc(&d_v, sizeof(double) * nentries));
  CU_TRY(cudaMalloc(&d_e, sizeof(double) * n));
  CU_TRY(cudaMalloc(&d_o, sizeof(double) * n));
  CU_TRY(cudaMalloc(&d_i, sizeof(int) * n));
  CU_TRY(cudaMemcpyAsync(d_k, keys_host, sizeof(double) * nentries, cudaMemcpyHostToDevice, c.stream));
  CU_TRY(cudaMemcpyAsync(d_v, values_host, sizeof(double) * nentries, cudaMemcpyHostToDevice, c.stream));
  CU_TRY(cudaMemcpyAsync(d_e, energies_host, sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
  // stage the table exactly as a timestep does, then run both lookups side by side
  const CsParams par = nentries >= 2
                           ? cs_params_from_ends(keys_host[0], keys_host[nentries - 1], nentries)
                           : CsParams();
  double2* d_kv = nullptr;
  int* d_bk = nullptr;
  CU_TRY(cudaMalloc(&d_kv, sizeof(double2) * nentries));
  CU_TRY(cudaMalloc(&d_bk, sizeof(int) * (par.nb + 1)));
  CU_TRY(cudaMemsetAsync(c.d_totals, 0, sizeof(unsigned long long) * kTotCount, c.stream));
  c.launches += launch_stage_cs(d_k, d_v, nentries, d_kv, d_bk, par.bits0, par.shift, par.nb,
                                nullptr, c.d_totals, c.stream);
  const CsStage staged{d_kv, d_bk, par.bits0, par.shift, par.nb, nentries};
  c.launches += launch_selftest_cs(d_k, d_v, nentries, staged, d_e, n, d_i, d_o, c.stream);
  CU_TRY(cudaMemcpyAsync(index_host, d_i, sizeof(int) * n, cudaMemcpyDeviceToHost, c.stream));
  CU_TRY(cudaMemcpyAsync(value_host, d_o, sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
  CU_TRY(cudaStreamSynchronize(c.stream));
  cudaFree(d_k); cudaFree(d_v); cudaFree(d_e); cudaFree(d_o); cudaFree(d_i);
  cudaFree(d_kv); cudaFree(d_bk);
  return 0;
}

extern "C" int nb200_selftest_div(const double* a_host, const double* b_host, int n,
                                  double* fast_host, double* ieee_host) {
  CTX_OR_RETURN(c);
  double* d[4] = {nullptr, nullptr, nullptr, nullptr};
  for (auto& p : d) CU_TRY(cudaMalloc(&p, sizeof(double) * n));
  CU_TRY(cudaMemcpyAsync(d[0], a_host, sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
  CU_TRY(cudaMemcpyAsync(d[1], b_host, sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
  c.launches += launch_selftest_div(d[0], d[1], d[2], d[3], n, c.stream);
  CU_TRY(cudaMemcpyAsync(fast_host, d[2], sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
  CU_TRY(cudaMemcpyAsync(ieee_host, d[3], sizeof(double) * n, cudaMemcpyDeviceToHost, c.stream));
  CU_TRY(cudaStreamSynchronize(c.stream));
  for (auto& p : d) cudaFree(p);
  return 0;
}

extern "C" int nb200_selftest_fastmath(const double* a_host, const double* b_host, int n,
                                       double* out_host) {
  CTX_OR_RETURN(c);
  double *d_a = nullptr, *d_b = nullptr, *d_o = nullptr;
  CU_TRY(cudaMalloc(&d_a, sizeof(double) * n));
  CU_TRY(cudaMalloc(&d_b, sizeof(double) * n));
  CU_TRY(cudaMalloc(&d_o, sizeof(double) * 6 * (size_t)n));
  CU_TRY(cudaMemcpyAsync(d_a, a_host, sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
  CU_TRY(cudaMemcpyAsync(d_b, b_host, sizeof(double) * n, cudaMemcpyHostToDevice, c.stream));
  c.launches += launch_selftest_fastmath(d_a, d_b, d_o, n, c.stream);
  CU_TRY(cudaMemcpyAsync(out_host, d_o, sizeof(double) * 6 * (size_t)n, cudaMemcpyDeviceToHost,
                         c.stream));
  CU_TRY(cudaStreamSynchronize(c.stream));
  cudaFree(d_a);
  cudaFree(d_b);
  cudaFree(d_o);
  return 0;
}

extern "C" void nb200_host_threefry2x64_20(uint64_t c0, uint64_t c1, uint64_t k0, uint64_t k1,
                                           uint64_t out[2]) {
  threefry2x64_20(c0, c1, k0, k1, out[0], out[1]);
}

extern "C" double nb200_host_log(double x) { return nb_log(x, &kHostLogTable); }
extern "C" double nb200_host_sin(double x) { return nb_sin(x, &kHostSinCosTable); }
extern "C" double nb200_host_cos(double x) { return nb_cos(x, &kHostSinCosTable); }

// Batch flavour of the two hooks above (the host build of the device source).
extern "C" void nb200_host_sincos(const double* x, long long n, double* s, double* c) {
#pragma omp parallel for schedule(static)
  for (long long i = 0; i < n; ++i) {
    s[i] = nb_sin(x[i], &kHostSinCosTable);
    c[i] = nb_cos(x[i], &kHostSinCosTable);
  }
}

// Compares the host build of nb_sin/nb_cos with this process's libm on n arguments; returns
// the number of arguments where either differs in any bit (first offender in *bad_x).
extern "C" long long nb200_selftest_host_sincos(const double* x, long long n, double* bad_x) {
  long long bad = 0;
  double first_bad = 0.0;
#pragma omp parallel for schedule(static) reduction(+ : bad)
  for (long long i = 0; i < n; ++i) {
    const double s = nb_sin(x[i], &kHostSinCosTable), c = nb_cos(x[i], &kHostSinCosTable);
    const double rs = sin(x[i]), rc = cos(x[i]);
    if (memcmp(&s, &rs, 8) != 0 || memcmp(&c, &rc, 8) != 0) {
      if (!bad) {
#pragma omp critical
        first_bad = x[i];
      }
      bad++;
    }
  }
  if (bad_x) *bad_x = first_bad;
  return bad;
}

// sin and cos of n host arguments, evaluated on the device.
extern "C" int nb200_selftest_sincos(const double* x_host, double* s_host, double* c_host,
                                     int n) {
  CTX_OR_RETURN(c);
  double *d_x = nullptr, *d_s = nullptr, *d_c = nullptr;
  CU_TRY(cudaMalloc(&d_x, sizeof(double) * n));
  CU_TRY(cudaMalloc(&d_s, sizeof(double) * n));
  CU_TRY(cudaMalloc(&d_c, sizeof(double) * n));
  CU_TRY(cudaMemcpy(d_x, x_host, sizeof(double) * n, cudaMemcpyHostToDevice));
  c.launches += launch_selftest_sincos(d_x, d_s, d_c, n, c.d_sct, c.stream);
  CU_TRY(cudaStreamSynchronize(c.stream));
  CU_TRY(cudaMemcpy(s_host, d_s, sizeof(double) * n, cudaMemcpyDeviceToHost));
  CU_TRY(cudaMemcpy(c_host, d_c, sizeof(double) * n, cudaMemcpyDeviceToHost));
  cudaFree(d_x);
  cudaFree(d_s);
  cudaFree(d_c);
  return 0;
}
