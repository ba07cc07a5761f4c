// transport.cuh - internal C++ interface between the C-ABI layer and the kernels.
#pragma once

#include "nb_bank.cuh"

namespace nb {

// Threads per CTA of the history kernels. The register file holds 25 warps of 80 registers
// (65536 / 2560): 6 CTAs of 128 threads use 24 of them, 5 CTAs of 160 threads all 25.
#ifndef NB_HISTORY_THREADS
#define NB_HISTORY_THREADS 128
#endif
constexpr int kHistoryThreads = NB_HISTORY_THREADS;

// Every launch_* returns the number of kernels it launched (for the launch counter).
int launch_history_direct(const StepArgs& a, cudaStream_t st);

// Phased pipeline (pipeline.cu): sort phase = begin-step/classify + scan + scatter into
// `alt`; history = event loop over the sorted live prefix.
int launch_sort_phase(const StepArgs& a, const SortArgs& s, const BankView& alt,
                      cudaStream_t st);
// bt.nbatches > 0 runs the batched variant (option tally_batches); a non-null `flux` the
// variant that also deposits the track-length flux there (nb200_bank_set_flux_tally).
int launch_history(const StepArgs& a, const BatchArgs& bt, double* flux, const unsigned* n_live,
                   int n_upper, bool fast_div, bool prereduce, const void* pin, size_t pin_bytes,
                   size_t pin_budget, int smem_pad, cudaStream_t st);
// Batch partial tallies (tally_batches.cu). The slab holds the B partial tallies S_b in the
// layout of batch_slot() and behind them one more array F of ncells: sum_b S_b as of the last
// flush. Flush: tally += sum_b S_b - F, F = sum_b S_b (summed in batch order).
int launch_batch_flush(double* slab, int B, size_t ncells, double* tally, cudaStream_t st);
// out = the B partial tallies batch-major ([b][cell]), whatever the slab's layout.
int launch_batch_export(const double* slab, int B, size_t ncells, double* out, cudaStream_t st);
// relerr[cell] = relative error of the batch mean (n: particles, split into B batches).
int launch_batch_relerr(const double* slab, int B, size_t ncells, int n, double* relerr,
                        cudaStream_t st);
// partial[b * blocks + k] = sum over block k's cells of S_b (blocks = kBatchSumBlocks).
constexpr int kBatchSumBlocks = 148;
int launch_batch_sums(const double* slab, int B, size_t ncells, double* partial, cudaStream_t st);
// Per-step staging of the read-only inputs (stage.cu).
int launch_stage_cs(const double* keys, const double* vals, int n, double2* kv, int* bucket,
                    unsigned long long bits0, int shift, int nb, const double* twin_keys,
                    unsigned long long* totals, cudaStream_t st);
int launch_compare_grids(const double* a, const double* b, int n, unsigned long long* totals,
                         cudaStream_t st);
// fine/coarse must hold tile_counts(nx, ny) doubles; *map receives the views.
int launch_stage_tiles(const double* density, int nx, int ny, double* fine, double* coarse,
                       TileMap* map, cudaStream_t st);
// out must hold 4 * stride doubles, stride >= max(nx, ny) + 1.
int launch_stage_edges(const double* edgex, int nx, const double* edgey, int ny, int stride,
                       double* out, cudaStream_t st);
int launch_selftest_div(const double* a, const double* b, double* fast, double* ieee, int n,
                        cudaStream_t st);
int launch_selftest_fastmath(const double* a, const double* b, double* out, int n,
                             cudaStream_t st);

// inject_particles on the device (transport.cu: k_inject). Edges are device pointers.
struct SinCosTable;
struct InjectArgs {
  const double* edgex;
  const double* edgey;
  int nx, ny;
  double left, bottom, width, height;  // the source box of neutral_data.c:39-95
  double dt, initial_energy;
};
int launch_inject(BankView b, int count, uint64_t first, const InjectArgs& ia,
                  const SinCosTable* sct, cudaStream_t st);
int launch_selftest_sincos(const double* x, double* s, double* c, int n, const SinCosTable* sct,
                           cudaStream_t st);

int launch_import_soa(BankView b, SoaView s, int n, int origin0, cudaStream_t st);
int launch_export_soa(BankView b, SoaView s, int n, cudaStream_t st);
int launch_import_aos(BankView b, const void* aos, int n, cudaStream_t st);
int launch_export_aos(BankView b, void* aos, int n, cudaStream_t st);

int launch_accumulate(double* dst, const double* src, size_t n, cudaStream_t st);
int launch_accumulate_clear(double* dst, double* src, size_t n, cudaStream_t st);

int launch_selftest_rng_log(uint64_t pkey0, uint64_t master_key, uint64_t counter, int n,
                            const LogTable* logt, uint64_t* raw, double* unit,
                            double* neglog, cudaStream_t st);
int launch_selftest_log(const double* x, double* y, int n, const LogTable* logt,
                        cudaStream_t st);
int launch_selftest_cs(const double* keys, const double* vals, int n_entries, CsStage staged,
                       const double* e, int n, int* ind, double* out, cudaStream_t st);

}  // namespace nb
