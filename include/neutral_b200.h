/*
 * neutral_b200.h - C ABI of the B200 (sm_100a) kernel set for UoB-HPC/neutral.
 *
 * libneutral_b200.so is a drop-in `KERNELS=b200` kernel set: it exports the three functions
 * of the reference plugin boundary (neutral_interface.h:11-36) with the reference's names,
 * argument order and meaning, plus the per-kernel-set allocation layer the reference's host
 * driver expects from its parent `arch` project (call sites neutral_data.c:54-62,97-105,
 * 146-147,168-169; main.c:63). The reference's unmodified main.c + neutral_data.c link
 * against it when compiled with -DSoA (the layout every GPU kernel set of the reference
 * uses, Makefile:60-71). Everything else in this header (nb200_*) is an extension for
 * callers that are not the C driver: FFI hosts, the parity tests, the bench harness.
 *
 * Plain C: pointers and sizes only. The types below are layout-compatible with the
 * reference's `Particle` (-DSoA, neutral_data.h:48-61) and `CrossSection`
 * (neutral_data.h:38-43); they carry their own names so this header can be included next
 * to, or without, the reference's neutral_data.h.
 *
 * Memory spaces. In the device-resident flavour (section 1) every array argument is DEVICE
 * memory on the current GPU (the bank's primary GPU when the bank is sharded over several), obtained from the allocation layer (section 2) or from any
 * other CUDA allocator (e.g. a torch tensor's data_ptr); scalars passed by pointer
 * (nlocal_particles, facet_events, collision_events) and the CrossSection structs
 * themselves are HOST memory. Section 3 has the host-buffer flavour.
 *
 * Errors. Like the reference (arch TERMINATE, used e.g. omp3/neutral.c:572) the three
 * boundary functions print a message and exit(EXIT_FAILURE) on a fatal error - including a
 * missing GPU: there is no CPU fallback. nb200_* functions return 0 on success and a
 * negative code on failure, with nb200_last_error() describing it.
 */
#ifndef NEUTRAL_B200_H
#define NEUTRAL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NB200_ABI_VERSION 2
/* nb200_set_option / nb200_get_option / nb200_bank_set_option: unknown name or value out of
 * range (option values themselves may be negative, e.g. tile_shift = -1). */
#define NB200_BAD_OPTION (-2147483647 - 1)
/* Bytes one rank contributes to nb200_mp_connect (CUDA IPC handle + NCCL id). */
#define NB200_MP_BLOB_BYTES 256

/* == reference `Particle` under -DSoA (neutral_data.h:48-61) */
typedef struct {
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
} nb200_particle_soa;

/* == reference AoS `Particle` (neutral_data.h:66-79), 80 bytes */
typedef struct {
  double x, y, omega_x, omega_y, energy, weight, dt_to_census, mfp_to_collision;
  int cellx, celly, dead;
} nb200_particle_aos;

/* == reference `CrossSection` (neutral_data.h:38-43) */
typedef struct {
  double* keys;
  double* values;
  int nentries;
} nb200_cross_section;

/* ------------------------------------------------------------------------------------
 * 1. The plugin boundary, device-resident flavour (replaces omp3/neutral.c:19-40,
 *    :520-557, :560-630 behind neutral_interface.h:11-36).
 * ---------------------------------------------------------------------------------- */

/* One timestep of the whole local bank. Replaces solve_transport_2d
 * (neutral_interface.h:11-20 / omp3/neutral.c:19-40). `particles` is the handle returned by
 * inject_particles (or nb200_bank_create); *facet_events and *collision_events are ADDED
 * to, as omp3 does (omp3/neutral.c:202-203); prints "Particles  <n>" (omp3/neutral.c:205).
 * reduce_array0..2, when non-null, are uint64[bank size] device arrays that receive the
 * cumulative per-particle facet / collision / census counts in injection order.
 * pad must be 0 and x_off = y_off = 0 (the only configuration main.c:34,101-110 produces).
 *
 * A bank sharded over several GPUs (NB200_NGPUS / option "ngpus", or a multi-process group,
 * section 5) transports every shard on its own GPU against replicas of the read-only inputs
 * and combines the tally inside the library (csrc/nb_group.cuh); the counts returned are the
 * sums over the shards. The caller-visible tally is then brought up to date lazily: by
 * validate, by copy_buffer / nb200_memcpy_d2h of it, or by nb200_tally_sync. */
void solve_transport_2d(
    const int nx, const int ny, const int global_nx, const int global_ny,
    const uint64_t master_key, const int pad, const int x_off, const int y_off,
    const double dt, const int ntotal_particles, int* nlocal_particles,
    const int* neighbours, nb200_particle_soa* particles, const double* density,
    const double* edgex, const double* edgey, const double* edgedx,
    const double* edgedy, nb200_cross_section* cs_scatter_table,
    nb200_cross_section* cs_absorb_table, double* energy_deposition_tally,
    uint64_t* reduce_array0, uint64_t* reduce_array1, uint64_t* reduce_array2,
    uint64_t* facet_events, uint64_t* collision_events);

/* Creates and fills the bank. Replaces inject_particles (neutral_interface.h:23-31 /
 * omp3/neutral.c:560-630): positions, cells and directions come from the same
 * Threefry-2x64 streams as the reference and from a bit-exact restatement of the libm cos/sin
 * the reference calls, generated on the device(s) where the bank lives (option
 * "device_inject" = 0: computed on the host with libm and uploaded; same bits).
 * Returns the bytes of device memory allocated (including the head-room of option
 * "headroom_pct"; omp3/neutral.c:570 allocates twice the bank). *particles receives an opaque
 * handle laid out as the reference's -DSoA struct of 11 pointers (neutral_data.h:48-61).
 * The pointers are NULL until something asks for them: nb200_bank_view / nb200_bank_export
 * make them a plain DEVICE SoA view; with option "host_mirror" = 1 (or NB200_HOST_MIRROR=1 in
 * the environment, for visit_dump decks: main.c:169-200 reads the bank on the host) they are
 * HOST arrays that the library refreshes after inject and after every collected timestep. */
size_t inject_particles(const int nparticles, const int global_nx, const int local_nx,
                        const int local_ny, const int pad,
                        const double local_particle_left_off,
                        const double local_particle_bottom_off,
                        const double local_particle_width,
                        const double local_particle_height, const int x_off,
                        const int y_off, const double dt, const double* edgex,
                        const double* edgey, const double initial_energy,
                        nb200_particle_soa** particles);

/* Sums the tally on the device and compares it with problems/neutral.tests at 1e-3
 * (relative: VALIDATE_TOLERANCE, neutral_data.h:27). Replaces validate
 * (neutral_interface.h:35-36 / omp3/neutral.c:520-557); same printed lines. When the
 * environment names a file in NB200_RESULTS_JSON the verdict is also written there as JSON:
 * deck, tally total, expected value, relative error, PASSED / FAILED / NOT_VALIDATED and the
 * per-timestep counts the library saw (SURVEY.md 8f 1). When the tally was deposited by a bank
 * with tally batches (section 6) the JSON also has "tally_batches": B and
 * "tally_total_relative_error": R of the total. */
void validate(const int nx, const int ny, const char* params_filename, const int rank,
              double* energy_tally);

/* ------------------------------------------------------------------------------------
 * 2. Allocation layer of the kernel set (arch `shared.h`; restated in archlite/shared.h).
 *    Kernel-set memory = device memory on the current GPU, zero-filled.
 * ---------------------------------------------------------------------------------- */
size_t allocate_data(double** buf, size_t len);
size_t allocate_float_data(float** buf, size_t len);
size_t allocate_int_data(int** buf, size_t len);
size_t allocate_uint64_data(uint64_t** buf, size_t len);
void allocate_host_data(double** buf, size_t len);       /* pinned host memory */
void allocate_host_float_data(float** buf, size_t len);  /* pinned host memory */
void deallocate_data(double* buf);
void deallocate_host_data(double* buf);
/* send != 0: host -> device, send == 0 (RECV): device -> host; len doubles. */
void copy_buffer(const size_t len, double** src, double** dst, int send);
/* Uploads len doubles to a fresh device buffer (*dst) and frees the host buffer. */
void move_host_buffer_to_device(const size_t len, double** src, double** dst);
/* Binds the process to GPU `rank % device count` (main.c:63). */
void initialise_devices(int rank);

/* ------------------------------------------------------------------------------------
 * 3. Host-buffer flavour: the omp3 signature on HOST arrays (AoS bank, as
 *    omp3/neutral.c:19-40 takes it). Every call uploads what it reads, runs the same
 *    kernels, and downloads what it writes (bank, tally). For FFI hosts and parity tests.
 * ---------------------------------------------------------------------------------- */
void nb200_solve_transport_2d_host(
    const int nx, const int ny, const int global_nx, const int global_ny,
    const uint64_t master_key, const int pad, const int x_off, const int y_off,
    const double dt, const int ntotal_particles, int* nlocal_particles,
    const int* neighbours, nb200_particle_aos* particles, const double* density,
    const double* edgex, const double* edgey, const double* edgedx,
    const double* edgedy, nb200_cross_section* cs_scatter_table,
    nb200_cross_section* cs_absorb_table, double* energy_deposition_tally,
    uint64_t* reduce_array0, uint64_t* reduce_array1, uint64_t* reduce_array2,
    uint64_t* facet_events, uint64_t* collision_events);

/* ------------------------------------------------------------------------------------
 * 4. Extensions
 * ---------------------------------------------------------------------------------- */
int nb200_abi_version(void);
const char* nb200_last_error(void);
/* Number of CUDA devices visible (0 = none: every compute entry point fails loudly). */
int nb200_device_count(void);
/* CUDA stream (cudaStream_t) all work of the CURRENT device is enqueued on; default 0 = the
 * legacy default stream. Refused (-4) while timesteps are enqueued and not collected. */
int nb200_set_stream(void* cuda_stream);

/* Particle sharding across GPUs: the next inject_particles builds only global particles
 * [first, first+count) of the nparticles it is asked for (RNG keys stay global), the same
 * contiguous split omp3 uses for its threads (omp3/neutral.c:64-74). count < 0 clears. */
int nb200_set_shard(int first, int count);

/* Bank from host SoA arrays holding global particles [pid_first, pid_first+count). */
int nb200_bank_create(const nb200_particle_soa* host, int count, int pid_first,
                      nb200_particle_soa** particles);
/* Copies the bank to host SoA arrays in injection order (count = bank size). */
int nb200_bank_download(nb200_particle_soa* particles, nb200_particle_soa* host);
/* Overwrites the bank from host SoA arrays (asynchronous on the library's stream; pinned
 * host memory makes the copies truly asynchronous). */
int nb200_bank_upload(nb200_particle_soa* particles, const nb200_particle_soa* host);
/* Refreshes the plain device SoA view behind the handle's 11 pointers. */
int nb200_bank_export(nb200_particle_soa* particles);
/* The plain device SoA view behind the handle (11 device arrays of bank-size elements,
 * allocated on first use), and the kernel that rebuilds the bank from it (asynchronous on
 * the library's stream): a host that moves banks with its own asynchronous copies fills the
 * view and calls nb200_bank_import, or calls nb200_bank_export and reads the view. */
int nb200_bank_view(nb200_particle_soa* particles, nb200_particle_soa* view_out);
int nb200_bank_import(nb200_particle_soa* particles);
/* Overwrites the bank's state from another bank of the same size (device to device). */
int nb200_bank_copy(nb200_particle_soa* dst, nb200_particle_soa* src);
int nb200_bank_size(nb200_particle_soa* particles);
/* Slots allocated (>= size: option "headroom_pct") and GPUs the bank is sharded over. */
int nb200_bank_capacity(nb200_particle_soa* particles);
int nb200_bank_gpus(nb200_particle_soa* particles);
/* Appends `count` particles (host SoA arrays) into the bank's head-room: they become
 * particles [size, size + count) in injection order with the next global indices as RNG keys.
 * -5 when they do not fit. Single-GPU banks. */
int nb200_bank_append(nb200_particle_soa* particles, const nb200_particle_soa* host, int count);
int nb200_bank_free(nb200_particle_soa* particles);
/* Bank operations that rewrite a bank (upload, import, copy, append, export, download) are
 * refused with -4 while timesteps of it are enqueued and not collected (defer_finish). */

/* Raw device/host copies for hosts without a CUDA binding of their own. */
int nb200_memcpy_h2d(void* dst_device, const void* src_host, size_t bytes);
int nb200_memcpy_d2h(void* dst_host, const void* src_device, size_t bytes);
/* Asynchronous flavours on a caller-supplied cudaStream_t (pinned host memory). */
int nb200_memcpy_h2d_async(void* dst_device, const void* src_host, size_t bytes, void* cuda_stream);
int nb200_memcpy_d2h_async(void* dst_host, const void* src_device, size_t bytes, void* cuda_stream);
int nb200_memset_d(void* dst_device, int value, size_t bytes);
int nb200_synchronize(void);

/* dst[i] += src[i] on the device: combines per-step tally deltas of a particle-sharded run
 * (after the all-reduce of the deltas, SURVEY.md 8e). dst and src need only the 8-byte
 * alignment of a double (e.g. base + 1 element); 16-byte aligned pointers take a vector path
 * with the same result. */
int nb200_accumulate(double* dst_device, const double* src_device, size_t n);
/* The same, and src[i] = 0 afterwards (the delta buffer is ready for its next timestep). */
int nb200_accumulate_clear(double* dst_device, double* src_device, size_t n);
/* The same on a caller-supplied cudaStream_t: lets a multi-GPU host fold a reduced delta
 * into the tally beside the next timestep's transport (neutral_b200/multi.py). */
int nb200_accumulate_clear_async(double* dst_device, double* src_device, size_t n,
                                 void* cuda_stream);

/* Options: "print" (1: print the reference's "Particles" line); "pipeline" (1, default:
 * phased timestep - begin-step/classify, counting sort by next-event type and tile, event
 * loop; 0: the direct one-thread-per-history kernel on the unsorted bank); "fast_div"
 * (1, default: exact division by loop-invariant divisors through their reciprocals);
 * "tile_shift" (log2 of the sort tile edge in cells, default 8; < 0: no spatial key);
 * "length_bins" (bins of expected history length in the sort key, default 512; <= 1: none);
 * "tally_prereduce" (1: combine same-cell tally flushes of a warp with shuffles before the
 * atomic; default 0); "l2_persist" (1: the history kernel's launch carries an access-policy
 * window that keeps the staged cross-section tables persisting in L2; 2: a window over the
 * tally instead, measured slower; default 0); "stage_overlap" (1, default: the density tile
 * maps and target-edge rows are staged on a side stream beside the sort phase); 
 * "history_smem_pad" (bytes of unused dynamic shared memory per CTA of the history kernel:
 * an occupancy / carve-out probe, default 0).
 * "device_inject" (1, default: inject_particles generates the bank on the device with the
 * bit-exact sin/cos of nb_sincos.cuh; 0: on the host with libm, then uploads it);
 * "defer_finish" (1: solve_transport_2d returns as soon as the timestep is enqueued on the
 * stream; the counts are collected - and the reference's "Particles" line printed - by
 * nb200_solve_finish; up to 4 timesteps of a bank may be in flight, so a host can keep the
 * GPU fed without a round trip per timestep; default 0).
 * "ngpus" (GPUs the NEXT inject_particles / nb200_bank_create shards its bank over, starting
 * with the current device; 0/1: one; environment NB200_NGPUS=<n>|all sets the default);
 * "collective" (how a sharded run combines its tally: 1, default: the library's own
 * peer-memory reduce-scatter kernel, csrc/nb_group.cuh; 0: NCCL reduce-scatter, bound at run
 * time; environment NB200_COLLECTIVE=nccl); "reduce_ctas" (grid of that kernel);
 * "tally_reduce_every" (timesteps a sharded run deposits into its private buffers between
 * reduce-scatters: 0, default: only when the tally is looked at - validate, downloads,
 * nb200_tally_sync -, which is all the reference's driver needs; 1: every timestep, beside the
 * next timestep's transport; n: every n timesteps);
 * "host_mirror" (see inject_particles); "headroom_pct" (extra bank slots in percent).
 * "stagger_at" / "stagger_share" / "stagger_min" (an experiment kept for the record, off: when
 * the collision class is at least stagger_min per mille of the live bank and fits the first wave
 * of CTAs, stagger_share percent of its CTAs are dispatched behind the first stagger_at percent
 * of the streamer CTAs; measured slower than class order, DESIGN.md 5).
 * "step_graph" (1, default: the timestep's kernels, memsets and event records are recorded
 * on a capture stream of the library's own, the device's executable CUDA graph is updated in
 * place with the step's parameters and submitted as ONE launch on the library's stream - same
 * kernels, same order, same results; 0: the ~23 driver calls are issued one by one. The
 * occupancy / L2 probes "history_smem_pad", "l2_persist" and "pipeline" = 0 always take the
 * call-by-call path).
 * "tally_batches" (0, default: off; 2..64: the NEXT inject_particles / nb200_bank_create makes a
 * bank whose tally carries B independent batch estimates, section 6; environment
 * NB200_TALLY_BATCHES=<B> sets the default; 1 is refused: one batch has no spread).
 * "tally_prereduce" = 1 implies "fast_div" = 1 (it has no separate IEEE-division build); it
 * is an experiment kept for the record (measured slower): its peer mask is the opportunistic
 * __activemask() pattern, which CUDA does not guarantee to be the converged set.
 * Options are process-wide defaults; nb200_bank_set_option overrides one for one bank (the
 * creation-time options ngpus / host_mirror / headroom_pct / device_inject / tally_batches
 * apply when the bank is created; nb200_bank_set_option refuses tally_batches, and pipeline = 0
 * or tally_prereduce = 1 on a bank with tally batches). Returns the previous value, or NB200_BAD_OPTION for an unknown name or a value
 * outside the option's range (nb200_last_error says which). */
int nb200_set_option(const char* name, int value);
int nb200_get_option(const char* name);
int nb200_bank_set_option(nb200_particle_soa* particles, const char* name, int value);
/* Completes a timestep enqueued under defer_finish=1: waits for the stream and ADDS the
 * step's counts to *facet_events / *collision_events (either may be null), like
 * omp3/neutral.c:202-203. */
int nb200_solve_finish(uint64_t* facet_events, uint64_t* collision_events);
/* The same for a named bank (nb200_solve_finish refers to the bank that enqueued last): collects
 * the OLDEST pending timestep; nb200_bank_pending says how many are pending. */
int nb200_bank_solve_finish(nb200_particle_soa* particles, uint64_t* facet_events,
                            uint64_t* collision_events);
int nb200_bank_pending(nb200_particle_soa* particles);

/* Statistics of the most recent solve_transport_2d: out[0..4] = facets, collisions,
 * particles processed, census events, deaths; out[5] = kernels launched by that call;
 * out[6] = nanoseconds the step's history kernel took on the stream (CUDA events);
 * out[7] = nanoseconds of the sort phase in front of it. */
int nb200_last_step_stats(uint64_t out[8]);
/* Kernels launched by this library since load (monotonic). */
uint64_t nb200_kernel_launches(void);

/* ------------------------------------------------------------------------------------
 * 5. Particle-sharded runs (SURVEY.md 8e). Histories are independent and keyed by the GLOBAL
 *    particle index (omp3/neutral.c:632-641), so GPU g of G transports the contiguous range of
 *    omp3's thread split (omp3/neutral.c:64-74) and only the additive tally is combined: each
 *    GPU deposits into a private buffer, and one library kernel per GPU reads its slice of
 *    every peer's buffer over NVLink and folds the sum into the slice of the cumulative tally
 *    it owns (csrc/nb_group.cuh) - when the tally is looked at, or every
 *    "tally_reduce_every" timesteps beside the next timestep's transport.
 *    Two ways to get there:
 *      - one process, several GPUs: option "ngpus" / NB200_NGPUS before inject_particles.
 *        Nothing else changes for the caller (this is how `NB200_NGPUS=8 ./neutral.b200 ...`
 *        runs the reference's unmodified main.c on 8 GPUs);
 *      - one process per GPU (torchrun, MPI): nb200_set_shard + nb200_mp_init on every rank,
 *        exchange the blobs with whatever the host has (torch.distributed.all_gather, MPI),
 *        nb200_mp_connect. From then on solve_transport_2d on that GPU takes part in the group.
 *    The tally of a sharded run, like that of a single-GPU one, may be any 8-byte aligned
 *    double array (e.g. base + 1 element): the gather into it takes 16-byte accesses only
 *    when the tally is 16-byte aligned.
 * ---------------------------------------------------------------------------------- */
/* Allocates this rank's part of the group for a tally of `ncells` doubles on the current GPU
 * and writes NB200_MP_BLOB_BYTES bytes the peers need into blob_out. */
int nb200_mp_init(int nranks, int rank, size_t ncells, void* blob_out);
/* blobs = nranks * NB200_MP_BLOB_BYTES bytes, rank order. -7: a peer's memory cannot be mapped
 * (no NVLink/PCIe peer path): finalize and retry with option "collective" = 0. */
int nb200_mp_connect(const void* blobs);
int nb200_mp_finalize(void);
/* Brings the caller-visible tally up to date with everything the group has deposited
 * (all-gather of the owned slices, added to the tally; NULL = every tracked tally).
 * In a multi-process group this is a collective: every rank calls it, equally often. */
int nb200_tally_sync(double* tally_device);
/* The other GPUs of a single-process sharded bank work on replicas of the read-only inputs
 * (density, edges, tables), made when a pointer is first seen: tell the library when the
 * caller has changed such an array in place. */
int nb200_update_replicas(void);

/* ------------------------------------------------------------------------------------
 * 6. Tally batches: a relative error beside every tally cell. A bank created with option
 *    "tally_batches" = B splits its N particles into B contiguous ranges of global particle
 *    index, omp3's thread split (batch b starts at b*(N/B) + min(b, N%B) and holds
 *    n_b = N/B + (b < N%B) particles). Every deposit goes to the partial tally S_b of the
 *    depositing particle's batch; histories, counts and the bank are exactly those of the
 *    unbatched run. The caller's tally receives what the batches gained lazily, wherever a
 *    sharded run's tally would (validate, copy_buffer RECV, nb200_memcpy_* / nb200_memset_d of
 *    it, nb200_tally_sync, nb200_bank_free, and the two calls below); afterwards it equals the
 *    unbatched run's tally up to summation order. The batches belong to the first tally and
 *    mesh a timestep of the bank deposits into; a timestep into another tally or mesh flushes
 *    and starts over. With x_b = S_b * N / n_b (an independent estimate of the whole tally),
 *    m = mean of x_b, s^2 = sum_b (x_b - m)^2 / (B - 1): R = sqrt(s^2 / B) / |m|, 0 where
 *    m == 0, per cell and for the tally total.
 *    Refused (error code, or a fatal error from inject_particles / solve_transport_2d): banks
 *    sharded over several GPUs or in a multi-process group, banks that do not hold particles
 *    [0, ntotal_particles) of the timestep, B > N, nb200_bank_append, pipeline = 0 and
 *    tally_prereduce = 1, and B * nx * ny >= 2^31. The host flavour
 *    nb200_solve_transport_2d_host has no batches.
 * ---------------------------------------------------------------------------------- */
/* Flushes, then writes the B cumulative partial tallies S_b as B consecutive arrays of ncells
 * doubles (batch-major) to device memory. Returns B, or a negative code (nb200_last_error):
 * not a batched bank, no timestep deposited yet, ncells not the batches' mesh. */
int nb200_bank_tally_batches(nb200_particle_soa* particles, double* out_device, size_t ncells);
/* Flushes, then writes R of every cell to relerr_device (ncells doubles, device memory) and R of
 * the tally total to *total_relerr_host. Either may be null. Returns 0 or a negative code. */
int nb200_bank_tally_relerr(nb200_particle_soa* particles, double* relerr_device,
                            double* total_relerr_host);

/* ------------------------------------------------------------------------------------
 * 7. Track-length flux tally beside the energy-deposition tally. A bank with a flux array
 *    attached adds w * l / ntotal_particles to flux[celly * nx + cellx] for every flight
 *    segment of every later timestep: l is the segment's length in the mesh's length unit,
 *    w the weight the particle carries along it (before an absorption at its end reduces
 *    it, the weight the energy deposit uses), ntotal_particles the solve_transport_2d
 *    argument. The array accumulates over timesteps; the caller zeroes it, as the energy
 *    tally. Divided by the cell's area it is the time-integrated scalar flux per source
 *    particle. Histories, counts, the bank and the energy tally do not change.
 *    Refused with an error code: banks sharded over several GPUs or in a multi-process group,
 *    banks with tally batches (section 8 gives them a batched flux), and pipeline = 0 or
 *    tally_prereduce = 1 (the bank's effective
 *    options); with a flux array attached nb200_bank_set_option refuses those two values. A
 *    fatal error from solve_transport_2d: nx * ny differs from the attached ncells, or the
 *    process-wide options have since turned pipeline = 0 or tally_prereduce = 1 on.
 *    deallocate_data of the attached array detaches it; nb200_bank_free drops the attachment;
 *    nb200_bank_copy copies particles only. The host flavour has no flux tally.
 * ---------------------------------------------------------------------------------- */
/* Attaches flux_device (ncells doubles, device memory on the bank's GPU) to the bank, or
 * detaches the current array when flux_device is null. Returns 0, -4 when timesteps of the bank
 * are pending, or another negative code (nb200_last_error). */
int nb200_bank_set_flux_tally(nb200_particle_soa* particles, double* flux_device, size_t ncells);

/* ------------------------------------------------------------------------------------
 * 8. Flux batches: a relative error beside every flux cell. A bank with tally batches
 *    (section 6) can have a flux array attached through the call below. Its flux deposits
 *    (section 7) then go to B partial fluxes, one per particle batch of section 6, held by the
 *    library ((B + 1) * ncells doubles on the bank's GPU, allocated and zeroed when the array
 *    is attached). The attached array receives what the batches gained lazily, wherever the
 *    energy tally of a batched bank does: nb200_memcpy_* / nb200_memset_d (flushed first, then
 *    zeroed) and copy_buffer RECV of it, nb200_tally_sync(NULL or the array), nb200_bank_free,
 *    a detach, and the two calls below. Afterwards it equals the unbatched flux up to
 *    summation order. The estimator is section 6's, on the flux batches. Histories, counts,
 *    the bank and the energy tally and its batches do not change.
 *    Refused with an error code (-4: timesteps of the bank pending; -3 otherwise): a handle
 *    that is not a bank, a bank without tally batches, pipeline = 0 or tally_prereduce = 1,
 *    an array that is not device memory on the bank's GPU, ncells = 0, B * ncells >= 2^31.
 *    A null array, in this call or in nb200_bank_set_flux_tally, detaches after flushing into
 *    the old array. deallocate_data of the attached array detaches it without a flush.
 *    nb200_bank_set_option and solve_transport_2d refuse as in section 7.
 * ---------------------------------------------------------------------------------- */
/* Attaches flux_device (ncells doubles, device memory on the bank's GPU) as a batched flux with
 * the bank's B, or detaches the current array when flux_device is null. Returns 0, -4 when
 * timesteps of the bank are pending, or another negative code (nb200_last_error). */
int nb200_bank_set_batched_flux_tally(nb200_particle_soa* particles, double* flux_device,
                                      size_t ncells);
/* Flushes, then writes the B cumulative partial fluxes as B consecutive arrays of ncells doubles
 * (batch-major) to device memory. Returns B, or a negative code: no batched flux attached, no
 * timestep deposited into it yet, ncells not the attached array's. */
int nb200_bank_flux_batches(nb200_particle_soa* particles, double* out_device, size_t ncells);
/* Flushes, then writes R of every flux cell to relerr_device (ncells doubles, device memory)
 * and R of the flux total to *total_relerr_host. Either may be null. Returns 0 or a negative
 * code, as nb200_bank_flux_batches. */
int nb200_bank_flux_relerr(nb200_particle_soa* particles, double* relerr_device,
                           double* total_relerr_host);

/* What the history kernel is bound by on facet-dominated decks, measured in place: FP64
 * reductions per second the L2 retires (csrc/microbench.cu; pattern 3 = the peak, 1 = a
 * particle's mesh walk, 0 = random cells, 5 / 6 = 32 / 4 lanes on consecutive cells) into a
 * footprint of footprint_bytes, `iters` reductions per thread on 2368 x 128 threads. */
int nb200_microbench_red(int pattern, size_t footprint_bytes, int iters,
                         double* reductions_per_s);

/* Known-answer hooks on the bit-exact building blocks (device and host builds of the same
 * source). raw/unit/neglog hold 2n entries: Threefry-2x64-20(ctr={counter,0},
 * key={pkey0+i, master_key}), the (0,1] doubles, and -log of them. */
int nb200_selftest_rng_log(uint64_t pkey0, uint64_t master_key, uint64_t counter, int n,
                           uint64_t* raw_host, double* unit_host, double* neglog_host);
int nb200_selftest_log(const double* x_host, double* y_host, int n);
/* fast[i] = a/b through the kernels' reciprocal-based exact division, ieee[i] = a/b. */
int nb200_selftest_div(const double* a_host, const double* b_host, int n, double* fast_host,
                       double* ieee_host);
/* The kernels' straight-line division / reciprocal / square-root cores (csrc/nb_fastmath.cuh)
 * next to the plain operators: out_host holds 6 arrays of n doubles - core a/b, a/b, core 1/b,
 * 1/b, core sqrt|a|, sqrt|a|. */
int nb200_selftest_fastmath(const double* a_host, const double* b_host, int n, double* out_host);
int nb200_selftest_cs(const double* keys_host, const double* values_host, int nentries,
                      const double* energies_host, int n, int* index_host,
                      double* value_host);
/* Host builds (no GPU needed). */
void nb200_host_threefry2x64_20(uint64_t c0, uint64_t c1, uint64_t k0, uint64_t k1,
                                uint64_t out[2]);
double nb200_host_log(double x);
/* sin/cos as inject_particles needs them: a transliteration of glibc's __sin_fma/__cos_fma
 * (nb_sincos.cuh). Device evaluation of n host arguments; host builds of the same source;
 * and a sweep that counts the arguments on which the host build and this process's libm
 * differ in any bit (first offender in *bad_x). */
int nb200_selftest_sincos(const double* x_host, double* sin_host, double* cos_host, int n);
double nb200_host_sin(double x);
double nb200_host_cos(double x);
void nb200_host_sincos(const double* x, long long n, double* sin_out, double* cos_out);
/* Which 128-slot group of the sorted bank the event loop's CTA `cta` works on under the
 * stagger_* options (host evaluation of the kernel's own map, history.cu: dispatch_group). */
unsigned nb200_selftest_dispatch_group(unsigned cta, unsigned n_live, unsigned n_coll,
                                       int stagger_at, int stagger_share, int stagger_min);
long long nb200_selftest_host_sincos(const double* x, long long n, double* bad_x);
/* The batch of global particle `pid` among `nbatches` batches of n particles (host evaluation
 * of the history kernel's own map, nb_bank.cuh: batch_of); UINT_MAX outside 1 <= nbatches <= n,
 * pid < n < 2^31. */
unsigned nb200_selftest_batch_of(uint64_t pid, uint64_t n, int nbatches);

#ifdef __cplusplus
}
#endif

#endif /* NEUTRAL_B200_H */
