// history.cu - the event loop of the b200 kernel set (sm_100a): phase P4 of pipeline.cu.
//
// k_history follows every live particle of the sorted bank from the first event of the
// timestep to its census or death. It restates the loop of handle_particles
// (omp3/neutral.c:134-197) and the three event functions
//   collision_event  omp3/neutral.c:209-300     facet_event   omp3/neutral.c:303-380
//   census_event     omp3/neutral.c:383-405     (+ :408-420, :423-471, :474-495, :498-517)
// with these differences in HOW, none in WHAT is computed:
//
//  * everything that is invariant between two events of one kind lives in registers and is
//    recomputed - with the reference's own expression - only when one of its inputs changes
//    (energy: collisions; density: tile crossings), so the facet iteration is ~25 FP64
//    operations instead of the reference's ~150 including 7 divides;
//  * divisions by the two loop-invariant divisors of a facet (speed, cell mean free path)
//    go through their correctly rounded reciprocals with a Markstein correction - the IEEE
//    quotient, bit for bit (nb_device.cuh: div_by_known);
//  * the cell step/reflect logic (:332-368) is computed on the crossed axis only, without
//    the reference's four-way branch, so a warp does not serialise over directions;
//  * the two edges a particle is heading for are carried in registers and only the crossed
//    axis reloads its next edge - from the staged edge rows (far / near edge per axis, the
//    open-bound correction pre-applied), issued before the event's arithmetic, consumed after;
//  * the density of the entered cell comes from the per-step tile maps (stage.cu) unless the
//    tile is mixed; cross sections come from the staged tables through the bucket index;
//  * the elastic scatter (:262-297) is one basic block of branch-free division / reciprocal /
//    square-root cores (nb_fastmath.cuh, nb_history.cuh) whenever its operands are in the
//    range where those are the operators' own bits, so its independent chains interleave;
//  * nothing that only collisions need is touched by a facet: energy deposited by collisions
//    is flushed by the first facet after them (a rarely taken block), not folded into every
//    facet's deposit.
//
// Compiled with -fmad=false: the only fused operations are the explicit fma() of nb_log,
// div_by_known and the cores.
#include <type_traits>
#ifdef NB_ASSERT_BATCH_SLOT
#include <cassert>
#endif

#include "nb_history.cuh"

namespace nb {

#ifndef NB_HISTORY_MIN_BLOCKS
#define NB_HISTORY_MIN_BLOCKS 6
#endif

// State that only collisions (and the rare density change) touch is parked in shared memory,
// one slot per thread, so that the facet loop's registers hold only what a facet reads:
// energy, Sigma_s and p_absorb, the density of the cell, and the energy deposited by
// collisions since the last tally flush (omp3/neutral.c:222-225 accumulates it across
// consecutive collisions; kFlagPending says the slot is non-zero).
// -DNB_PARK_SMEM=0 keeps them in registers instead (for A/B measurements).
#ifndef NB_PARK_SMEM
#define NB_PARK_SMEM 1
#endif
struct Parked {
  double e[kHistoryThreads];
  double Sig_s[kHistoryThreads];
  double p_absorb[kHistoryThreads];
  double rho[kHistoryThreads];
  double edep[kHistoryThreads];
  int origin[kHistoryThreads];  // index in injection order: RNG key and counter slot
  unsigned nc[kHistoryThreads];  // collisions so far this step = the RNG counter state
  int slot[kHistoryThreads];     // the thread's slot of the bank (dispatch_group is not the
                                 // identity any more: parked, or the event loop spills for it)
};

#ifdef NB_HISTORY_MAXNREG  // experiments: cap the registers directly instead of through min blocks
#define NB_HISTORY_BOUNDS __maxnreg__(NB_HISTORY_MAXNREG)
#else
#define NB_HISTORY_BOUNDS __launch_bounds__(kHistoryThreads, NB_HISTORY_MIN_BLOCKS)
#endif
#ifdef NB_TRACE_WARPS
// Measurement build (never the product): every warp records when it started and ended, on
// which SM, and what it did (tools/warp_trace.py turns that into a timeline of the launch).
// NB200_DEFINES=-DNB_TRACE_WARPS NB200_LIB=libneutral_b200.trace.so python -m neutral_b200.build
__device__ unsigned long long* g_warp_trace = nullptr;  // 6 words per warp of the grid
extern "C" int nb200_debug_set_warp_trace(void* p) {
  return (int)cudaMemcpyToSymbol(g_warp_trace, &p, sizeof(p));
}
__device__ __forceinline__ unsigned long long trace_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#endif

// Which 128-slot group of the sorted bank the CTA with this index works on. CTAs are dispatched
// in index order, and the sorted bank has the collision class in front: all its warps start at
// once and hold their slots for the ~1000 dependent collisions of a collider (2.3 ms on csp),
// latency-bound and unimpressed by their neighbours, while the streamers beside them get
// what is left of the issue slots - and then have the SMs to themselves, bound by the L2's
// reduction rate with issue slots to spare (profiles/r02/warp_trace_r2b_csp_step*.txt). The
// streamers' rate is a concave function of the colliders resident beside them, so the same
// collider residency spread over the launch costs them less: when the colliders are a
// sizeable share of the bank but fit the first wave, `stagger_share` percent of their CTAs go
// out behind the first `stagger_at` percent of the streamer CTAs instead of in front. A
// permutation of whole groups inside the live prefix; no history changes.
__host__ __device__ __forceinline__ unsigned dispatch_group(const StepArgs& a, unsigned b,
                                                            unsigned n_live, unsigned n_coll) {
  if (a.stagger_at <= 0) return b;
  const unsigned T = n_live / kHistoryThreads;   // full groups of the live prefix
  const unsigned NC = n_coll / kHistoryThreads;  // groups of colliders only
  if (b >= T || NC >= T || NC > 148u * NB_HISTORY_MIN_BLOCKS ||
      (unsigned long long)n_coll * 1000ull < (unsigned long long)a.stagger_min * n_live)
    return b;
  const unsigned nB = NC * (unsigned)a.stagger_share / 100u;  // delayed collider groups
  const unsigned A = NC - nB;
  const unsigned P = A + (unsigned)(((unsigned long long)(T - NC) * (unsigned)a.stagger_at) / 100ull);
  if (b < A) return b;                  // the colliders that start with the launch
  if (b < P) return NC + (b - A);       // the first streamers
  if (b < P + nB) return A + (b - P);   // the delayed colliders
  return b;                             // the remaining streamers: NC + (P - A) + (b - P - nB)
}

// Host-side evaluation of the map (pure integer arithmetic), for tests/test_cabi.py: it has
// to be a permutation of the groups of the live prefix for any arguments.
extern "C" unsigned nb200_selftest_dispatch_group(unsigned cta, unsigned n_live, unsigned n_coll,
                                                  int stagger_at, int stagger_share,
                                                  int stagger_min) {
  StepArgs a{};
  a.stagger_at = stagger_at;
  a.stagger_share = stagger_share;
  a.stagger_min = stagger_min;
  return dispatch_group(a, cta, n_live, n_coll);
}

// kBatched (option tally_batches): every deposit goes to the partial tally of the particle's
// batch (StepArgs::batch_slab). The batch follows from the global pid, once per history; it
// is parked beside `origin` and turned into an address at each deposit.
struct ParkedBatched : Parked {
  int batch[kHistoryThreads];
};

template <bool kBatched, class P>
__device__ __forceinline__ int parked_batch(const P& park) {
  if constexpr (kBatched) return park.batch[threadIdx.x];
  else return 0;
}

// Index of `cell` of batch b in the slab (32 bits: the host refuses B * ncells >= 2^31).
__device__ __forceinline__ int batch_index(const StepArgs& a, const BatchArgs& bt, int b,
                                           int cell) {
  const int i = (int)batch_slot(b, (size_t)(unsigned)cell, bt.nbatches, (size_t)(a.nx * a.ny));
#ifdef NB_ASSERT_BATCH_SLOT  // checking build: NB200_DEFINES=-DNB_ASSERT_BATCH_SLOT
  assert(b >= 0 && b < bt.nbatches && cell >= 0 && cell < a.nx * a.ny && i >= 0 &&
         i < bt.nbatches * a.nx * a.ny);
#endif
  return i;
}

// kFlux (nb200_bank_set_flux_tally): every flight segment also adds w * length / ntotal to the
// caller's flux array, at the places the energy deposits go. The track length of collisions
// since the last flush is parked beside `edep` and flushed with it.
struct ParkedFlux : Parked {
  double flux[kHistoryThreads];
};

// kBatched and kFlux together (nb200_bank_set_batched_flux_tally): `flux` is the library's flux
// batch slab, indexed like the energy batches, and the flux parks beside the batch.
struct ParkedBatchedFlux : ParkedBatched {
  double flux[kHistoryThreads];
};

// `flux` is a kernel parameter behind the other three for the reason BatchArgs is one: a field
// appended to StepArgs would move the offsets of the parameters that follow it.
template <bool kFastDiv, bool kPreReduce, bool kBatched, bool kFlux>
__global__ void NB_HISTORY_BOUNDS
k_history(const StepArgs a, const unsigned* __restrict__ n_live, const BatchArgs bt,
          double* __restrict__ flux) {
#if NB_PARK_SMEM
  __shared__ std::conditional_t<kBatched, std::conditional_t<kFlux, ParkedBatchedFlux, ParkedBatched>,
                                std::conditional_t<kFlux, ParkedFlux, Parked>> park;
#define PARKED(name) park.name[threadIdx.x]
#define PARKED_BATCH parked_batch<kBatched>(park)
#else
  double park_e, park_Sig_s, park_p_absorb, park_rho, park_edep, park_flux;
  int park_origin, park_slot, park_batch = 0;
  unsigned park_nc;
#define PARKED(name) park_##name
#define PARKED_BATCH park_batch
#endif
  const unsigned live = n_live[0];
  unsigned nf = 0, census = 0, processed = 0, died = 0;
  PARKED(nc) = 0;
  PARKED(slot) = (int)(dispatch_group(a, blockIdx.x, live, n_live[1]) * blockDim.x + threadIdx.x);
#ifdef NB_TRACE_WARPS
  const unsigned long long trace_t0 = trace_now();
#endif

  int4 m = make_int4(0, 0, 1, 0);
  if (PARKED(slot) < (int)live) m = a.bank.meta[PARKED(slot)];

  if (!m.z) {
    processed = 1;
    double2 pos, dir, ew, tm;
    {
      const int slot = PARKED(slot);
      pos = a.bank.pos[slot];
      dir = a.bank.dir[slot];
      ew = a.bank.ew[slot];
      tm = a.bank.tm[slot];  // k_begin_step left (dt, first path sample) here
    }
    double x = pos.x, y = pos.y, ox = dir.x, oy = dir.y, w = ew.y;
    double dtc = tm.x, mfp = tm.y;
    int cx = m.x, cy = m.y;
#define NB_CELL (cy * a.nx + cx)  // tally / density index of the current cell
    // the base and index a deposit into `cell` goes to: the caller's tally, or the batch's slot
#define NB_TALLY_AT(cell) \
  (kBatched ? bt.slab : a.tally), (kBatched ? batch_index(a, bt, PARKED_BATCH, (cell)) : (cell))
    // ... and a flux deposit: the caller's array, or (batched) the batch's slot of the flux slab
#define NB_FLUX_AT(cell) flux, (kBatched ? batch_index(a, bt, PARKED_BATCH, (cell)) : (cell))
    unsigned flags = same_grid(a) ? kFlagSameGrid : 0u;
    PARKED(e) = ew.x;
    PARKED(edep) = 0.0;
    if constexpr (kFlux) PARKED(flux) = 0.0;
    PARKED(origin) = m.w;
    if constexpr (kBatched) {
      const int b = (int)batch_of((unsigned)(a.pid0 + (uint64_t)(unsigned)m.w), (unsigned)bt.n,
                                  (unsigned)bt.nbatches);
#if NB_PARK_SMEM
      park.batch[threadIdx.x] = b;
#else
      park_batch = b;
#endif
    }
    // RNG counter: k_begin_step drew counter 0 (omp3/neutral.c:129); collision number k of
    // this step draws counters 2k-1 and 2k (:235, :294), so the collision count nc is the
    // counter state.

    // ---- the density of the cell (changes on tile crossings only) ...
    double nd;
    {
      double rho = coarse_value(a, cx, cy);
      if (is_mixed_tile(rho)) {
        flags |= kFlagCoarseMixed;
        rho = fine_value(a, cx, cy);
        if (is_mixed_tile(rho)) {
          flags |= kFlagFineMixed;
          rho = __ldg(a.density + NB_CELL);
        }
      }
      PARKED(rho) = rho;
      nd = number_density(rho);
    }
    // ---- ... what follows from the energy (changes on collisions only) ...
    Derived d;
    derive(a, ew.x, nd, d, PARKED(Sig_s), PARKED(p_absorb), flags);
    double v = speed_of(ew.x);
    double v_inv = 0.0;  // recomputed on demand (kFlagInvStale is set)
    double uxi = 1.0 / (ox * v);
    double uyi = 1.0 / (oy * v);
    // ---- ... and the edges the particle is heading for (change when it crosses or turns)
    double ex = target_edge(a.edgex, cx, axis_step(ox));
    double ey = target_edge(a.edgey, cy, axis_step(oy));

    while (dtc > 0.0) {
      // calc_distance_to_facet, omp3/neutral.c:423-471
      const double gx = ex - x;
      const double gy = ey - y;
      const bool x_facet = (gx * uxi) < (gy * uyi);
      const double d_facet = ((x_facet ? gx : gy) * v) * (x_facet ? uxi : uyi);
      const double d_coll = mfp * d.cell_mfp;  // :144-146
      const double d_census = v * dtc;
      const bool collide = d_coll < d_facet && d_coll < d_census;

#ifdef NB_PROBE_COLLISION_ONLY
      // Compile-time probe (never a product build): what the event loop needs in registers
      // when it leaves at the first event that is not a collision. The kernel built on it was
      // measured and rejected, profiles/r01/experiments/session4/collide_kernel_variant.diff.
      //   NB200_DEFINES="-DNB_PROBE_COLLISION_ONLY -DNB_HISTORY_MIN_BLOCKS=7" NB200_LIB=probe.so \
      //     python -m neutral_b200.build      ->  ptxas: 72 registers, 0 bytes of spills
      if (!collide) break;
      if (false) {
#else
      if (!collide && d_facet < d_census) {
#endif
        // ---- facet_event, :303-380
        // :332-368 on the crossed axis only: step one cell, or reflect at the mesh boundary.
        // Decided first so that the next target edge is in flight during the arithmetic.
        const int c = x_facet ? cx : cy;
        const int s = axis_step_from_reciprocal(x_facet ? uxi : uyi);
        const int cn = c + s;
        const bool reflect = (unsigned)cn >= (unsigned)(x_facet ? a.nx : a.ny);
        const bool up_next = (reflect ? -s : s) >= 0;
        // next target edge from the staged rows: [axis] for the far edge, [2 + axis] for the
        // near edge with the open-bound correction already applied (:442-444, 448-450)
        const int e_row = (x_facet ? 0 : 1) + (up_next ? 0 : 2);
        const int e_at = e_row * a.edge_stride + (reflect ? c : cn) + (up_next ? 1 : 0);
        double e_next = __ldg(a.edges4 + e_at);
        nf++;
        double q_mfp, q_dtc;
        if (flags & (kFlagInvStale | kFlagPending)) {  // first facet after a collision / new density
          if (flags & kFlagPending) {
            // :222-225 accumulates the deposits of consecutive collisions and :321-327 flushes
            // them with this facet's own; here they go to the same cell as a reduction of
            // their own (the tally's tolerance covers the different rounding of the sum), which
            // keeps the parked slot out of the per-facet code
            tally_add<kPreReduce>(NB_TALLY_AT(NB_CELL), PARKED(edep) * a.inv_ntotal);
            PARKED(edep) = 0.0;
            if constexpr (kFlux) {
              tally_add<false>(NB_FLUX_AT(NB_CELL), PARKED(flux) * a.inv_ntotal);
              PARKED(flux) = 0.0;
            }
            flags &= ~kFlagPending;
          }
          if (!kFastDiv) flags &= ~kFlagInvStale;  // no reciprocals to refresh in this variant
          if (kFastDiv && (flags & kFlagInvStale)) {
            flags &= ~kFlagInvStale;
            if (fm_safe(v) & fm_safe(d.cell_mfp)) {  // both reciprocals side by side
              v_inv = rcp_core(v);
              d.cell_mfp_inv = rcp_core(d.cell_mfp);
              flags &= ~kFlagDivBad;
            }  // else: kFlagDivBad stays set and every facet takes the plain divisions
          }
        }
        // 2^-255 <= d_facet < 2^257 and both reciprocals valid, as one range test: the flag is the
        // top bit, a negative or NaN dividend has it set too
        const unsigned div_key = (unsigned)__double2hiint(d_facet) | (flags & kFlagDivBad);
        if (kFastDiv && div_key - 0x30000000u < 0x20000000u) {
          q_mfp = div_by_known_unchecked(d_facet, d.cell_mfp, d.cell_mfp_inv);
          q_dtc = div_by_known_unchecked(d_facet, v, v_inv);
        } else {
          q_mfp = d_facet / d.cell_mfp;
          q_dtc = d_facet / v;
        }
        mfp -= q_mfp;
        dtc -= q_dtc;
        // :321-327 - deposit, flush to the tally (update_tallies, :408-420), reset
        const double edep = deposition(w, d_facet, d.stb, d.heat, nd);
        tally_add<kPreReduce>(NB_TALLY_AT(NB_CELL), edep * a.inv_ntotal);
        if constexpr (kFlux) tally_add<false>(NB_FLUX_AT(NB_CELL), (w * d_facet) * a.inv_ntotal);
        x += d_facet * ox;
        y += d_facet * oy;
        // the edge load is consumed here, after the arithmetic it overlapped with
        asm volatile("" : "+d"(e_next));
        if (x_facet) ex = e_next; else ey = e_next;
        if (reflect) {
          if (x_facet) { ox = -ox; uxi = -uxi; } else { oy = -oy; uyi = -uyi; }
        } else {
          if (x_facet) cx = cn; else cy = cn;
          // :372-378 - the macroscopic cross sections follow the density of the new cell.
          // Inside a uniform coarse tile the density cannot change; otherwise the coarse map,
          // the fine map and finally the mesh itself are consulted.
          const int crossed = cn ^ c;
          if ((crossed >> kCoarseShift) || (flags & kFlagAnyMixed)) {
            double rho_new;
            bool known = false;
            if (crossed >> kCoarseShift) {
              rho_new = coarse_value(a, cx, cy);
              // common case: from one uniform coarse tile into another of the same density
              if (!(flags & kFlagAnyMixed) &&
                  double_to_bits(rho_new) == double_to_bits(PARKED(rho)))
                continue;
              if (is_mixed_tile(rho_new)) {
                flags |= kFlagCoarseMixed;
              } else {
                flags &= ~kFlagAnyMixed;
                known = true;
              }
            }
            if (!known && (flags & kFlagCoarseMixed)) {
              if ((crossed >> kTileShift) || (crossed >> kCoarseShift)) {
                rho_new = fine_value(a, cx, cy);
                if (is_mixed_tile(rho_new)) {
                  flags |= kFlagFineMixed;
                } else {
                  flags &= ~kFlagFineMixed;
                  known = true;
                }
              } else if (!(flags & kFlagFineMixed)) {
                continue;  // still inside the same uniform fine tile
              }
            }
            if (!known) rho_new = __ldg(a.density + NB_CELL);  // mixed fine tile: the mesh itself
            if (double_to_bits(rho_new) != double_to_bits(PARKED(rho))) {
              PARKED(rho) = rho_new;
              nd = number_density(rho_new);
              derive(a, PARKED(e), nd, d, PARKED(Sig_s), PARKED(p_absorb), flags);
            }
          }
        }
#ifdef NB_EXPERIMENT_NO_COLLISION
      } else if (collide) {
        break;  // experiment: how fast is a facet-only kernel (stream deck only)
      } else if (false) {
#else
      } else if (collide) {
#endif
        // ---- collision_event, :209-300
        const unsigned nc = PARKED(nc) + 1;
        PARKED(nc) = nc;
        const uint64_t pkey = a.pid0 + (uint64_t)(unsigned)PARKED(origin);
        const double e = PARKED(e);
        const double p_absorb = PARKED(p_absorb);
        const double edep = PARKED(edep) + deposition(w, d_coll, d.stb, d.heat, nd);  // :222-225
        if constexpr (kFlux) PARKED(flux) = PARKED(flux) + w * d_coll;  // before absorption
        x += d_coll * ox;
        y += d_coll * oy;
        double a0, a1;
        random_pair(pkey, a.master_key, 2ull * nc - 1ull, a0, a1);
        // The draw of :294 does not depend on the outcome of the collision: taken here, its
        // Threefry evaluation interleaves with the one above (two independent chains).
        const double neglog = -nb_log(random_first(pkey, a.master_key, 2ull * nc), a.logt);
        // :296 - the time to census shrinks by the flight time at the pre-collision speed.
        // Branch-free core beside the Threefry chains; the plain operator takes over below
        // for operands outside the core's range.
        const bool q_ok = kFastDiv && (fm_safe(d_coll) & fm_safe(v));
        double q_dtc = kFastDiv ? div_core(d_coll, v) : d_coll / v;
        if (kFastDiv && !q_ok) q_dtc = d_coll / v;
        if (a0 < p_absorb) {
          w *= (1.0 - p_absorb);
          if (e < kMinEnergyOfInterest) {  // :243-252 - the history ends here
            flags |= kFlagDead;
            tally_add<kPreReduce>(NB_TALLY_AT(NB_CELL), edep * a.inv_ntotal);
            if constexpr (kFlux) tally_add<false>(NB_FLUX_AT(NB_CELL), PARKED(flux) * a.inv_ntotal);
            break;
          }
          // Energy and direction are unchanged: the lookups of :285-291 return the values
          // already held, so nothing that depends on them needs recomputing.
          mfp = neglog / PARKED(Sig_s);
        } else {
          bool done = false;
          if (kFastDiv && (flags & kFlagSameGrid)) {
            // The whole scatter as one basic block (nb_history.cuh). It writes the state in
            // place; what the plain code below would need again if an operand turns out to be
            // outside the block's range is parked in the two slots this branch no longer
            // reads (the direction) or recomputed (the second random number).
            PARKED(Sig_s) = ox;
            PARKED(p_absorb) = oy;
            double e_new, S_s, pa;
            done = scatter_fast_same_grid(a, e, a1, nd, neglog, cx, cy, ox, oy, v, uxi, uyi, ex,
                                          ey, mfp, d, e_new, S_s, pa);
            if (done) {
              PARKED(e) = e_new;
              PARKED(Sig_s) = S_s;
              PARKED(p_absorb) = pa;
              flags |= kFlagInvStale | kFlagDivBad;
            } else {
              ox = PARKED(Sig_s);
              oy = PARKED(p_absorb);
              random_pair(pkey, a.master_key, 2ull * nc - 1ull, a0, a1);
            }
          }
          if (!done) {
            const double mu = 1.0 - 2.0 * a1;
            const double e_num = e * ((kMassNo * kMassNo + (2.0 * kMassNo) * mu) + 1.0);
            const double e_new = kFastDiv ? NB_DIV_CONST(e_num, (kMassNo + 1.0) * (kMassNo + 1.0))
                                          : e_num / ((kMassNo + 1.0) * (kMassNo + 1.0));
            const double ct = 0.5 * ((kMassNo + 1.0) * sqrt(e_new / e) -
                                     (kMassNo - 1.0) * sqrt(e / e_new));
            const double st = sqrt(1.0 - ct * ct);
            const double nox = ox * ct - oy * st;
            const double noy = ox * st + oy * ct;
            ox = nox;
            oy = noy;
            PARKED(e) = e_new;
            derive(a, e_new, nd, d, PARKED(Sig_s), PARKED(p_absorb), flags);
            v = kFastDiv ? speed_of_fast(e_new) : speed_of(e_new);
            flags |= kFlagInvStale | kFlagDivBad;  // v_inv is recomputed on demand
            uxi = 1.0 / (ox * v);
            uyi = 1.0 / (oy * v);
            ex = target_edge(a.edgex, cx, axis_step(ox));
            ey = target_edge(a.edgey, cy, axis_step(oy));
            mfp = neglog / PARKED(Sig_s);
          }
        }
        PARKED(edep) = edep;
        flags |= kFlagPending;
        dtc -= q_dtc;
      } else {
        // ---- census_event, :383-405
        census = 1;
        x += d_census * ox;
        y += d_census * oy;
        mfp -= d_census / d.cell_mfp;
        double edep = deposition(w, d_census, d.stb, d.heat, nd);
        if (flags & kFlagPending) edep = PARKED(edep) + edep;
        tally_add<kPreReduce>(NB_TALLY_AT(NB_CELL), edep * a.inv_ntotal);
        if constexpr (kFlux) {
          double fl = w * d_census;
          if (flags & kFlagPending) fl = PARKED(flux) + fl;
          tally_add<false>(NB_FLUX_AT(NB_CELL), fl * a.inv_ntotal);
        }
        dtc = 0.0;
        break;
      }
    }

    died = (flags & kFlagDead) ? 1u : 0u;
    const int slot = PARKED(slot);
    a.bank.pos[slot] = make_double2(x, y);
    a.bank.dir[slot] = make_double2(ox, oy);
    a.bank.ew[slot] = make_double2(PARKED(e), w);
    a.bank.tm[slot] = make_double2(dtc, mfp);
    const int origin = PARKED(origin);
    a.bank.meta[slot] = make_int4(cx, cy, (int)died, origin);
    if (a.p_facets) a.p_facets[origin] += nf;
    if (a.p_collisions) a.p_collisions[origin] += PARKED(nc);
    if (a.p_census) a.p_census[origin] += census;
  }
#ifdef NB_TRACE_WARPS
  if (g_warp_trace) {
    const unsigned long long wf = warp_sum(nf), wc = warp_sum(PARKED(nc)), wp = warp_sum(processed);
    if ((threadIdx.x & 31) == 0) {
      unsigned smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      unsigned long long* t = g_warp_trace + 6ull * (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5));  // dispatch order
      t[0] = trace_t0; t[1] = trace_now(); t[2] = smid; t[3] = wf; t[4] = wc; t[5] = wp;
    }
  }
#endif
  flush_totals(a.totals, nf, PARKED(nc), processed, census, died);
#undef PARKED
#undef NB_CELL
#undef NB_TALLY_AT
#undef NB_FLUX_AT
#undef PARKED_BATCH
}

static inline int blocks_for(int n, int threads) { return (n + threads - 1) / threads; }

// `pin`/`pin_bytes` (optional) name the staged cross-section block: the launch then carries an
// access-policy window that keeps it persisting in L2 (north_star phase 3), while the rest of
// the kernel's traffic - the tally atomics above all - streams through the remainder.
int launch_history(const StepArgs& a, const BatchArgs& bt, double* flux, const unsigned* n_live,
                   int n_upper, bool fast_div, bool prereduce, const void* pin, size_t pin_bytes, size_t pin_budget,
                   int smem_pad, cudaStream_t st) {
  if (n_upper <= 0) return 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(blocks_for(n_upper, kHistoryThreads));
  cfg.blockDim = dim3(kHistoryThreads);
  cfg.stream = st;
  if (smem_pad > 0) {
    // Occupancy probe (option history_smem_pad): unused dynamic shared memory that lowers
    // the number of resident CTAs per SM without touching the code.
    static int granted = 0;
    if (smem_pad > granted) {
      cudaFuncSetAttribute(k_history<true, true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_pad);
      cudaFuncSetAttribute(k_history<true, false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_pad);
      cudaFuncSetAttribute(k_history<false, false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_pad);
      cudaFuncSetAttribute(k_history<true, false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_pad);
      cudaFuncSetAttribute(k_history<false, false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_pad);
      cudaFuncSetAttribute(k_history<true, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_pad);
      cudaFuncSetAttribute(k_history<false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_pad);
      cudaFuncSetAttribute(k_history<true, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_pad);
      cudaFuncSetAttribute(k_history<false, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_pad);
      granted = smem_pad;
    }
    cfg.dynamicSmemBytes = (size_t)smem_pad;
  }
  cudaLaunchAttribute attr[1];
  if (pin && pin_bytes) {
    attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
    attr[0].val.accessPolicyWindow.base_ptr = const_cast<void*>(pin);
    attr[0].val.accessPolicyWindow.num_bytes = pin_bytes;
    // a window larger than the set-aside persists a random `hitRatio` share of its lines
    attr[0].val.accessPolicyWindow.hitRatio =
        pin_budget && pin_bytes > pin_budget ? (float)((double)pin_budget / (double)pin_bytes) : 1.0f;
    attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  // A batched bank always runs a batched variant (the host refuses prereduce for it), so the
  // step graph of a device updates in place from one of its timesteps to the next. Banks with
  // and without batches alternating on one device change the graph's kernel and re-instantiate
  // it instead, which is correct and costs an instantiation per switch. A bank with a flux
  // array attached is the same: the host refuses prereduce for it, and a batched bank's flux is
  // always batched (its `flux` is the flux batch slab).
  if (flux && bt.nbatches > 0) {
    if (fast_div)
      cudaLaunchKernelEx(&cfg, k_history<true, false, true, true>, a, n_live, bt, flux);
    else
      cudaLaunchKernelEx(&cfg, k_history<false, false, true, true>, a, n_live, bt, flux);
  } else if (flux) {
    if (fast_div)
      cudaLaunchKernelEx(&cfg, k_history<true, false, false, true>, a, n_live, bt, flux);
    else
      cudaLaunchKernelEx(&cfg, k_history<false, false, false, true>, a, n_live, bt, flux);
  } else if (bt.nbatches > 0) {
    if (fast_div)
      cudaLaunchKernelEx(&cfg, k_history<true, false, true, false>, a, n_live, bt, flux);
    else
      cudaLaunchKernelEx(&cfg, k_history<false, false, true, false>, a, n_live, bt, flux);
  } else if (prereduce) {
    cudaLaunchKernelEx(&cfg, k_history<true, true, false, false>, a, n_live, bt, flux);
  } else if (fast_div) {
    cudaLaunchKernelEx(&cfg, k_history<true, false, false, false>, a, n_live, bt, flux);
  } else {
    cudaLaunchKernelEx(&cfg, k_history<false, false, false, false>, a, n_live, bt, flux);
  }
  return 1;
}

}  // namespace nb
