// transport.cu - the particle-history kernels of the b200 kernel set (sm_100a).
//
// Restates, as hand-written CUDA, the transport sweep of the reference omp3 kernel set:
//   handle_particles          omp3/neutral.c:43-206
//   calc_distance_to_facet    omp3/neutral.c:423-471
//   collision_event           omp3/neutral.c:209-300
//   facet_event               omp3/neutral.c:303-380
//   census_event              omp3/neutral.c:383-405
//   update_tallies            omp3/neutral.c:408-420
//   microscopic_cs_for_energy omp3/neutral.c:498-517
// Arithmetic contract: compiled with -fmad=false; expression order as in the reference
// (SURVEY.md 7.2) so that every particle field replays bit-identically.
#include "transport.cuh"
#include "nb_device.cuh"
#include "nb_sincos.cuh"

namespace nb {

// --------------------------------------------------------------------------------------
// k_history_direct: one thread follows one particle from the start of the timestep to its
// census or death. This is the straight restatement used to close parity; the phased
// pipeline in this file is measured against it.
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kHistoryThreads) k_history_direct(const StepArgs a) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long nf = 0, nc = 0, nz = 0, np = 0, nd_ = 0;

  int4 m = make_int4(0, 0, 1, 0);
  if (slot < a.n) m = a.bank.meta[slot];

  if (!m.z) {
    np = 1;
    const uint64_t pkey = a.pid0 + (uint64_t)(unsigned)m.w;
    double2 pos = a.bank.pos[slot];
    double2 dir = a.bank.dir[slot];
    const double2 ew = a.bank.ew[slot];
    double x = pos.x, y = pos.y, ox = dir.x, oy = dir.y, e = ew.x, w = ew.y;
    int cx = m.x, cy = m.y;
    int dead = 0;

    // omp3/neutral.c:103-118
    double rho = __ldg(a.density + (size_t)cy * a.nx + cx);
    double sig_s, sig_a;
    cs_lookup_pair(a, e, sig_s, sig_a);
    double nd = number_density(rho);
    double Sig_s = macroscopic(nd, sig_s);
    double Sig_a = macroscopic(nd, sig_a);
    double v = speed_of(e);
    double edep = 0.0;

    // omp3/neutral.c:122-131 (`initial` is always 1, :36)
    uint64_t counter = 0;
    double dtc = a.dt;
    double mfp = -nb_log(random_first(pkey, a.master_key, counter++), a.logt) / Sig_s;

    while (dtc > 0.0) {
      const double cell_mfp = 1.0 / (Sig_s + Sig_a);

      // calc_distance_to_facet, :423-471
      const double uxi = 1.0 / (ox * v);
      const double uyi = 1.0 / (oy * v);
      const double gx = (ox >= 0.0) ? (__ldg(a.edgex + cx + 1) - x)
                                    : ((__ldg(a.edgex + cx) - kOpenBoundCorrection) - x);
      const double gy = (oy >= 0.0) ? (__ldg(a.edgey + cy + 1) - y)
                                    : ((__ldg(a.edgey + cy) - kOpenBoundCorrection) - y);
      const double tx = gx * uxi;
      const double ty = gy * uyi;
      const bool x_facet = tx < ty;
      const double d_facet = x_facet ? (gx * v) * uxi : (gy * v) * uyi;

      const double d_coll = mfp * cell_mfp;  // :144-146
      const double d_census = v * dtc;

      if (d_coll < d_facet && d_coll < d_census) {
        // collision_event, :209-300
        nc++;
        const double sig_t = sig_s + sig_a;
        edep += deposition(w, d_coll, sig_t * kBarns, heating_response(e, sig_a, sig_t), nd);
        x += d_coll * ox;
        y += d_coll * oy;
        const double p_absorb = Sig_a / (Sig_s + Sig_a);
        double a0, a1;
        random_pair(pkey, a.master_key, counter++, a0, a1);
        if (a0 < p_absorb) {
          w *= (1.0 - p_absorb);
          if (e < kMinEnergyOfInterest) {
            dead = 1;
            nd_ = 1;
            atomicAdd(a.tally + (size_t)cy * a.nx + cx, edep * a.inv_ntotal);
            edep = 0.0;
            break;
          }
        } else {
          const double mu = 1.0 - 2.0 * a1;
          const double e_new = (e * ((kMassNo * kMassNo + (2.0 * kMassNo) * mu) + 1.0)) /
                               ((kMassNo + 1.0) * (kMassNo + 1.0));
          const double ct = 0.5 * ((kMassNo + 1.0) * sqrt(e_new / e) -
                                   (kMassNo - 1.0) * sqrt(e / e_new));
          const double st = sqrt(1.0 - ct * ct);
          const double nox = ox * ct - oy * st;
          const double noy = ox * st + oy * ct;
          ox = nox;
          oy = noy;
          e = e_new;
        }
        cs_lookup_pair(a, e, sig_s, sig_a);
        nd = number_density(rho);
        Sig_s = macroscopic(nd, sig_s);
        Sig_a = macroscopic(nd, sig_a);
        mfp = -nb_log(random_first(pkey, a.master_key, counter++), a.logt) / Sig_s;
        dtc -= d_coll / v;
        v = speed_of(e);
      } else if (d_facet < d_census) {
        // facet_event, :303-380
        nf++;
        mfp -= d_facet / cell_mfp;
        dtc -= d_facet / v;
        const double sig_t = sig_s + sig_a;
        edep += deposition(w, d_facet, sig_t * kBarns, heating_response(e, sig_a, sig_t), nd);
        atomicAdd(a.tally + (size_t)cy * a.nx + cx, edep * a.inv_ntotal);
        edep = 0.0;
        x += d_facet * ox;
        y += d_facet * oy;
        if (x_facet) {
          if (ox > 0.0) {
            if (cx >= a.nx - 1) ox = -ox; else cx++;
          } else if (ox < 0.0) {
            if (cx <= 0) ox = -ox; else cx--;
          }
        } else {
          if (oy > 0.0) {
            if (cy >= a.ny - 1) oy = -oy; else cy++;
          } else if (oy < 0.0) {
            if (cy <= 0) oy = -oy; else cy--;
          }
        }
        rho = __ldg(a.density + (size_t)cy * a.nx + cx);
        nd = number_density(rho);
        Sig_s = macroscopic(nd, sig_s);
        Sig_a = macroscopic(nd, sig_a);
      } else {
        // census_event, :383-405
        nz++;
        x += d_census * ox;
        y += d_census * oy;
        mfp -= d_census / cell_mfp;
        const double sig_t = sig_s + sig_a;
        edep += deposition(w, d_census, sig_t * kBarns, heating_response(e, sig_a, sig_t), nd);
        atomicAdd(a.tally + (size_t)cy * a.nx + cx, edep * a.inv_ntotal);
        dtc = 0.0;
        break;
      }
    }

    a.bank.pos[slot] = make_double2(x, y);
    a.bank.dir[slot] = make_double2(ox, oy);
    a.bank.ew[slot] = make_double2(e, w);
    a.bank.tm[slot] = make_double2(dtc, mfp);
    a.bank.meta[slot] = make_int4(cx, cy, dead, m.w);
    if (a.p_facets) a.p_facets[m.w] += nf;
    if (a.p_collisions) a.p_collisions[m.w] += nc;
    if (a.p_census) a.p_census[m.w] += nz;
  }

  flush_totals(a.totals, nf, nc, np, nz, nd_);
}

// --------------------------------------------------------------------------------------
// k_inject: inject_particles (omp3/neutral.c:560-630) on the device, straight into the packed
// bank. Particle kk of the global bank draws its position from Threefry(ctr={0,0},
// key={kk,0}) (:581-584) and its angle from ctr={1,0} (:611-614); cos/sin replay glibc's
// operation sequence (nb_sincos.cuh), so the bank equals the host-injected one bit for bit.
// --------------------------------------------------------------------------------------

// First cell whose half-open interval [edge[c], edge[c+1]) holds v; 0 when there is none -
// what the reference's linear scan over the cells leaves behind (:590-603), by bisection.
__device__ __forceinline__ int locate_cell(const double* __restrict__ edge, int ncells,
                                           double v) {
  if (!(v >= __ldg(edge))) return 0;
  int lo = 0, hi = ncells;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (v >= __ldg(edge + mid)) lo = mid; else hi = mid;
  }
  return (v >= __ldg(edge + lo) && v < __ldg(edge + lo + 1)) ? lo : 0;
}

__global__ void __launch_bounds__(256) k_inject(BankView b, int count, uint64_t first,
                                                InjectArgs ia, const SinCosTable* sct) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= count) return;
  const uint64_t kk = first + (uint64_t)s;
  double r0, r1;
  random_pair(kk, 0, 0, r0, r1);
  const double x = ia.left + r0 * ia.width;
  const double y = ia.bottom + r1 * ia.height;
  const int cx = locate_cell(ia.edgex, ia.nx, x);
  const int cy = locate_cell(ia.edgey, ia.ny, y);
  random_pair(kk, 0, 1, r0, r1);
  const double theta = 2.0 * 3.14159265358979323846 * r0;
  b.pos[s] = make_double2(x, y);
  b.dir[s] = make_double2(nb_cos(theta, sct), nb_sin(theta, sct));
  b.ew[s] = make_double2(ia.initial_energy, 1.0);
  b.tm[s] = make_double2(ia.dt, 0.0);
  b.meta[s] = make_int4(cx, cy, 0, s);
}

__global__ void k_selftest_sincos(const double* x, double* s, double* c, int n,
                                  const SinCosTable* sct) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  s[i] = nb_sin(x[i], sct);
  c[i] = nb_cos(x[i], sct);
}

// --------------------------------------------------------------------------------------
// Boundary conversions between the packed-pair bank and the reference's two layouts.
// --------------------------------------------------------------------------------------
__global__ void k_import_soa(BankView b, SoaView s, int n, int origin0) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  b.pos[i] = make_double2(s.x[i], s.y[i]);
  b.dir[i] = make_double2(s.omega_x[i], s.omega_y[i]);
  b.ew[i] = make_double2(s.energy[i], s.weight[i]);
  b.tm[i] = make_double2(s.dt_to_census[i], s.mfp_to_collision[i]);
  b.meta[i] = make_int4(s.cellx[i], s.celly[i], s.dead[i], origin0 + i);
}

// Writes slot i to position meta.w (injection order), whatever the bank order is.
__global__ void k_export_soa(BankView b, SoaView s, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int4 m = b.meta[i];
  const double2 pos = b.pos[i], dir = b.dir[i], ew = b.ew[i], tm = b.tm[i];
  const int o = m.w;
  s.x[o] = pos.x;
  s.y[o] = pos.y;
  s.omega_x[o] = dir.x;
  s.omega_y[o] = dir.y;
  s.energy[o] = ew.x;
  s.weight[o] = ew.y;
  s.dt_to_census[o] = tm.x;
  s.mfp_to_collision[o] = tm.y;
  s.cellx[o] = m.x;
  s.celly[o] = m.y;
  s.dead[o] = m.z;
}

// AoS record of the omp3 kernel set (neutral_data.h:66-79): 8 doubles, 3 ints, 4 pad bytes.
struct AosParticle {
  double x, y, omega_x, omega_y, energy, weight, dt_to_census, mfp_to_collision;
  int cellx, celly, dead, pad_;
};
static_assert(sizeof(AosParticle) == 80, "AoS particle must be 80 bytes");

__global__ void k_import_aos(BankView b, const AosParticle* __restrict__ p, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double2* q = reinterpret_cast<const double2*>(p + i);
  b.pos[i] = q[0];
  b.dir[i] = q[1];
  b.ew[i] = q[2];
  b.tm[i] = q[3];
  const int4 t = *reinterpret_cast<const int4*>(q + 4);
  b.meta[i] = make_int4(t.x, t.y, t.z, i);
}

__global__ void k_export_aos(BankView b, AosParticle* __restrict__ p, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int4 m = b.meta[i];
  double2* q = reinterpret_cast<double2*>(p + m.w);
  q[0] = b.pos[i];
  q[1] = b.dir[i];
  q[2] = b.ew[i];
  q[3] = b.tm[i];
  *reinterpret_cast<int4*>(q + 4) = make_int4(m.x, m.y, m.z, 0);
}

// --------------------------------------------------------------------------------------
// Device self-tests of the bit-exact building blocks (used by tests/ through the C-ABI).
// --------------------------------------------------------------------------------------
__global__ void k_selftest_rng_log(uint64_t pkey0, uint64_t master_key, uint64_t counter,
                                   int n, const LogTable* logt, uint64_t* raw,
                                   double* unit, double* neglog) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t o0, o1;
  threefry2x64_20(counter, 0, pkey0 + i, master_key, o0, o1);
  raw[2 * i] = o0;
  raw[2 * i + 1] = o1;
  unit[2 * i] = u64_to_unit(o0);
  unit[2 * i + 1] = u64_to_unit(o1);
  neglog[2 * i] = -nb_log(unit[2 * i], logt);
  neglog[2 * i + 1] = -nb_log(unit[2 * i + 1], logt);
}

__global__ void k_selftest_log(const double* x, double* y, int n, const LogTable* logt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = nb_log(x[i], logt);
}

// Both lookups side by side: the staged one (bucket index, what the pipeline uses) must find
// the interval of the plain bisection; a disagreement is reported as index -1.
__global__ void k_selftest_cs(const double* keys, const double* vals, int n_entries,
                              CsStage staged, const double* e, int n, int* ind, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int b = cs_bracket(keys, n_entries, e[i]);
  const int bs = cs_bracket_staged(staged, e[i]);
  const double2 p0 = staged.kv[bs], p1 = staged.kv[bs + 1];
  const double v_staged = p0.y + ((e[i] - p0.x) / (p1.x - p0.x)) * (p1.y - p0.y);
  const double v_plain = cs_interp(keys, vals, b, e[i]);
  const bool agree = b == bs && double_to_bits(v_staged) == double_to_bits(v_plain);
  ind[i] = agree ? bs : -1;
  out[i] = v_staged;
}

// dst += src over the tally mesh (combining per-step tally deltas of a sharded run). 16-byte
// accesses when both pointers allow them, a scalar loop when either is only 8-byte aligned.
__global__ void k_accumulate(double* __restrict__ dst, const double* __restrict__ src,
                             size_t n) {
  if ((((uintptr_t)dst | (uintptr_t)src) & 15) != 0) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
      dst[i] += src[i];
    return;
  }
  size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 2;
  const size_t stride = (size_t)gridDim.x * blockDim.x * 2;
  for (; i + 1 < n; i += stride) {
    double2 d = *reinterpret_cast<double2*>(dst + i);
    const double2 s = *reinterpret_cast<const double2*>(src + i);
    d.x += s.x;
    d.y += s.y;
    *reinterpret_cast<double2*>(dst + i) = d;
  }
  if (i < n) dst[i] += src[i];
}

// dst += src; src = 0: folds a reduced per-step delta into the cumulative tally and leaves the
// delta buffer ready for its next timestep in the same pass.
__global__ void k_accumulate_clear(double* __restrict__ dst, double* __restrict__ src, size_t n) {
  if ((((uintptr_t)dst | (uintptr_t)src) & 15) != 0) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
      dst[i] += src[i];
      src[i] = 0.0;
    }
    return;
  }
  size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 2;
  const size_t stride = (size_t)gridDim.x * blockDim.x * 2;
  for (; i + 1 < n; i += stride) {
    double2 d = *reinterpret_cast<double2*>(dst + i);
    const double2 s = *reinterpret_cast<const double2*>(src + i);
    d.x += s.x;
    d.y += s.y;
    *reinterpret_cast<double2*>(dst + i) = d;
    *reinterpret_cast<double2*>(src + i) = make_double2(0.0, 0.0);
  }
  if (i < n) {
    dst[i] += src[i];
    src[i] = 0.0;
  }
}

// --------------------------------------------------------------------------------------
// Launch wrappers
// --------------------------------------------------------------------------------------
static inline int blocks_for(int n, int threads) { return (n + threads - 1) / threads; }

int launch_history_direct(const StepArgs& a, cudaStream_t st) {
  if (a.n <= 0) return 0;
  k_history_direct<<<blocks_for(a.n, kHistoryThreads), kHistoryThreads, 0, st>>>(a);
  return 1;
}

int launch_import_soa(BankView b, SoaView s, int n, int origin0, cudaStream_t st) {
  if (n <= 0) return 0;
  k_import_soa<<<blocks_for(n, 256), 256, 0, st>>>(b, s, n, origin0);
  return 1;
}

int launch_export_soa(BankView b, SoaView s, int n, cudaStream_t st) {
  if (n <= 0) return 0;
  k_export_soa<<<blocks_for(n, 256), 256, 0, st>>>(b, s, n);
  return 1;
}

int launch_import_aos(BankView b, const void* aos, int n, cudaStream_t st) {
  if (n <= 0) return 0;
  k_import_aos<<<blocks_for(n, 256), 256, 0, st>>>(b, (const AosParticle*)aos, n);
  return 1;
}

int launch_export_aos(BankView b, void* aos, int n, cudaStream_t st) {
  if (n <= 0) return 0;
  k_export_aos<<<blocks_for(n, 256), 256, 0, st>>>(b, (AosParticle*)aos, n);
  return 1;
}

int launch_inject(BankView b, int count, uint64_t first, const InjectArgs& ia,
                  const SinCosTable* sct, cudaStream_t st) {
  if (count <= 0) return 0;
  k_inject<<<(count + 255) / 256, 256, 0, st>>>(b, count, first, ia, sct);
  return 1;
}

int launch_selftest_sincos(const double* x, double* s, double* c, int n, const SinCosTable* sct,
                           cudaStream_t st) {
  k_selftest_sincos<<<(n + 255) / 256, 256, 0, st>>>(x, s, c, n, sct);
  return 1;
}

int launch_accumulate(double* dst, const double* src, size_t n, cudaStream_t st) {
  if (n == 0) return 0;
  k_accumulate<<<148 * 8, 256, 0, st>>>(dst, src, n);
  return 1;
}

int launch_accumulate_clear(double* dst, double* src, size_t n, cudaStream_t st) {
  if (n == 0) return 0;
  k_accumulate_clear<<<148 * 8, 256, 0, st>>>(dst, src, n);
  return 1;
}

int launch_selftest_rng_log(uint64_t pkey0, uint64_t master_key, uint64_t counter, int n,
                            const LogTable* logt, uint64_t* raw, double* unit,
                            double* neglog, cudaStream_t st) {
  k_selftest_rng_log<<<blocks_for(n, 256), 256, 0, st>>>(pkey0, master_key, counter, n, logt,
                                                         raw, unit, neglog);
  return 1;
}

int launch_selftest_log(const double* x, double* y, int n, const LogTable* logt,
                        cudaStream_t st) {
  k_selftest_log<<<blocks_for(n, 256), 256, 0, st>>>(x, y, n, logt);
  return 1;
}

int launch_selftest_cs(const double* keys, const double* vals, int n_entries, CsStage staged,
                       const double* e, int n, int* ind, double* out, cudaStream_t st) {
  k_selftest_cs<<<blocks_for(n, 256), 256, 0, st>>>(keys, vals, n_entries, staged, e, n, ind,
                                                    out);
  return 1;
}

}  // namespace nb
