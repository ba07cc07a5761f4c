/*
 * flux_reference.c - TEST INFRASTRUCTURE, not product code: the reference of the track-length
 * flux tally (nb200_bank_set_flux_tally).
 *
 * flux_reference_transport_step is oracle_transport_step (oracle/neutral_oracle.c, included
 * below unchanged, with its helpers) plus one optional output: `flux` (may be NULL) receives
 * w * l * inv_ntotal for every flight segment of length l, with the weight w the particle
 * carries along it (before an absorption at its end reduces it, the `w` the energy deposit
 * uses). It is accumulated across consecutive collisions and flushed exactly where `edep` is:
 * at the next facet, at census and at death. Everything else is the oracle's loop, line for line;
 * tests/test_flux_tally_cpu.py checks that banks, counts, counters and the energy tally are
 * bit-identical to oracle_transport_step's, with and without `flux`.
 *
 * Built by tests/flux_reference.py into a temporary directory with the oracle port's flags.
 */
#include "../oracle/neutral_oracle.c"

void flux_reference_transport_step(int nx, int ny, uint64_t master_key, double dt,
                           int ntotal_particles, int pid0, int count,
                           OracleBank* bank, const double* density,
                           const double* edgex, const double* edgey,
                           const double* s_keys, const double* s_values, int s_n,
                           const double* a_keys, const double* a_values, int a_n,
                           double* tally, uint64_t* p_facets,
                           uint64_t* p_collisions, uint64_t* p_census,
                           uint64_t totals[3], double* flux) {
  uint64_t tot_f = 0, tot_c = 0, tot_p = 0;
  const double inv_ntotal = 1.0 / (double)ntotal_particles; /* :120 */

#pragma omp parallel for schedule(dynamic, 64) reduction(+ : tot_f, tot_c, tot_p)
  for (int s = 0; s < count; ++s) {
    if (bank->dead[s]) continue; /* :91-93 */
    tot_p++;

    const uint64_t pkey = (uint64_t)(pid0 + s);
    double x = bank->x[s], y = bank->y[s];
    double ox = bank->omega_x[s], oy = bank->omega_y[s];
    double e = bank->energy[s], w = bank->weight[s];
    int cx = bank->cellx[s], cy = bank->celly[s];
    int dead = 0;
    uint64_t nf = 0, nc = 0, nz = 0;

    /* :103-118 */
    double rho = density[(size_t)cy * nx + cx];
    double sig_s = oracle_cs_lookup(s_keys, s_values, s_n, e);
    double sig_a = oracle_cs_lookup(a_keys, a_values, a_n, e);
    double nd = (rho * O_AVOGADROS / O_MOLAR_MASS);
    double Sig_s = nd * sig_s * O_BARNS;
    double Sig_a = nd * sig_a * O_BARNS;
    double v = speed_of(e);
    double edep = 0.0;
    double fl = 0.0; /* weight x track length since the last flush */

    /* :122-131 - `initial` is always 1 (omp3/neutral.c:36) */
    uint64_t counter = 0;
    double r0, r1;
    double dtc = dt;
    oracle_random_pair(pkey, master_key, counter++, &r0, &r1);
    double mfp = -log(r0) / Sig_s;

    while (dtc > 0.0) { /* :134 */
      const double cell_mfp = 1.0 / (Sig_s + Sig_a);

      /* calc_distance_to_facet, :423-471 */
      const double uxi = 1.0 / (ox * v);
      const double uyi = 1.0 / (oy * v);
      const double tx = (ox >= 0.0) ? ((edgex[cx + 1]) - x) * uxi
                                    : ((edgex[cx] - O_OPEN_BOUND) - x) * uxi;
      const double ty = (oy >= 0.0) ? ((edgey[cy + 1]) - y) * uyi
                                    : ((edgey[cy] - O_OPEN_BOUND) - y) * uyi;
      const int x_facet = (tx < ty);
      double d_facet;
      if (x_facet) {
        d_facet = (ox >= 0.0) ? ((edgex[cx + 1]) - x) * v * uxi
                              : ((edgex[cx] - O_OPEN_BOUND) - x) * v * uxi;
      } else {
        d_facet = (oy >= 0.0) ? ((edgey[cy + 1]) - y) * v * uyi
                              : ((edgey[cy] - O_OPEN_BOUND) - y) * v * uyi;
      }

      const double d_coll = mfp * cell_mfp; /* :144-146 */
      const double d_census = v * dtc;

      if (d_coll < d_facet && d_coll < d_census) {
        /* collision_event, :209-300 */
        nc++;
        edep += energy_deposition(e, w, d_coll, nd, sig_a, sig_s + sig_a);
        fl += w * d_coll;
        x += d_coll * ox;
        y += d_coll * oy;
        const double p_absorb = Sig_a / (Sig_s + Sig_a);
        double a0, a1;
        oracle_random_pair(pkey, master_key, counter++, &a0, &a1);
        if (a0 < p_absorb) {
          w *= (1.0 - p_absorb);
          if (e < O_MIN_ENERGY) {
            dead = 1;
#pragma omp atomic update
            tally[(size_t)cy * nx + cx] += edep * inv_ntotal;
            edep = 0.0;
            if (flux) {
#pragma omp atomic update
              flux[(size_t)cy * nx + cx] += fl * inv_ntotal;
            }
            fl = 0.0;
            break;
          }
        } else {
          const double mu = 1.0 - 2.0 * a1;
          const double e_new =
              e * (O_MASS_NO * O_MASS_NO + 2.0 * O_MASS_NO * mu + 1.0) /
              ((O_MASS_NO + 1.0) * (O_MASS_NO + 1.0));
          const double ct = 0.5 * ((O_MASS_NO + 1.0) * sqrt(e_new / e) -
                                   (O_MASS_NO - 1.0) * sqrt(e / e_new));
          const double st = sqrt(1.0 - ct * ct);
          const double nox = (ox * ct - oy * st);
          const double noy = (ox * st + oy * ct);
          ox = nox;
          oy = noy;
          e = e_new;
        }
        sig_s = oracle_cs_lookup(s_keys, s_values, s_n, e);
        sig_a = oracle_cs_lookup(a_keys, a_values, a_n, e);
        nd = (rho * O_AVOGADROS / O_MOLAR_MASS);
        Sig_s = nd * sig_s * O_BARNS;
        Sig_a = nd * sig_a * O_BARNS;
        oracle_random_pair(pkey, master_key, counter++, &r0, &r1);
        mfp = -log(r0) / Sig_s;
        dtc -= d_coll / v;
        v = speed_of(e);
      } else if (d_facet < d_census) {
        /* facet_event, :303-380 */
        nf++;
        mfp -= (d_facet / cell_mfp);
        dtc -= (d_facet / v);
        edep += energy_deposition(e, w, d_facet, nd, sig_a, sig_s + sig_a);
#pragma omp atomic update
        tally[(size_t)cy * nx + cx] += edep * inv_ntotal;
        edep = 0.0;
        fl += w * d_facet;
        if (flux) {
#pragma omp atomic update
          flux[(size_t)cy * nx + cx] += fl * inv_ntotal;
        }
        fl = 0.0;
        x += d_facet * ox;
        y += d_facet * oy;
        if (x_facet) {
          if (ox > 0.0) {
            if (cx >= nx - 1) ox = -ox; else cx++;
          } else if (ox < 0.0) {
            if (cx <= 0) ox = -ox; else cx--;
          }
        } else {
          if (oy > 0.0) {
            if (cy >= ny - 1) oy = -oy; else cy++;
          } else if (oy < 0.0) {
            if (cy <= 0) oy = -oy; else cy--;
          }
        }
        rho = density[(size_t)cy * nx + cx];
        nd = (rho * O_AVOGADROS / O_MOLAR_MASS);
        Sig_s = nd * sig_s * O_BARNS;
        Sig_a = nd * sig_a * O_BARNS;
      } else {
        /* census_event, :383-405 */
        nz++;
        x += d_census * ox;
        y += d_census * oy;
        mfp -= (d_census / cell_mfp);
        edep += energy_deposition(e, w, d_census, nd, sig_a, sig_s + sig_a);
#pragma omp atomic update
        tally[(size_t)cy * nx + cx] += edep * inv_ntotal;
        fl += w * d_census;
        if (flux) {
#pragma omp atomic update
          flux[(size_t)cy * nx + cx] += fl * inv_ntotal;
        }
        dtc = 0.0;
        break;
      }
    }

    bank->x[s] = x;
    bank->y[s] = y;
    bank->omega_x[s] = ox;
    bank->omega_y[s] = oy;
    bank->energy[s] = e;
    bank->weight[s] = w;
    bank->dt_to_census[s] = dtc;
    bank->mfp_to_collision[s] = mfp;
    bank->cellx[s] = cx;
    bank->celly[s] = cy;
    bank->dead[s] = dead;
    if (p_facets) p_facets[s] += nf;
    if (p_collisions) p_collisions[s] += nc;
    if (p_census) p_census[s] += nz;
    tot_f += nf;
    tot_c += nc;
  }
  totals[0] += tot_f;
  totals[1] += tot_c;
  totals[2] += tot_p;
}
