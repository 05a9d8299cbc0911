/* tests/oracle_constraint.c -- the constraint part of `mjx.forward`'s Data from the float64 oracle, for the tests of the
 * contact outputs (tests/contact_util.py).  Test infrastructure: it compiles oracle/mjstep.c into the same translation unit,
 * so it reuses the oracle's forward() and its row data unchanged, and adds one export. */
#include "../oracle/mjstep.c"

/* One `mjx.forward` like oracle_forward, with the constraint part of its Data at the accepted qacc (MJX's solver finish:
 * Jaref = J qacc - aref, efc_force = -D Jaref on the rows where Jaref < 0, else 0), or at `qacc_at` [nv] when that is
 * given (the same rows and parameters, another acceleration; qacc still returns the solver's):
 *   efc_force [nefc] in make_constraint's row order (the limit rows, then four pyramid rows per active slot, slot order),
 *   qfrc_constraint [nv] = efc_J^T efc_force,
 *   con_force [ncon][3] per slot: the force in the contact frame decoded from its pyramid rows as mju_decodePyramid does
 *   (normal = sum f, tangent i = mu (f[2i] - f[2i+1])); zeros for an inactive slot.
 * con_dist / con_pos / con_frame per slot as in oracle_forward; *nlim = limit rows.  Any output may be NULL. */
int oracle_forward_constraint(const omodel *m, const double *qpos, const double *qvel, const double *warm, const double *qacc_at, double *qacc,
                              double *con_dist, double *con_pos, double *con_frame, double *efc_force, double *qfrc_constraint,
                              double *con_force, int *nefc, int *nlim) {
  odata *d = calloc(1, sizeof(odata));
  for (int i = 0; i < m->nq; i++) d->qpos[i] = (real)qpos[i];
  for (int i = 0; i < m->nv; i++) { d->qvel[i] = (real)qvel[i]; d->qacc_warmstart[i] = warm ? (real)warm[i] : (real)0; }
  forward(m, d);
  real *f = calloc(d->nefc + 1, sizeof(real));
  for (int r = 0; r < d->nefc; r++) {
    real jaref = -d->efc_aref[r];
    for (int i = 0; i < m->nv; i++) jaref += d->efc_J[r][i] * (qacc_at ? (real)qacc_at[i] : d->qacc[i]);
    f[r] = jaref < 0 ? -d->efc_D[r] * jaref : (real)0;
  }
  int nactive = 0;
  for (int c = 0; c < m->ncon; c++) nactive += d->con_dist[c] < 0;
  const int nl = d->nefc - 4 * nactive;
  if (qacc) for (int i = 0; i < m->nv; i++) qacc[i] = d->qacc[i];
  if (con_dist) for (int c = 0; c < m->ncon; c++) con_dist[c] = d->con_dist[c];
  if (con_pos) for (int c = 0; c < m->ncon; c++) for (int k = 0; k < 3; k++) con_pos[3*c+k] = d->con_pos[c][k];
  if (con_frame) for (int c = 0; c < m->ncon; c++) for (int k = 0; k < 9; k++) con_frame[9*c+k] = d->con_frame[c][k];
  if (efc_force) for (int r = 0; r < d->nefc; r++) efc_force[r] = f[r];
  if (qfrc_constraint) for (int i = 0; i < m->nv; i++) {
    real s = 0;
    for (int r = 0; r < d->nefc; r++) s += d->efc_J[r][i] * f[r];
    qfrc_constraint[i] = s;
  }
  if (con_force) {
    int r = nl;
    for (int c = 0; c < m->ncon; c++) {
      for (int k = 0; k < 3; k++) con_force[3*c+k] = 0;
      if (!(d->con_dist[c] < 0)) continue;
      const int g1 = d->con_g1[c], g2 = d->con_g2[c];
      const real mu = (real)(m->geom_friction[g1][0] > m->geom_friction[g2][0] ? m->geom_friction[g1][0] : m->geom_friction[g2][0]);
      con_force[3*c] = f[r] + f[r+1] + f[r+2] + f[r+3];
      con_force[3*c+1] = mu * (f[r] - f[r+1]);
      con_force[3*c+2] = mu * (f[r+2] - f[r+3]);
      r += 4;
    }
  }
  if (nefc) *nefc = d->nefc;
  if (nlim) *nlim = nl;
  free(f);
  free(d);
  count_flush();
  return 0;
}

