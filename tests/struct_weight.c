/* Test infrastructure: the Boltzmann weight of ONE secondary structure under the CPU oracle's partition-function model -- the
 * oracle's own struct_weight() (oracle/orc_fold.c: integer loop energies, smoothed dangle / mismatch factors), compiled here
 * with one exported entry point so that the oracle itself stays as it is.  Built and loaded by tests/struct_weight.py. */
#include "../oracle/orc_fold.c"

/* weight of dot-bracket `db` on single-strand `seq` (n nt); *e_out: its energy in dcal/mol.  -1.0 for an unbalanced db. */
double orc_struct_weight(const orc_params *P, const char *seq, int n, const char *db, int *e_out) {
  ctx_t X;
  ctx_init(&X, P, seq, n, 0, NULL);
  enum_t E;
  memset(&E, 0, sizeof E);
  E.X = &X; E.n = n; E.pt = (int *)calloc(n + 2, sizeof(int));
  double w = -1.0;
  if (make_pt(db, n, E.pt) == 0) w = struct_weight(&E, e_out);
  free(E.pt); ctx_free(&X);
  return w;
}

/* kT of the loaded parameter set, cal/mol */
double orc_kT(const orc_params *P) { return P->kT; }
