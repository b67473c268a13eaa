/* Test infrastructure: probabilities of unpaired stretches as ratios of partition functions, P_u(i, u) = Z(i .. i+u-1 may not
 * pair) / Z, on the CPU oracle's own functions (oracle/orc_fold.c).  The masked inside is the single-strand branch of orc_pf's
 * inside with the nopair mask passed to ctx_init (orc_pf itself passes NULL); the pair-type table built from ptype_slow honours
 * the mask.  It shares nothing with the device formulation but the model.  Built and loaded by tests/unpaired_ref.py. */
#include <pthread.h>

#include "../oracle/orc_fold.c"

/* ln of the partition function of single strand seq (n nt) with the positions where nopair != 0 unpaired; nopair may be NULL */
double orc_masked_lnz(const orc_params *P, const char *seq, int n, const unsigned char *nopair) {
  ctx_t X;
  ctx_init(&X, P, seq, n, 0, nopair);
  const int W = n + 2;
  int *S = X.S;
  const double kT = P->kT;
  const double pf_scale = exp(185.0 / kT);
  double *scl = (double *)malloc(sizeof(double) * (n + 3));
  scl[0] = 1.0;
  for (int k = 1; k <= n + 2; k++) scl[k] = scl[k - 1] / pf_scale;
  double *qb = (double *)calloc((size_t)W * W, sizeof(double)), *qm = (double *)calloc((size_t)W * W, sizeof(double));
  double *qm1 = (double *)calloc((size_t)W * W, sizeof(double)), *q5 = (double *)calloc(n + 3, sizeof(double));
  const double xMLb = boltz(P, P->MLbase), xMLc = boltz(P, P->MLclosing);
  double *bu = (double *)malloc(sizeof(double) * (n + 3));
  bu[0] = 1.0;
  for (int k = 1; k <= n + 2; k++) bu[k] = bu[k - 1] * xMLb / pf_scale;
#define QB(i, j) qb[(size_t)(i) * W + (j)]
#define QM(i, j) qm[(size_t)(i) * W + (j)]
#define QM1(i, j) qm1[(size_t)(i) * W + (j)]
  for (int i = n; i >= 1; i--)
    for (int j = i + 1; j <= n; j++) {
      int t = ptype(&X, i, j);
      double s = 0.0;
      if (t) {
        s = X_hairpin(P, j - i - 1, t, S[i + 1], S[j - 1], X.seqU, i, j) * scl[j - i + 1];
        int pmax = MIN2(j - 2, i + MAXLOOP + 1);
        for (int p = i + 1; p <= pmax; p++) {
          int minq = j - i + p - MAXLOOP - 2;
          if (minq < p + 1) minq = p + 1;
          for (int q = j - 1; q >= minq; q--) {
            int t2 = ptype(&X, p, q);
            if (!t2) continue;
            s += QB(p, q) * X_intloop(P, p - i - 1, j - q - 1, t, RTYPE[t2], S[i + 1], S[j - 1], S[p - 1], S[q + 1]) * scl[p - i + j - q];
          }
        }
        double dec = 0.0;
        for (int u = i + 2; u <= j - 1; u++) dec += QM(i + 1, u - 1) * QM1(u, j - 1);
        s += dec * xMLc * X_mlstem(P, RTYPE[t], S[j - 1], S[i + 1]) * scl[2];
      }
      QB(i, j) = s;
      double m1 = QM1(i, j - 1) * bu[1];
      if (t && i > 1 && j < n) m1 += s * X_mlstem(P, t, S[i - 1], S[j + 1]);
      QM1(i, j) = m1;
      double m = 0.0;
      for (int u = i; u <= j; u++) m += ((u == i) ? 1.0 : bu[u - i] + QM(i, u - 1)) * QM1(u, j);
      QM(i, j) = m;
    }
  q5[0] = 1.0;
  for (int j = 1; j <= n; j++) {
    double s = q5[j - 1] * scl[1];
    for (int i = 1; i < j; i++) {
      int t = ptype(&X, i, j);
      if (t) s += q5[i - 1] * QB(i, j) * x_ext_stem(&X, i, j, t);
    }
    q5[j] = s;
  }
#undef QB
#undef QM
#undef QM1
  const double lnz = log(q5[n]) + n * log(pf_scale);
  free(scl); free(bu); free(qb); free(qm); free(qm1); free(q5); ctx_free(&X);
  return lnz;
}

typedef struct {
  const orc_params *P;
  const char *seq;
  int n, k, nthreads, tid;
  const int *is, *us;
  double lnz, *out;
} up_job;

static void *up_worker(void *arg) {
  up_job *J = (up_job *)arg;
  unsigned char *mask = (unsigned char *)calloc(J->n + 1, 1);
  for (int x = J->tid; x < J->k; x += J->nthreads) {
    memset(mask, 0, J->n);
    for (int p = J->is[x]; p < J->is[x] + J->us[x]; p++) mask[p - 1] = 1;
    J->out[x] = exp(orc_masked_lnz(J->P, J->seq, J->n, mask) - J->lnz);
  }
  free(mask);
  return NULL;
}

/* out[x] = P_u(is[x], us[x]) (1-based i, i + u - 1 <= n) for x < k, over nthreads threads */
void orc_unpaired(const orc_params *P, const char *seq, int n, int k, const int *is, const int *us, double *out, int nthreads) {
  if (nthreads < 1) nthreads = 1;
  const double lnz = orc_masked_lnz(P, seq, n, NULL);
  pthread_t th[64];
  up_job J[64];
  if (nthreads > 64) nthreads = 64;
  for (int t = 0; t < nthreads; t++) {
    J[t] = (up_job){P, seq, n, k, nthreads, t, is, us, lnz, out};
    pthread_create(&th[t], NULL, up_worker, &J[t]);
  }
  for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
}
