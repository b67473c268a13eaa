/* Test infrastructure: E_pair(i,j), the lowest energy of a structure containing the pair (i,j), restated in plain C on the CPU
 * oracle's own energy functions (oracle/orc_fold.c): the oracle's single-strand MFE fill (c, fML), then an outside recursion
 * written out directly -- right-hand parts RF / RU of every cell by an explicit loop over the closing pair, no row
 * accumulators -- so that it shares nothing with the device kernel but the recursion's definition.  O(n^3) time, O(n^2) memory.
 * Built and loaded by tests/pair_mfe_ref.py. */
#include "../oracle/orc_fold.c"

/* e_pair: n*n ints, [(i-1)*n + (j-1)] for i < j, INF elsewhere.  nopair: NULL or n bytes.  Returns the MFE. */
int orc_pair_mfe(const orc_params *P, const char *seq, int n, const unsigned char *nopair, int *e_pair) {
  ctx_t X;
  ctx_init(&X, P, seq, n, 0, nopair);
  const int W = n + 2;
  int *S = X.S;
  const size_t WW = (size_t)W * W;
  int *c = malloc(sizeof(int) * WW), *fML = malloc(sizeof(int) * WW), *CO = malloc(sizeof(int) * WW), *G = malloc(sizeof(int) * WW);
  int *RF = malloc(sizeof(int) * WW), *RU = malloc(sizeof(int) * WW);
  int *f5 = calloc(n + 2, sizeof(int)), *f3 = calloc(n + 2, sizeof(int));
#define C(i, j) c[(size_t)(i) * W + (j)]
#define M(i, j) fML[(size_t)(i) * W + (j)]
#define O(i, j) CO[(size_t)(i) * W + (j)]
#define GG(i, j) G[(size_t)(i) * W + (j)]
  for (size_t k = 0; k < WW; k++) { c[k] = INF; fML[k] = INF; CO[k] = INF; G[k] = INF; RF[k] = INF; RU[k] = INF; }
  for (int k = 0; k < n * n; k++) e_pair[k] = INF;
  /* inside: the single-strand branch of orc_mfe */
  for (int i = n; i >= 1; i--)
    for (int j = i + 1; j <= n; j++) {
      int t = ptype(&X, i, j), e = INF;
      if (t) {
        e = E_hairpin(P, j - i - 1, t, S[i + 1], S[j - 1], X.seqU, i, j);
        int pmax = MIN2(j - 2, i + MAXLOOP + 1);
        for (int p = i + 1; p <= pmax; p++) {
          int minq = j - i + p - MAXLOOP - 2;
          if (minq < p + 1) minq = p + 1;
          for (int q = j - 1; q >= minq; q--) {
            int t2 = ptype(&X, p, q);
            if (!t2 || C(p, q) >= INF) continue;
            e = MIN2(e, C(p, q) + E_intloop(P, p - i - 1, j - q - 1, t, RTYPE[t2], S[i + 1], S[j - 1], S[p - 1], S[q + 1]));
          }
        }
        int dec = INF;
        for (int u = i + 2; u <= j - 1; u++)
          if (M(i + 1, u - 1) < INF && M(u, j - 1) < INF) dec = MIN2(dec, M(i + 1, u - 1) + M(u, j - 1));
        if (dec < INF) e = MIN2(e, dec + P->MLclosing + E_mlstem(P, RTYPE[t], S[j - 1], S[i + 1]));
        if (e > INF) e = INF;
      }
      C(i, j) = e;
      int m = INF;
      if (e < INF && i > 1 && j < n) m = e + E_mlstem(P, t, S[i - 1], S[j + 1]);
      if (M(i + 1, j) < INF) m = MIN2(m, M(i + 1, j) + P->MLbase);
      if (M(i, j - 1) < INF) m = MIN2(m, M(i, j - 1) + P->MLbase);
      for (int u = i + 1; u <= j; u++)
        if (M(i, u - 1) < INF && M(u, j) < INF) m = MIN2(m, M(i, u - 1) + M(u, j));
      M(i, j) = m;
    }
  for (int j = 1; j <= n; j++) {
    int e = f5[j - 1];
    for (int i = 1; i < j; i++) { int t = ptype(&X, i, j); if (t && C(i, j) < INF) e = MIN2(e, f5[i - 1] + C(i, j) + ext_stem(&X, i, j, t)); }
    f5[j] = e;
  }
  for (int i = n; i >= 1; i--) {
    int e = f3[i + 1];
    for (int j = i + 1; j <= n; j++) { int t = ptype(&X, i, j); if (t && C(i, j) < INF) e = MIN2(e, C(i, j) + ext_stem(&X, i, j, t) + f3[j + 1]); }
    f3[i] = e;
  }
  /* outside, longest pairs first */
  for (int d = n - 1; d >= 1; d--) {
    /* RF(i,j) / RU(i,j): best closing pair (i,q) of a multiloop whose stem ends at j, with fML(j+1,q-1) / only unpaired bases between */
    for (int i = 1; i + d <= n; i++) {
      const int j = i + d;
      int rf = INF, ru = INF;
      for (int q = j + 1; q <= n; q++) {
        if (GG(i, q) >= INF) continue;
        if (M(j + 1, q - 1) < INF) rf = MIN2(rf, GG(i, q) + M(j + 1, q - 1));
        ru = MIN2(ru, GG(i, q) + P->MLbase * (q - 1 - j));
      }
      RF[(size_t)i * W + j] = rf;
      RU[(size_t)i * W + j] = ru;
    }
    for (int i = 1; i + d <= n; i++) {
      const int j = i + d, t = ptype(&X, i, j);
      if (!t || C(i, j) >= INF) continue;
      int e = f5[i - 1] + ext_stem(&X, i, j, t) + f3[j + 1];
      for (int p = i - 1; p >= 1 && i - p - 1 <= MAXLOOP; p--)
        for (int q = j + 1; q <= n && (i - p - 1) + (q - j - 1) <= MAXLOOP; q++) {
          if (O(p, q) >= INF) continue;
          e = MIN2(e, O(p, q) + E_intloop(P, i - p - 1, q - j - 1, ptype(&X, p, q), RTYPE[t], S[p + 1], S[q - 1], S[i - 1], S[j + 1]));
        }
      if (i > 1 && j < n) {
        int best = INF;
        for (int p = 1; p <= i - 1; p++) {
          const int rf = RF[(size_t)p * W + j], ru = RU[(size_t)p * W + j], lf = M(p + 1, i - 1);
          if (rf < INF) best = MIN2(best, P->MLbase * (i - 1 - p) + rf);
          if (lf < INF && rf < INF) best = MIN2(best, lf + rf);
          if (lf < INF && ru < INF) best = MIN2(best, lf + ru);
        }
        if (best < INF) e = MIN2(e, best + E_mlstem(P, t, S[i - 1], S[j + 1]));
      }
      if (e >= INF) continue;
      O(i, j) = e;
      GG(i, j) = e + P->MLclosing + E_mlstem(P, RTYPE[t], S[j - 1], S[i + 1]);
      e_pair[(size_t)(i - 1) * n + (j - 1)] = C(i, j) + e;
    }
  }
  const int mfe = f5[n];
#undef C
#undef M
#undef O
#undef GG
  free(c); free(fML); free(CO); free(G); free(RF); free(RU); free(f5); free(f3);
  ctx_free(&X);
  return mfe;
}
