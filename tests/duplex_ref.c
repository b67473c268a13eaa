/* Test infrastructure: the duplex MFE of strands a and b (ViennaRNA duplexfold's recurrence, RNAduplex) restated in plain C on the
 * CPU oracle's own energy functions (oracle/orc_fold.c), with the engine's tie rules, and a brute force that enumerates every duplex
 * chain and scores it with orc_eval on a&b.  Built and loaded by tests/duplex_ref.py.
 *
 * A duplex is a chain of pairs (k1,l1), ..., (km,lm), a[k] with b[l], k increasing, l decreasing, at most MAXLOOP unpaired
 * nucleotides between consecutive pairs.  Ties: the end cell is the first minimum over i = 1..n1 ascending, j = n2..1 descending; the
 * backtrack from (i,j) takes the first (k,l) reproducing c(i,j), k = i-1 downwards, then l = j+1 upwards. */
#include "../oracle/orc_fold.c"

/* ss: n1 + n2 + 2 chars (a-part '&' b-part NUL), or NULL.  Returns the energy, INF when no pair is possible. */
int orc_duplex(const orc_params *P, const char *a, int n1, const char *b, int n2, char *ss) {
  int *A = calloc(n1 + 2, sizeof(int)), *B = calloc(n2 + 2, sizeof(int));
  for (int i = 1; i <= n1; i++) A[i] = enc(a[i - 1]);
  for (int j = 1; j <= n2; j++) B[j] = enc(b[j - 1]);
  const int W = n2 + 2;
  int *c = malloc(sizeof(int) * (size_t)(n1 + 2) * W);
#define C(i, j) c[(size_t)(i) * W + (j)]
  int emin = INF, imin = 0, jmin = 0;
  for (int i = 1; i <= n1; i++)
    for (int j = n2; j >= 1; j--) {
      const int t = PTYPE[A[i]][B[j]];
      C(i, j) = INF;
      if (!t) continue;
      int e = P->DuplexInit + E_ext(P, t, i > 1 ? A[i - 1] : -1, j < n2 ? B[j + 1] : -1);
      for (int k = i - 1; k >= 1 && i - k - 1 <= MAXLOOP; k--)
        for (int l = j + 1; l <= n2 && (i - k - 1) + (l - j - 1) <= MAXLOOP; l++) {
          const int tk = PTYPE[A[k]][B[l]];
          if (!tk || C(k, l) >= INF) continue;
          e = MIN2(e, C(k, l) + E_intloop(P, i - k - 1, l - j - 1, tk, RTYPE[t], A[k + 1], B[l - 1], A[i - 1], B[j + 1]));
        }
      C(i, j) = e;
      const int v = e + E_ext(P, RTYPE[t], j > 1 ? B[j - 1] : -1, i < n1 ? A[i + 1] : -1);
      if (v < emin) { emin = v; imin = i; jmin = j; }
    }
  if (ss) {
    memset(ss, '.', n1 + n2 + 1);
    ss[n1] = '&';
    ss[n1 + n2 + 1] = '\0';
    int i = imin, j = jmin;
    while (emin < INF) {
      ss[i - 1] = '(';
      ss[n1 + j] = ')';
      const int t = PTYPE[A[i]][B[j]];
      int found = 0;
      for (int k = i - 1; k >= 1 && i - k - 1 <= MAXLOOP && !found; k--)
        for (int l = j + 1; l <= n2 && (i - k - 1) + (l - j - 1) <= MAXLOOP; l++) {
          const int tk = PTYPE[A[k]][B[l]];
          if (!tk || C(k, l) >= INF) continue;
          if (C(i, j) == C(k, l) + E_intloop(P, i - k - 1, l - j - 1, tk, RTYPE[t], A[k + 1], B[l - 1], A[i - 1], B[j + 1])) {
            i = k; j = l; found = 1;
            break;
          }
        }
      if (!found) break;
    }
  }
#undef C
  free(c); free(A); free(B);
  return emin;
}

typedef struct {
  const orc_params *P;
  const char *ab;  /* a then b, n1 + n2 chars */
  int n1, n2, best;
  int *A, *B;
  char *db;        /* n1 + n2 chars + NUL, no '&' */
} brute_t;

static void brute_rec(brute_t *E, int k, int l) {
  /* (k,l) is the innermost pair so far: score the chain as it stands, then extend it inwards */
  const int e = orc_eval(E->P, E->ab, E->n1 + E->n2, E->n1 + 1, E->db);
  if (e < E->best) E->best = e;
  for (int i = k + 1; i <= E->n1 && i - k - 1 <= MAXLOOP; i++)
    for (int j = l - 1; j >= 1 && (i - k - 1) + (l - j - 1) <= MAXLOOP; j--) {
      if (!PTYPE[E->A[i]][E->B[j]]) continue;
      E->db[i - 1] = '('; E->db[E->n1 + j - 1] = ')';
      brute_rec(E, i, j);
      E->db[i - 1] = '.'; E->db[E->n1 + j - 1] = '.';
    }
}

/* every duplex chain of (a, b) scored by orc_eval on a&b: the least energy, INF when there is none */
int orc_duplex_brute(const orc_params *P, const char *a, int n1, const char *b, int n2) {
  brute_t E;
  E.P = P; E.n1 = n1; E.n2 = n2; E.best = INF;
  char *ab = malloc(n1 + n2 + 1);
  memcpy(ab, a, n1); memcpy(ab + n1, b, n2); ab[n1 + n2] = '\0';
  E.ab = ab;
  E.A = calloc(n1 + 2, sizeof(int)); E.B = calloc(n2 + 2, sizeof(int));
  for (int i = 1; i <= n1; i++) E.A[i] = enc(a[i - 1]);
  for (int j = 1; j <= n2; j++) E.B[j] = enc(b[j - 1]);
  E.db = malloc(n1 + n2 + 1);
  memset(E.db, '.', n1 + n2); E.db[n1 + n2] = '\0';
  for (int k = 1; k <= n1; k++)
    for (int l = n2; l >= 1; l--) {
      if (!PTYPE[E.A[k]][E.B[l]]) continue;
      E.db[k - 1] = '('; E.db[n1 + l - 1] = ')';
      brute_rec(&E, k, l);
      E.db[k - 1] = '.'; E.db[n1 + l - 1] = '.';
    }
  free(ab); free(E.A); free(E.B); free(E.db);
  return E.best;
}
