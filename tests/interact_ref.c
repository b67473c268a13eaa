/* Test infrastructure: the accessibility-aware interaction of strands a and b (bf_interact) restated in plain C on the CPU oracle's
 * energy functions (oracle/orc_fold.c, through tests/duplex_ref.c), with the engine's span, score, tie and trace rules, and a brute
 * force over every chain scored by orc_eval on a&b.  Built and loaded by tests/interact_ref.py.
 *
 * A site is a duplex chain (k1,l1), ..., (km,lm) with km - k1 + 1 <= span and l1 - lm + 1 <= span.  H is the chain's energy,
 * E = (double)H / 100.0 + ED_a + ED_b with ED_a = ed_a[(k1-1) * span + km-k1], ED_b = ed_b[(lm-1) * span + l1-lm] (kcal/mol, +inf:
 * the stretch is never unpaired; a NULL row set: 0).  The result is the least E, ties to the first site in the order k1 ascending,
 * l1 descending, km ascending, lm descending; the structure is traced inside the fixed-start table of (k1,l1) with bf_duplex's rule
 * (the first (k,l) reproducing h(i,j), k = i-1 downwards, then l = j+1 upwards). */
#include <math.h>

#include "duplex_ref.c"

/* h(k1+di, l1-dj) of start (k1,l1) over wa x wb cells: hh[di * span + dj], INF where unreachable */
static void ix_fill(const orc_params *P, const int *A, const int *B, int n1, int n2, int k1, int l1, int span, int wa, int wb, int *hh) {
  for (int di = 0; di < wa; di++)
    for (int dj = 0; dj < wb; dj++) {
      const int i = k1 + di, j = l1 - dj, t = PTYPE[A[i]][B[j]];
      int e = INF;
      if (t && di == 0 && dj == 0) e = P->DuplexInit + E_ext(P, t, i > 1 ? A[i - 1] : -1, j < n2 ? B[j + 1] : -1);
      else if (t)
        for (int k = i - 1; k >= k1 && i - k - 1 <= MAXLOOP; k--)
          for (int l = j + 1; l <= l1 && (i - k - 1) + (l - j - 1) <= MAXLOOP; l++) {
            const int tk = PTYPE[A[k]][B[l]], hk = hh[(k - k1) * span + (l1 - l)];
            if (!tk || hk >= INF) continue;
            e = MIN2(e, hk + E_intloop(P, i - k - 1, l - j - 1, tk, RTYPE[t], A[k + 1], B[l - 1], A[i - 1], B[j + 1]));
          }
      hh[di * span + dj] = e;
    }
}

static double ix_ed(const double *ed, int span, int k, int u) { return ed ? ed[(size_t)(k - 1) * span + u - 1] : 0.0; }

/* out_e: E (+inf: no site); out_h: H (INF); site: k1, km, lm, l1 (0: none); ss: n1 + n2 + 2 chars or NULL; gap: E of the best site
 * with other bounds minus E (+inf when there is none) */
void orc_interact(const orc_params *P, const char *a, int n1, const char *b, int n2, int span, const double *ed_a, const double *ed_b,
                  double *out_e, int *out_h, int *site, char *ss, double *gap) {
  int *A = calloc(n1 + 2, sizeof(int)), *B = calloc(n2 + 2, sizeof(int)), *hh = malloc(sizeof(int) * span * span);
  for (int i = 1; i <= n1; i++) A[i] = enc(a[i - 1]);
  for (int j = 1; j <= n2; j++) B[j] = enc(b[j - 1]);
  double best = INFINITY, second = INFINITY;
  int bh = INF, bs[4] = {0, 0, 0, 0};
  for (int k1 = 1; k1 <= n1; k1++)
    for (int l1 = n2; l1 >= 1; l1--) {
      if (!PTYPE[A[k1]][B[l1]]) continue;
      const int wa = MIN2(span, n1 - k1 + 1), wb = MIN2(span, l1);
      ix_fill(P, A, B, n1, n2, k1, l1, span, wa, wb, hh);
      for (int di = 0; di < wa; di++)   /* rank order within the start: km ascending, lm descending */
        for (int dj = 0; dj < wb; dj++) {
          const int i = k1 + di, j = l1 - dj, h = hh[di * span + dj];
          if (h >= INF) continue;
          const int v = h + E_ext(P, RTYPE[PTYPE[A[i]][B[j]]], j > 1 ? B[j - 1] : -1, i < n1 ? A[i + 1] : -1);
          const double e = (double)v / 100.0 + ix_ed(ed_a, span, k1, di + 1) + ix_ed(ed_b, span, j, dj + 1);
          if (!(e < INFINITY)) continue;
          if (e < best) {
            second = best; best = e; bh = v;
            bs[0] = k1; bs[1] = i; bs[2] = j; bs[3] = l1;
          } else if (e < second) {
            second = e;
          }
        }
    }
  *out_e = best; *out_h = bh; *gap = second - best;
  if (bh >= INF) *gap = INFINITY;
  memcpy(site, bs, sizeof(bs));
  if (ss) {
    memset(ss, '.', n1 + n2 + 1);
    ss[n1] = '&';
    ss[n1 + n2 + 1] = '\0';
    if (bh < INF) {
      const int k1 = bs[0], l1 = bs[3];
      ix_fill(P, A, B, n1, n2, k1, l1, span, bs[1] - k1 + 1, l1 - bs[2] + 1, hh);
      int i = bs[1], j = bs[2];
      while (1) {
        ss[i - 1] = '(';
        ss[n1 + j] = ')';
        if (i == k1 && j == l1) break;
        const int t = PTYPE[A[i]][B[j]], hij = hh[(i - k1) * span + (l1 - j)];
        int found = 0;
        for (int k = i - 1; k >= k1 && i - k - 1 <= MAXLOOP && !found; k--)
          for (int l = j + 1; l <= l1 && (i - k - 1) + (l - j - 1) <= MAXLOOP; l++) {
            const int tk = PTYPE[A[k]][B[l]], hk = hh[(k - k1) * span + (l1 - l)];
            if (!tk || hk >= INF) continue;
            if (hij == hk + E_intloop(P, i - k - 1, l - j - 1, tk, RTYPE[t], A[k + 1], B[l - 1], A[i - 1], B[j + 1])) {
              i = k; j = l; found = 1;
              break;
            }
          }
        if (!found) break;
      }
    }
  }
  free(A); free(B); free(hh);
}

typedef struct {
  brute_t D;
  int span, k1, l1;
  const double *ed_a, *ed_b;
  double best;
  long long rank;
  int h, site[4];
} ibrute_t;

static void ibrute_rec(ibrute_t *E, int k, int l) {
  /* (k,l) is the innermost pair so far: score the site as it stands, then extend it inwards within the spans */
  brute_t *D = &E->D;
  const int H = orc_eval(D->P, D->ab, D->n1 + D->n2, D->n1 + 1, D->db);
  const double e = (double)H / 100.0 + ix_ed(E->ed_a, E->span, E->k1, k - E->k1 + 1) + ix_ed(E->ed_b, E->span, l, E->l1 - l + 1);
  const long long rank = (((long long)(E->k1 - 1) * D->n2 + (D->n2 - E->l1)) * 64 + (k - E->k1)) * 64 + (E->l1 - l);
  if (e < INFINITY && (e < E->best || (e == E->best && rank < E->rank))) {
    E->best = e; E->rank = rank; E->h = H;
    E->site[0] = E->k1; E->site[1] = k; E->site[2] = l; E->site[3] = E->l1;
  }
  for (int i = k + 1; i <= D->n1 && i - k - 1 <= MAXLOOP && i - E->k1 < E->span; i++)
    for (int j = l - 1; j >= 1 && (i - k - 1) + (l - j - 1) <= MAXLOOP && E->l1 - j < E->span; j--) {
      if (!PTYPE[D->A[i]][D->B[j]]) continue;
      D->db[i - 1] = '('; D->db[D->n1 + j - 1] = ')';
      ibrute_rec(E, i, j);
      D->db[i - 1] = '.'; D->db[D->n1 + j - 1] = '.';
    }
}

/* every site of (a, b) scored by orc_eval on a&b and the ED rows: the least E with the engine's tie order */
void orc_interact_brute(const orc_params *P, const char *a, int n1, const char *b, int n2, int span, const double *ed_a, const double *ed_b,
                        double *out_e, int *out_h, int *site) {
  ibrute_t E;
  memset(&E, 0, sizeof(E));
  brute_t *D = &E.D;
  D->P = P; D->n1 = n1; D->n2 = n2;
  char *ab = malloc(n1 + n2 + 1);
  memcpy(ab, a, n1); memcpy(ab + n1, b, n2); ab[n1 + n2] = '\0';
  D->ab = ab;
  D->A = calloc(n1 + 2, sizeof(int)); D->B = calloc(n2 + 2, sizeof(int));
  for (int i = 1; i <= n1; i++) D->A[i] = enc(a[i - 1]);
  for (int j = 1; j <= n2; j++) D->B[j] = enc(b[j - 1]);
  D->db = malloc(n1 + n2 + 1);
  memset(D->db, '.', n1 + n2); D->db[n1 + n2] = '\0';
  E.span = span; E.ed_a = ed_a; E.ed_b = ed_b; E.best = INFINITY; E.rank = -1; E.h = INF;
  for (int k = 1; k <= n1; k++)
    for (int l = n2; l >= 1; l--) {
      if (!PTYPE[D->A[k]][D->B[l]]) continue;
      E.k1 = k; E.l1 = l;
      D->db[k - 1] = '('; D->db[n1 + l - 1] = ')';
      ibrute_rec(&E, k, l);
      D->db[k - 1] = '.'; D->db[n1 + l - 1] = '.';
    }
  *out_e = E.best; *out_h = E.h;
  memcpy(site, E.site, sizeof(E.site));
  free(ab); free(D->A); free(D->B); free(D->db);
}
