/* Test infrastructure: bf_findpath's breadth-limited search over direct refolding paths restated in plain C on the CPU oracle
 * (oracle/orc_fold.c), every structure scored by a full orc_eval, plus an exact subset DP over all direct paths.  Built and loaded
 * by tests/findpath_ref.py.
 *
 * One run (a -> b, width w): moves are the pairs of a not in b (deletions, ascending i), then the pairs of b not in a (insertions,
 * ascending i).  Level 0 is {a} with saddle E(a); level t+1 holds every valid one-move successor of the kept states, saddle =
 * max(parent saddle, E(child)); successors with the same move set are one state keeping the least (saddle, parent rank, move);
 * states are ordered by (saddle, E, parent rank, move) and the first w kept.  A call runs w = 1, 2, 4, ... (powers of two below W),
 * then W, each forward then reverse; the result is the run of least saddle, ties to the first run.  The path is reported from s1:
 * moves (i, j) positive for an insertion, negative for a deletion, and the k + 1 energies. */
#include <stdint.h>

#include "../oracle/orc_fold.c"

typedef struct { int sad, e, par, mv; } fp_cand;

static int fp_cand_cmp(const void *x, const void *y) {
  const fp_cand *a = x, *b = y;
  if (a->sad != b->sad) return a->sad < b->sad ? -1 : 1;
  if (a->e != b->e) return a->e < b->e ? -1 : 1;
  if (a->par != b->par) return a->par < b->par ? -1 : 1;
  return a->mv < b->mv ? -1 : a->mv > b->mv;
}

/* pairs (i<<16|j) of x not in y, ascending i */
static int fp_diff(const int *px, const int *py, int n, int *out) {
  int k = 0;
  for (int i = 1; i <= n; i++)
    if (px[i] > i && py[i] != px[i]) out[k++] = i << 16 | px[i];
  return k;
}

static int fp_pt(const char *db, int n, int *pt) {
  int *st = malloc(sizeof(int) * (n + 1)), sp = 0;
  for (int i = 0; i <= n + 1; i++) pt[i] = 0;
  for (int i = 1; i <= n; i++) {
    if (db[i - 1] == '(') st[sp++] = i;
    else if (db[i - 1] == ')') { int o = st[--sp]; pt[o] = i; pt[i] = o; }
  }
  free(st);
  return 0;
}

/* the structure (pair table pt) with pair (i, j) added is valid */
static int fp_can_add(const int *pt, int i, int j) {
  if (pt[i] || pt[j]) return 0;
  for (int x = i + 1; x < j; x++)
    if (pt[x] && (pt[x] < i || pt[x] > j)) return 0;
  return 1;
}

static int fp_energy(const orc_params *P, const char *seq, int n, const int *pt, char *db) {
  for (int i = 1; i <= n; i++) db[i - 1] = pt[i] == 0 ? '.' : pt[i] > i ? '(' : ')';
  db[n] = 0;
  return orc_eval(P, seq, n, 0, db);
}

/* one run from pair table pa with moves mv[0 .. k-1] (the first nd deletions); returns the saddle, writes the move indices of the
 * path in order (mo) and its k + 1 energies (pe); *max_level: the most distinct states any level held before truncation */
static int fp_run(const orc_params *P, const char *seq, int n, const int *pa, const int *mv, int k, int nd, int w, int *mo, int *pe,
                  int *max_level) {
  const int ps = n + 2;
  int cap = 1;
  int *cur_pt = malloc(sizeof(int) * ps), *cur_e = malloc(sizeof(int)), *cur_sad = malloc(sizeof(int));
  unsigned char *cur_set = calloc(k + 1, 1);
  char *db = malloc(n + 1);
  memcpy(cur_pt, pa, sizeof(int) * ps);
  cur_e[0] = cur_sad[0] = fp_energy(P, seq, n, pa, db);
  int npar = 1;
  /* back-pointers: level t (1..k), rank s */
  int *bpar = malloc(sizeof(int) * (size_t)(k + 1) * w), *bmv = malloc(sizeof(int) * (size_t)(k + 1) * w), *be = malloc(sizeof(int) * (size_t)(k + 1) * w);
  const int e0 = cur_e[0];
  int *tmp = malloc(sizeof(int) * ps);
  for (int t = 0; t < k; t++) {
    fp_cand *c = malloc(sizeof(fp_cand) * (size_t)npar * k + 1);
    int N = 0;
    for (int p = 0; p < npar; p++)
      for (int m = 0; m < k; m++) {
        if (cur_set[(size_t)p * (k + 1) + m]) continue;
        const int i = mv[m] >> 16, j = mv[m] & 0xffff;
        memcpy(tmp, cur_pt + (size_t)p * ps, sizeof(int) * ps);
        if (m < nd) { tmp[i] = 0; tmp[j] = 0; }
        else {
          if (!fp_can_add(tmp, i, j)) continue;
          tmp[i] = j; tmp[j] = i;
        }
        const int e = fp_energy(P, seq, n, tmp, db);
        c[N++] = (fp_cand){cur_sad[p] > e ? cur_sad[p] : e, e, p, m};
      }
    qsort(c, N, sizeof(fp_cand), fp_cand_cmp);
    /* distinct move sets in key order: the first of each set survives */
    int *sel = malloc(sizeof(int) * (N + 1)), nsel = 0;
    unsigned char *a = malloc(k + 1), *b = malloc(k + 1);
    for (int x = 0; x < N; x++) {
      memcpy(a, cur_set + (size_t)c[x].par * (k + 1), k + 1);
      a[c[x].mv] = 1;
      int dup = 0;
      for (int s = 0; s < nsel && !dup; s++) {
        memcpy(b, cur_set + (size_t)c[sel[s]].par * (k + 1), k + 1);
        b[c[sel[s]].mv] = 1;
        dup = memcmp(a, b, k + 1) == 0;
      }
      if (!dup) sel[nsel++] = x;
    }
    if (nsel > *max_level) *max_level = nsel;
    if (nsel > w) nsel = w;
    int *npt = malloc(sizeof(int) * (size_t)nsel * ps), *ne = malloc(sizeof(int) * nsel), *nsad = malloc(sizeof(int) * nsel);
    unsigned char *nset = malloc((size_t)nsel * (k + 1));
    for (int s = 0; s < nsel; s++) {
      const fp_cand *x = &c[sel[s]];
      const int i = mv[x->mv] >> 16, j = mv[x->mv] & 0xffff;
      memcpy(npt + (size_t)s * ps, cur_pt + (size_t)x->par * ps, sizeof(int) * ps);
      if (x->mv < nd) { npt[(size_t)s * ps + i] = 0; npt[(size_t)s * ps + j] = 0; }
      else { npt[(size_t)s * ps + i] = j; npt[(size_t)s * ps + j] = i; }
      memcpy(nset + (size_t)s * (k + 1), cur_set + (size_t)x->par * (k + 1), k + 1);
      nset[(size_t)s * (k + 1) + x->mv] = 1;
      ne[s] = x->e; nsad[s] = x->sad;
      bpar[(size_t)t * w + s] = x->par; bmv[(size_t)t * w + s] = x->mv; be[(size_t)t * w + s] = x->e;
    }
    free(cur_pt); free(cur_e); free(cur_sad); free(cur_set); free(c); free(sel); free(a); free(b);
    cur_pt = npt; cur_e = ne; cur_sad = nsad; cur_set = nset; npar = nsel;
    cap = nsel;
  }
  (void)cap;
  const int sad = cur_sad[0];
  int rank = 0;
  for (int t = k; t >= 1; t--) {
    mo[t - 1] = bmv[(size_t)(t - 1) * w + rank];
    pe[t] = be[(size_t)(t - 1) * w + rank];
    rank = bpar[(size_t)(t - 1) * w + rank];
  }
  pe[0] = e0;
  free(cur_pt); free(cur_e); free(cur_sad); free(cur_set); free(db); free(bpar); free(bmv); free(be); free(tmp);
  return sad;
}

/* bf_findpath for one instance: returns the saddle; n_moves, moves (2 per move) and path_e (k + 1) as the engine reports them;
 * max_level: the most distinct states of any level of any run before truncation */
int orc_findpath(const orc_params *P, const char *seq, int n, const char *s1, const char *s2, int W, int *n_moves, int *moves,
                 int *path_e, int *max_level) {
  int *p1 = malloc(sizeof(int) * (n + 2)), *p2 = malloc(sizeof(int) * (n + 2)), *fw = malloc(sizeof(int) * (n + 1)),
      *rv = malloc(sizeof(int) * (n + 1));
  fp_pt(s1, n, p1);
  fp_pt(s2, n, p2);
  const int d1 = fp_diff(p1, p2, n, fw), d2 = fp_diff(p2, p1, n, fw + d1), k = d1 + d2;
  memcpy(rv, fw + d1, sizeof(int) * d2);
  memcpy(rv + d2, fw, sizeof(int) * d1);
  int *mo = malloc(sizeof(int) * (k + 1)), *pe = malloc(sizeof(int) * (k + 1));
  int best = 0, have = 0;
  *max_level = 1;
  for (int w = 1;; w *= 2) {
    const int ww = w < W ? w : W;
    for (int dir = 0; dir < 2; dir++) {
      const int sad = fp_run(P, seq, n, dir ? p2 : p1, dir ? rv : fw, k, dir ? d2 : d1, ww, mo, pe, max_level);
      if (!have || sad < best) {
        have = 1; best = sad;
        for (int s = 0; s < k; s++) {
          /* step s of the path from s1 */
          const int t = dir ? k - 1 - s : s, m = mo[t], ij = (dir ? rv : fw)[m];
          const int del = m < (dir ? d2 : d1), ins = dir ? del : !del;
          moves[2 * s] = ins ? ij >> 16 : -(ij >> 16);
          moves[2 * s + 1] = ins ? ij & 0xffff : -(ij & 0xffff);
        }
        for (int s = 0; s <= k; s++) path_e[s] = pe[dir ? k - s : s];
      }
    }
    if (ww == W) break;
  }
  *n_moves = k;
  free(p1); free(p2); free(fw); free(rv); free(mo); free(pe);
  return best;
}

/* the least saddle over all direct paths from s1 to s2 (k <= 20): a DP over the subsets of moves, every valid structure scored by
 * orc_eval; INF when k > 20 */
int orc_findpath_dp(const orc_params *P, const char *seq, int n, const char *s1, const char *s2) {
  int *p1 = malloc(sizeof(int) * (n + 2)), *p2 = malloc(sizeof(int) * (n + 2)), *mv = malloc(sizeof(int) * (n + 1));
  fp_pt(s1, n, p1);
  fp_pt(s2, n, p2);
  const int d1 = fp_diff(p1, p2, n, mv), k = d1 + fp_diff(p2, p1, n, mv + d1);
  if (k > 20) { free(p1); free(p2); free(mv); return INF; }
  const uint32_t full = (1u << k) - 1;
  int *best = malloc(sizeof(int) * ((size_t)full + 1)), *pt = malloc(sizeof(int) * (n + 2));
  char *db = malloc(n + 1);
  for (uint32_t s = 0; s <= full; s++) {
    /* the structure of move set s, when valid */
    memcpy(pt, p1, sizeof(int) * (n + 2));
    int ok = 1;
    for (int m = 0; m < d1; m++)
      if (s >> m & 1) { pt[mv[m] >> 16] = 0; pt[mv[m] & 0xffff] = 0; }
    for (int m = d1; m < k && ok; m++)
      if (s >> m & 1) {
        const int i = mv[m] >> 16, j = mv[m] & 0xffff;
        if (!fp_can_add(pt, i, j)) ok = 0;
        else { pt[i] = j; pt[j] = i; }
      }
    best[s] = INF;
    if (!ok) continue;
    const int e = fp_energy(P, seq, n, pt, db);
    if (s == 0) { best[s] = e; continue; }
    int b = INF;
    for (int m = 0; m < k; m++)
      if ((s >> m & 1) && best[s & ~(1u << m)] < b) b = best[s & ~(1u << m)];
    if (b < INF) best[s] = b > e ? b : e;
  }
  const int r = best[full];
  free(p1); free(p2); free(mv); free(best); free(pt); free(db);
  return r;
}
