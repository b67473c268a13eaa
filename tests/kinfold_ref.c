/* Test infrastructure: bf_kinfold's folding kinetics restated in plain C on the CPU oracle (oracle/orc_fold.c).  Every neighbour of
 * every state is scored by a full orc_eval; the rate table, the splitmix64 streams and the group-of-32 scan summation are restated
 * exactly, so that the moves, energies and structures of a trajectory match the engine's bit for bit (times to rounding: the device
 * log is not glibc's).  Built and loaded by tests/kinfold_ref.py.  The model is defined in include/b200fold.h (bf_kinfold). */
#include <stdint.h>

#include "../oracle/orc_fold.c"

static int kf_code(char c) {
  switch (c) {
    case 'A': case 'a': return 1;
    case 'C': case 'c': return 2;
    case 'G': case 'g': return 3;
    case 'U': case 'u': case 'T': case 't': return 4;
    default: return 0;
  }
}

static void kf_pt(const char *db, int n, int *pt) {
  int *st = malloc(sizeof(int) * (n + 1)), sp = 0;
  for (int i = 0; i <= n + 1; i++) pt[i] = 0;
  if (db)
    for (int i = 1; i <= n; i++) {
      if (db[i - 1] == '(') st[sp++] = i;
      else if (db[i - 1] == ')') { int o = st[--sp]; pt[o] = i; pt[i] = o; }
    }
  free(st);
}

static void kf_db(const int *pt, int n, char *db) {
  for (int i = 1; i <= n; i++) db[i - 1] = pt[i] == 0 ? '.' : pt[i] > i ? '(' : ')';
  db[n] = 0;
}

static int kf_energy(const orc_params *P, const char *seq, int n, const int *pt, char *db) {
  kf_db(pt, n, db);
  return orc_eval(P, seq, n, 0, db);
}

/* the valid moves of structure pt in canonical order: (i << 16 | j) and dE = orc_eval(neighbour) - e0; returns their count */
static int kf_moves_pt(const orc_params *P, const char *seq, int n, int *pt, int e0, int *mv, int *de, char *db) {
  int cnt = 0;
  for (int i = 1; i <= n; i++)
    for (int j = i + 4; j <= n; j++) {
      const int del = pt[i] == j;
      if (!del) {
        if (pt[i] || pt[j] || !PTYPE[kf_code(seq[i - 1])][kf_code(seq[j - 1])]) continue;
        int ok = 1;
        for (int x = i + 1; x < j && ok; x++)
          if (pt[x] && (pt[x] < i || pt[x] > j)) ok = 0;
        if (!ok) continue;
      }
      pt[i] = del ? 0 : j; pt[j] = del ? 0 : i;
      const int e = kf_energy(P, seq, n, pt, db);
      pt[i] = del ? j : 0; pt[j] = del ? i : 0;
      mv[cnt] = i << 16 | j;
      de[cnt] = e - e0;
      cnt++;
    }
  return cnt;
}

/* exported: the valid moves of dot-bracket db (mv, de: room for every canonical pair) */
int kf_moves(const orc_params *P, const char *seq, int n, const char *db, int *mv, int *de) {
  int *pt = malloc(sizeof(int) * (n + 2));
  char *buf = malloc(n + 1);
  kf_pt(db, n, pt);
  const int e0 = kf_energy(P, seq, n, pt, buf);
  const int c = kf_moves_pt(P, seq, n, pt, e0, mv, de, buf);
  free(pt); free(buf);
  return c;
}

double kf_kT(const orc_params *P) { return P->kT; }

/* the rate table of rule 0 / 1: k(dE) at [dE + 32768] */
void kf_rate_table(const orc_params *P, int rule, double *rate) {
  const double kT = P->kT;
  for (int x = 0; x < 65536; x++) {
    const double de = (double)(x - 32768);
    if (rule == 0) rate[x] = exp(-de * 10.0 / (2.0 * kT));
    else {
      const double k = exp(-de * 10.0 / kT);
      rate[x] = k < 1.0 ? k : 1.0;
    }
  }
}

static uint64_t kf_sm64(uint64_t *s) {
  *s += 0x9E3779B97F4A7C15ull;
  uint64_t z = *s;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
static double kf_u01(uint64_t *s) { return (double)(kf_sm64(s) >> 11) * (1.0 / 9007199254740992.0); }

/* 5-step inclusive scan of 32 doubles, all lanes at once */
static void kf_scan32(double *v) {
  double w[32];
  for (int o = 1; o < 32; o <<= 1) {
    memcpy(w, v, sizeof(w));
    for (int l = o; l < 32; l++) v[l] = w[l] + w[l - o];
  }
}

static double kf_rel(double a, double b) {
  const double m = fabs(a) > fabs(b) ? fabs(a) : fabs(b);
  return m > 0 ? fabs(a - b) / m : 0.0;
}

/* one trajectory (instance r, trajectory k) of bf_kinfold; start / stop may be NULL.  *margin: the least relative distance of any
 * time comparison that decided the outcome (t + dt against t_max, snapshot times against t + dt), 1 if there was none */
void kf_traj(const orc_params *P, const char *seq, int n, const char *start, const char *stop, int rule, double t_max, uint64_t seed,
             int r, int k, long long max_steps, int n_snap, const double *t_snap, const double *rate, int *status, double *t_end,
             long long *steps_out, int *e_end, char *ss_end, int *e_snap, char *ss_snap, double *margin) {
  int *pt = malloc(sizeof(int) * (n + 2)), *ps = malloc(sizeof(int) * (n + 2));
  const size_t cap = (size_t)n * n / 2 + 32;
  int *mv = malloc(sizeof(int) * cap), *de = malloc(sizeof(int) * cap);
  double *R = malloc(sizeof(double) * (cap / 32 + 2));
  char *db = malloc(n + 1);
  kf_pt(start, n, pt);
  kf_pt(stop, n, ps);
  int e = kf_energy(P, seq, n, pt, db), diff = 0;
  for (int x = 1; x <= n; x++) diff += (pt[x] > x && ps[x] != pt[x]) + (ps[x] > x && pt[x] != ps[x]);
  uint64_t s0 = seed;
  uint64_t s1 = kf_sm64(&s0) ^ (((uint64_t)(uint32_t)r << 32) | (uint32_t)k);
  uint64_t rs = kf_sm64(&s1);
  double t = 0.0;
  long long steps = 0;
  int st = 0, s = 0;
  *margin = 1.0;
  int done = stop && diff == 0;
  if (done) st = 1;
  while (!done) {
    const int nm = kf_moves_pt(P, seq, n, pt, e, mv, de, db);
    int pick;
    if (rule == 2) {
      pick = -1;
      for (int x = 0; x < nm; x++)
        if (de[x] < 0 && (pick < 0 || de[x] < de[pick])) pick = x;
      if (pick < 0) break;
    } else {
      if (nm == 0) { t = t_max; break; }
      const int G = (nm + 31) / 32;
      double run = 0.0, v[32];
      for (int g = 0; g < G; g++) {
        for (int l = 0; l < 32; l++) v[l] = g * 32 + l < nm ? rate[de[g * 32 + l] + 32768] : 0.0;
        kf_scan32(v);
        run += v[31];
        R[g] = run;
      }
      const double K = run;
      const double u1 = kf_u01(&rs), u2 = kf_u01(&rs);
      const double tn = t + -log(1.0 - u1) / K;
      const double mt = kf_rel(tn, t_max);
      if (mt < *margin) *margin = mt;
      for (int y = 0; y < n_snap; y++) {
        const double ms = kf_rel(t_snap[y], tn);
        if (ms < *margin) *margin = ms;
      }
      if (tn > t_max) { t = t_max; break; }
      for (; s < n_snap && t_snap[s] < tn; s++) {
        e_snap[s] = e;
        kf_db(pt, n, ss_snap + (size_t)s * (n + 1));
      }
      t = tn;
      const double target = u2 * K;
      int g = -1;
      for (int y = 0; y < G && g < 0; y++)
        if (R[y] > target) g = y;
      if (g < 0) pick = nm - 1;
      else {
        for (int l = 0; l < 32; l++) v[l] = g * 32 + l < nm ? rate[de[g * 32 + l] + 32768] : 0.0;
        kf_scan32(v);
        const double rp = g > 0 ? R[g - 1] : 0.0;
        const int cnt = nm - g * 32 < 32 ? nm - g * 32 : 32;
        pick = g * 32 + cnt - 1;
        for (int l = 0; l < cnt; l++)
          if (rp + v[l] > target) { pick = g * 32 + l; break; }
      }
    }
    const int i = mv[pick] >> 16, j = mv[pick] & 0xffff, del = pt[i] == j;
    pt[i] = del ? 0 : j; pt[j] = del ? 0 : i;
    e += de[pick];
    diff += ((ps[i] == j) == del) ? 1 : -1;
    steps++;
    if (stop && diff == 0) { st = 1; break; }
    if (steps >= max_steps) { st = 2; break; }
  }
  const int blank = st == 2 || rule == 2;
  for (; s < n_snap; s++) {
    e_snap[s] = blank ? INF : e;
    if (blank) ss_snap[(size_t)s * (n + 1)] = 0;
    else kf_db(pt, n, ss_snap + (size_t)s * (n + 1));
  }
  *status = st; *t_end = t; *steps_out = steps; *e_end = e;
  kf_db(pt, n, ss_end);
  free(pt); free(ps); free(mv); free(de); free(R); free(db);
}
