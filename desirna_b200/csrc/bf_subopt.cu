// bf_subopt.cu -- suboptimal structures within an energy band (Wuchty enumeration) on the DP tables of the GPU MFE fill.
//
// Replaces fc.subopt_cb(delta, cb, data) with RNA.cvar.uniq_ML = 1 as called from
// get_first_suboptimal_structure_and_energy (utils/energy_scores.py:453-488 in the reference; SURVEY.md A.10):
// every secondary structure whose energy is within `delta` dcal/mol of the MFE, each exactly once.
//
// The O(N^3) work (c and fML tables) is done by the fill kernels; what runs here on the host is the
// output-sensitive walk over those tables, on an UNAMBIGUOUS decomposition so that no structure is produced twice:
//   f5(j)     = f5(j-1)  |  f5(i-1) + c(i,j) + ext(i,j)
//   c(i,j)    = hairpin  |  c(p,q) + interior(i,j,p,q)  |  fML(i+1,u-1) + fM1(u,j-1) + closing        (rightmost stem starts at u)
//   fML(i,j)  = fML(i,u-1) + fM1(u,j)  |  (u-i) MLbase + fM1(u,j)
//   fM1(i,j)  = c(i,l) + mlstem(i,l) + (j-l) MLbase                                                   (exactly one stem, starting at i)
// fM1 and f5 are O(N^2) and are derived here from c.  A partial structure is extended only while
// (energy decided so far) + (sum of the optima of the open intervals) <= MFE + delta.
#include <algorithm>
#include <string>
#include <vector>

#include "bf_device.cuh"
#include "bf_kernels.h"

namespace {

struct Iv { int i, j, kind; };  // kind 0: f5 up to j; 1: fML(i,j); 2: c(i,j) (pair already written); 3: fM1(i,j)

struct Walker {
  const BfParams *P;
  const BfSmallI *T;
  int n, thr, cap;
  const uint8_t *S, *SP;
  const int *c, *fm;         // packed diagonal-major triangles (d >= 4)
  std::vector<int> fm1, f5;  // fm1: (n+2)^2
  std::vector<Iv> st;
  std::string ss;
  std::vector<std::pair<int, std::string>> *out;
  long long found = 0;
  bool overflow = false, first_only = false;   // first_only: stop at the first structure (bf_zuker_host's completions)

  int off(int d) const { return (d - 4) * n - (d * (d - 1) / 2 - 6); }
  int C(int i, int j) const { return (j - i > BF_TURN && i >= 1 && j <= n) ? c[off(j - i) + i - 1] : BF_INF; }
  int M(int i, int j) const { return (j - i > BF_TURN && i >= 1 && j <= n) ? fm[off(j - i) + i - 1] : BF_INF; }
  int &M1(int i, int j) { return fm1[(size_t)i * (n + 2) + j]; }
  int pt(int i, int j) const { return bf_ptype_bases(SP[i], SP[j]); }
  int ext(int i, int j, int t) const { return bf_e_ext(*T, t, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1); }
  int best(const Iv &v) {
    switch (v.kind) {
      case 0: return f5[v.j];
      case 1: return M(v.i, v.j);
      case 2: return C(v.i, v.j);
      default: return (v.j - v.i > BF_TURN) ? M1(v.i, v.j) : BF_INF;
    }
  }

  void prepare() {
    fm1.assign((size_t)(n + 2) * (n + 2), BF_INF);
    for (int i = 2; i <= n; i++)
      for (int j = i + BF_TURN + 1; j < n; j++) {
        int m = M1(i, j - 1) < BF_INF ? M1(i, j - 1) + T->MLbase : BF_INF;
        const int t = pt(i, j), cc = C(i, j);
        if (t && cc < BF_INF) m = std::min(m, cc + bf_e_mlstem(*T, t, S[i - 1], S[j + 1]));
        M1(i, j) = m;
      }
    f5.assign(n + 2, 0);
    for (int j = 1; j <= n; j++) {
      int e = f5[j - 1];
      for (int i = 1; i < j - BF_TURN; i++) {
        const int t = pt(i, j), cc = C(i, j);
        if (t && cc < BF_INF) e = std::min(e, f5[i - 1] + cc + ext(i, j, t));
      }
      f5[j] = e;
    }
  }

  // acc: energy decided so far; rest: sum of the optima of the intervals on the stack
  void rec(int acc, int rest) {
    if (overflow) return;
    if (st.empty()) {
      found++;
      if ((int)out->size() < cap) out->emplace_back(acc, ss);
      else overflow = true;
      if (first_only) overflow = true;
      return;
    }
    const Iv v = st.back();
    st.pop_back();
    rest -= best(v);
    auto go = [&](int e_dec, const Iv *subs, int nsub) {
      int bs = 0;
      for (int k = 0; k < nsub; k++) {
        const int b = best(subs[k]);
        if (b >= BF_INF) return;
        bs += b;
      }
      if (acc + e_dec + rest + bs > thr) return;
      for (int k = 0; k < nsub; k++) st.push_back(subs[k]);
      rec(acc + e_dec, rest + bs);
      for (int k = 0; k < nsub; k++) st.pop_back();
    };
    const int i = v.i, j = v.j;
    if (v.kind == 0) {
      if (j == 0) go(0, nullptr, 0);
      else {
        { Iv s1[1] = {{1, j - 1, 0}}; go(0, s1, 1); }
        for (int u = j - BF_TURN - 1; u >= 1; u--) {
          const int t = pt(u, j);
          if (!t || C(u, j) >= BF_INF) continue;
          ss[u - 1] = '('; ss[j - 1] = ')';
          Iv s2[2] = {{1, u - 1, 0}, {u, j, 2}};
          go(ext(u, j, t), s2, 2);
          ss[u - 1] = '.'; ss[j - 1] = '.';
        }
      }
    } else if (v.kind == 2) {
      const int t = pt(i, j), si1 = S[i + 1], sj1 = S[j - 1];
      go(bf_e_hairpin(P, *T, S, i, j, t), nullptr, 0);
      for (int p = i + 1; p <= std::min(j - 2 - BF_TURN, i + BF_MAXLOOP + 1); p++) {
        const int minq = std::max(p + BF_TURN + 1, j - i + p - BF_MAXLOOP - 2);
        for (int q = j - 1; q >= minq; q--) {
          const int t2 = pt(p, q);
          if (!t2 || C(p, q) >= BF_INF) continue;
          ss[p - 1] = '('; ss[q - 1] = ')';
          Iv s1[1] = {{p, q, 2}};
          go(bf_e_intloop(P, *T, p - i - 1, j - q - 1, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1]), s1, 1);
          ss[p - 1] = '.'; ss[q - 1] = '.';
        }
      }
      const int close = T->MLclosing + bf_e_mlstem(*T, bf_rtype(t), sj1, si1);
      for (int u = i + 2 + BF_TURN + 1; u <= j - 1 - BF_TURN - 1; u++) {
        Iv s2[2] = {{i + 1, u - 1, 1}, {u, j - 1, 3}};
        go(close, s2, 2);
      }
    } else if (v.kind == 1) {
      for (int u = i; u <= j - BF_TURN - 1; u++) {
        if (u > i) { Iv s2[2] = {{i, u - 1, 1}, {u, j, 3}}; go(0, s2, 2); }
        Iv s1[1] = {{u, j, 3}};
        go((u - i) * T->MLbase, s1, 1);
      }
    } else {
      for (int l = i + BF_TURN + 1; l <= j; l++) {
        const int t = pt(i, l);
        if (!t || C(i, l) >= BF_INF || i <= 1 || l >= n) continue;
        ss[i - 1] = '('; ss[l - 1] = ')';
        Iv s1[1] = {{i, l, 2}};
        go(bf_e_mlstem(*T, t, S[i - 1], S[l + 1]) + (j - l) * T->MLbase, s1, 1);
        ss[i - 1] = '.'; ss[l - 1] = '.';
      }
    }
    st.push_back(v);
  }
};

}  // namespace

// Enumerate every structure with energy <= MFE + delta.  c / fm: host copies of the packed tables of ONE sequence.
// Returns the number of structures found (capped at `cap`: *truncated is set when the band holds more).
int bf_wuchty_host(const BfParams *P, int n, const uint8_t *S, const uint8_t *SP, const int *c, const int *fm, int delta, int cap,
                   std::vector<std::pair<int, std::string>> *out, int *mfe_out, bool *truncated) {
  Walker w;
  w.P = P; w.T = &P->si; w.n = n; w.S = S; w.SP = SP; w.c = c; w.fm = fm; w.cap = cap; w.out = out;
  w.prepare();
  const int mfe = w.f5[n];
  if (mfe_out) *mfe_out = mfe;
  w.thr = mfe + delta;
  w.ss.assign(n, '.');
  w.st.push_back({1, n, 0});
  w.rec(0, mfe);
  if (truncated) *truncated = w.overflow;
  std::sort(out->begin(), out->end());
  return (int)out->size();
}

// Zuker suboptimals (fc.subopt_zuker()): pairs in order of (E_pair, i, j); for each pair no listed structure contains yet, one
// structure of energy E_pair containing it.  Its outside part is traced back from Cout = E_pair - C, the exterior, interior and
// multiloop cases of bf_k_mfe_out tried in that order; what it leaves open (the pair itself, exterior prefixes and suffixes,
// multiloop segments) is completed by the Walker above with the band closed at the sum of their optima, so that its first
// leaf is an optimal completion.
int bf_zuker_host(const BfParams *P, int n, const uint8_t *S, const uint8_t *SP, const int *c, const int *fm, const int *e_pair, int cap,
                  std::vector<std::pair<int, std::string>> *out, bool *truncated) {
  Walker w;
  w.P = P; w.T = &P->si; w.n = n; w.S = S; w.SP = SP; w.c = c; w.fm = fm; w.cap = 1; w.first_only = true;
  w.prepare();
  const BfSmallI &T = P->si;
  std::vector<int> f3(n + 2, 0);
  for (int i = n; i >= 1; i--) {
    int e = f3[i + 1];
    for (int j = i + BF_TURN + 1; j <= n; j++) {
      const int t = w.pt(i, j), cc = w.C(i, j);
      if (t && cc < BF_INF) e = std::min(e, cc + w.ext(i, j, t) + f3[j + 1]);
    }
    f3[i] = e;
  }
  auto E = [&](int i, int j) { return e_pair[(size_t)(i - 1) * n + (j - 1)]; };
  auto CO = [&](int i, int j) { return (i >= 1 && j <= n && E(i, j) < BF_INF) ? E(i, j) - w.C(i, j) : BF_INF; };
  struct Pr { int e, i, j; };
  std::vector<Pr> pairs;
  for (int i = 1; i <= n; i++)
    for (int j = i + BF_TURN + 1; j <= n; j++)
      if (E(i, j) < BF_INF) pairs.push_back({E(i, j), i, j});
  std::sort(pairs.begin(), pairs.end(), [](const Pr &x, const Pr &y) { return x.e != y.e ? x.e < y.e : x.i != y.i ? x.i < y.i : x.j < y.j; });
  std::vector<char> covered((size_t)(n + 1) * (n + 1), 0);
  const int ml = T.MLbase;
  *truncated = false;
  for (const Pr &pr : pairs) {
    if (covered[(size_t)pr.i * (n + 1) + pr.j]) continue;
    if ((int)out->size() >= cap) { *truncated = true; break; }
    std::string ss(n, '.');
    std::vector<Iv> open;
    open.push_back({pr.i, pr.j, 2});
    int a = pr.i, b = pr.j, v = CO(a, b);
    for (;;) {
      ss[a - 1] = '('; ss[b - 1] = ')';
      const int t = w.pt(a, b);
      if (v == w.f5[a - 1] + w.ext(a, b, t) + f3[b + 1]) {
        if (a > 1) open.push_back({1, a - 1, 0});
        for (int i = b + 1; i <= n;) {   // the suffix f3[b+1], traced here (the Walker's exterior kind is a prefix)
          if (f3[i] == f3[i + 1]) { i++; continue; }
          int j = i + BF_TURN + 1;
          for (; j <= n; j++) {
            const int tt = w.pt(i, j), cc = w.C(i, j);
            if (tt && cc < BF_INF && f3[i] == cc + w.ext(i, j, tt) + f3[j + 1]) break;
          }
          if (j > n) return -1;
          ss[i - 1] = '('; ss[j - 1] = ')';
          open.push_back({i, j, 2});
          i = j + 1;
        }
        break;
      }
      bool found = false;
      for (int s = 0; s <= BF_MAXLOOP && !found; s++)
        for (int u1 = 0; u1 <= s && !found; u1++) {
          const int i = a - 1 - u1, j = b + 1 + s - u1;
          if (i < 1 || j > n) continue;
          const int co = CO(i, j);
          if (co >= BF_INF) continue;
          if (v == co + bf_e_intloop(P, T, u1, s - u1, w.pt(i, j), bf_rtype(t), S[i + 1], S[j - 1], S[a - 1], S[b + 1])) {
            a = i; b = j; v = co; found = true;
          }
        }
      if (found) continue;
      const int stem = (a > 1 && b < n) ? bf_e_mlstem(T, t, S[a - 1], S[b + 1]) : BF_INF;
      for (int i = a - 1; i >= 1 && !found && stem < BF_INF; i--)
        for (int j = b + 1; j <= n && !found; j++) {
          const int co = CO(i, j);
          if (co >= BF_INF) continue;
          const int base = co + T.MLclosing + bf_e_mlstem(T, bf_rtype(w.pt(i, j)), S[j - 1], S[i + 1]) + stem;
          const int lu = (a - 1 - i) * ml, lf = w.M(i + 1, a - 1), ru = (j - 1 - b) * ml, rf = w.M(b + 1, j - 1);
          const int opt[3][2] = {{lf, ru}, {lu, rf}, {lf, rf}};
          for (int k = 0; k < 3 && !found; k++) {
            if (opt[k][0] >= BF_INF || opt[k][1] >= BF_INF || v != base + opt[k][0] + opt[k][1]) continue;
            if (k != 1) open.push_back({i + 1, a - 1, 1});
            if (k != 0) open.push_back({b + 1, j - 1, 1});
            a = i; b = j; v = co; found = true;
          }
        }
      if (!found) return -1;
    }
    // complete the open intervals optimally
    std::vector<std::pair<int, std::string>> one;
    int rest = 0;
    for (const Iv &iv : open) rest += w.best(iv);
    w.st = open; w.ss = ss; w.out = &one; w.thr = rest; w.found = 0; w.overflow = false;
    w.rec(0, rest);
    if (one.empty()) return -1;
    const std::string &s1 = one[0].second;
    std::vector<int> stk;
    for (int k = 1; k <= n; k++) {
      if (s1[k - 1] == '(') stk.push_back(k);
      else if (s1[k - 1] == ')') { covered[(size_t)stk.back() * (n + 1) + k] = 1; stk.pop_back(); }
    }
    out->emplace_back(pr.e, s1);
  }
  std::sort(out->begin(), out->end());
  return (int)out->size();
}
