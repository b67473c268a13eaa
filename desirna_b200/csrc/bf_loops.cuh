// bf_loops.cuh -- exact energy changes of single-pair moves on one strand (sm_100a), shared by bf_findpath.cu and bf_kinfold.cu.
//
// With dangles = 2 every loop energy is local, so adding or removing one pair changes only the loop the pair closes and its
// enclosing loop: dE is the difference of those loop energies, exact integer arithmetic, each loop scored as bf_k_eval scores it
// (non-standard pairs as type 7).
#pragma once
#include "bf_device.cuh"

namespace {

// pair table of a state with one pair added (ai, aj) or removed (di, dj); -1: none
struct FpView {
  const short *pt;
  int ai, aj, di, dj;
  __device__ __forceinline__ int operator()(int x) const {
    if (x == ai) return aj;
    if (x == aj) return ai;
    if (x == di || x == dj) return 0;
    return pt[x];
  }
};

__device__ __forceinline__ int fp_type(const uint8_t *S, int i, int j) {
  const int t = bf_ptype_bases(S[i], S[j]);
  return t ? t : 7;
}

// energy of the loop closed by (i, v(i)), or of the exterior loop (i = 0), exactly as bf_k_eval scores it for one strand
__device__ int fp_loop(const BfParams *__restrict__ P, const BfSmallI &T, const uint8_t *S, int n, const FpView v, int i) {
  if (i == 0) {
    int e = 0;
    for (int x = 1; x <= n; x++) {
      const int q = v(x);
      if (q > x) {
        e += bf_e_ext(T, fp_type(S, x, q), x > 1 ? S[x - 1] : -1, q < n ? S[q + 1] : -1);
        x = q;
      }
    }
    return e;
  }
  const int j = v(i), t = fp_type(S, i, j);
  int nstem = 0, p1 = 0, q1 = 0, mlsum = 0, unp = 0;
  for (int x = i + 1; x < j;) {
    const int q = v(x);
    if (q > x) {
      if (!nstem) { p1 = x; q1 = q; }
      nstem++;
      mlsum += bf_e_mlstem(T, fp_type(S, x, q), S[x - 1], S[q + 1]);
      x = q + 1;
    } else {
      unp++;
      x++;
    }
  }
  if (nstem == 0) return bf_e_hairpin(P, T, S, i, j, t);
  if (nstem == 1) return bf_e_intloop(P, T, p1 - i - 1, j - q1 - 1, t, fp_type(S, q1, p1), S[i + 1], S[j - 1], S[p1 - 1], S[q1 + 1]);
  return T.MLclosing + bf_e_mlstem(T, bf_rtype(t), S[j - 1], S[i + 1]) + mlsum + unp * T.MLbase;
}

// the closing pair (its 5' end) of the loop that holds pair (i, j) or would hold it; 0: the exterior loop
__device__ int fp_enclosing(const short *pt, int i) {
  for (int x = i - 1; x >= 1;) {
    const int q = pt[x];
    if (q == 0) x--;
    else if (q > x) return x;
    else x = q - 1;
  }
  return 0;
}

__device__ int fp_eval(const BfParams *__restrict__ P, const BfSmallI &T, const uint8_t *S, int n, const short *pt) {
  const FpView v{pt, -1, -1, -1, -1};
  int e = fp_loop(P, T, S, n, v, 0);
  for (int x = 1; x <= n; x++)
    if (pt[x] > x) e += fp_loop(P, T, S, n, v, x);
  return e;
}

}  // namespace
