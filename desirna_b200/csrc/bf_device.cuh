// bf_device.cuh -- device-side building blocks shared by the fold kernels (sm_100a).
//
// Loop-energy functions follow SURVEY.md A.3 (ViennaRNA E_Hairpin / E_IntLoop / E_MLstem /
// E_ExtLoop as reached from utils/energy_scores.py:147-157 in the reference).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "bf_params.h"

#define BF_FULL 0xffffffffu
// The loop-energy functions below also run on the host (bf_subopt.cu walks the DP tables there): the read-only
// load intrinsic is used on the device only.
#ifdef __CUDA_ARCH__
#define BF_LDG(p) __ldg(p)
#else
#define BF_LDG(p) (*(p))
#endif
#define BF_HD __host__ __device__ __forceinline__
#define BF_WARPS 8
#define BF_THREADS (BF_WARPS * 32)
#define BF_NCAND 496  // (u1,u2) with u1+u2 <= 30

struct BfBatchDev {
  int B, stride;            // stride = bytes between consecutive sequences
  const char *seq;          // B x stride ASCII (ACGU/T, any case)
  const int *len;           // B
  const int *cut;           // B or null; 1-based first index of strand B, 0 = single strand
  const uint8_t *nopair;    // B x stride or null; 1 = position may not pair ('x' hard constraint)
};

// Packed triangular DP table of one sequence, stored by anti-diagonal: entry (i,j), d = j-i >= 4, at tri_off(n, d) + i-1.
BF_HD int tri_off(int n, int d) { return (d - 4) * n - (d * (d - 1) / 2 - 6); }
BF_HD size_t tri_size(int n) { return n >= 5 ? (size_t)tri_off(n, n) : 0; }

// dynamic shared memory a fold kernel's CTA may ask for: the 227 KB of sm_100 less its static tables and a reserve
constexpr size_t kSmemBudget = 232448 - 1024 - 256;

// per-sequence fold context held in shared memory
struct BfCtx {
  int n, cp, W;
  const uint8_t *S;   // bases 0..4, index 0..n+1
  const uint8_t *SP;  // S, but 0 where pairing is forbidden
};

BF_HD int bf_base_code(char c) {
  switch (c) {
    case 'A': case 'a': return 1;
    case 'C': case 'c': return 2;
    case 'G': case 'g': return 3;
    case 'U': case 'u': case 'T': case 't': return 4;
    default: return 0;
  }
}

// pair type of bases (a,b) in 1..4: CG=1 GC=2 GU=3 UG=4 AU=5 UA=6, 0 = no pair.  3 bits per entry.
BF_HD int bf_ptype_bases(int a, int b) {
  const unsigned long long K = (5ull << 9) | (1ull << 18) | (2ull << 27) | (3ull << 33) | (6ull << 36) | (4ull << 42);
  if (a == 0 || b == 0) return 0;
  return (int)((K >> (3 * ((a - 1) * 4 + (b - 1)))) & 7ull);
}
BF_HD int bf_rtype(int t) {
  // {0,2,1,4,3,6,5,7}
  return (int)((0x75634120u >> (4 * t)) & 15u);
}

template <bool TWO>
__device__ __forceinline__ bool bf_same(const BfCtx &X, int a, int b) {
  if (!TWO) return true;
  return (a >= X.cp) == (b >= X.cp);
}

// pair type honoured by the recursions (0 = may not pair): canonical, not masked, TURN within a strand
template <bool TWO>
__device__ __forceinline__ int bf_ptype(const BfCtx &X, int i, int j) {
  int t = bf_ptype_bases(X.SP[i], X.SP[j]);
  if (t && j - i <= BF_TURN && bf_same<TWO>(X, i, j)) t = 0;
  return t;
}

__device__ __forceinline__ int bf_warp_min(int v) { return __reduce_min_sync(BF_FULL, v); }
__device__ __forceinline__ double bf_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(BF_FULL, v, o);
  return v;
}

// splitmix64: the next 64-bit output of the stream whose state is s, and a uniform double in [0, 1) from it
__device__ __forceinline__ unsigned long long sm64(unsigned long long &s) {
  s += 0x9E3779B97F4A7C15ull;
  unsigned long long z = s;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ double u01(unsigned long long &s) { return (double)(sm64(s) >> 11) * (1.0 / 9007199254740992.0); }

// ------------------------------------------------------------------ special hairpins
BF_HD int bf_loop_key(const uint8_t *S, int i, int len, bool *valid) {
  int key = 0;
  bool ok = true;
  for (int k = 0; k < len; k++) {
    int b = S[i + k];
    ok = ok && (b != 0);
    key = (key << 2) | ((b - 1) & 3);
  }
  *valid = ok;
  return key;
}

// returns true and the table slot if (i,j) closes a tabulated tri/tetra/hexaloop
BF_HD bool bf_special_hp(const BfParams *__restrict__ P, const uint8_t *S, int i, int j, int *slot, int *kind) {
  int u = j - i - 1;
  bool valid;
  if (u == 4 && P->n_tetra) {
    int key = bf_loop_key(S, i, 6, &valid);
    if (valid && BF_LDG(&P->tetra_e[key]) != BF_NO_SPECIAL) { *slot = key; *kind = 4; return true; }
  } else if (u == 3 && P->n_tri) {
    int key = bf_loop_key(S, i, 5, &valid);
    if (valid && BF_LDG(&P->tri_e[key]) != BF_NO_SPECIAL) { *slot = key; *kind = 3; return true; }
  } else if (u == 6 && P->n_hexa) {
    int key = bf_loop_key(S, i, 8, &valid);
    if (valid)
      for (int k = 0; k < P->n_hexa; k++)
        if (BF_LDG(&P->hexa_key[k]) == key) { *slot = k; *kind = 6; return true; }
  }
  return false;
}

BF_HD int bf_e_hairpin(const BfParams *__restrict__ P, const BfSmallI &T, const uint8_t *S, int i, int j, int t) {
  int u = j - i - 1;
  int e = (u <= 30) ? T.hairpin[u] : T.hairpin[30] + BF_LDG(&P->ext_log[min(u, BF_EXT_TAB - 1)]);
  if (u < 3) return e;
  int slot, kind;
  if (bf_special_hp(P, S, i, j, &slot, &kind))
    return kind == 4 ? BF_LDG(&P->tetra_e[slot]) : kind == 3 ? BF_LDG(&P->tri_e[slot]) : BF_LDG(&P->hexa_e[slot]);
  if (u == 3) return e + (t > 2 ? T.TerminalAU : 0);
  return e + T.mmH[t][S[i + 1]][S[j - 1]];
}

__device__ __forceinline__ double bf_x_hairpin(const BfParams *__restrict__ P, const BfSmallD &T, const uint8_t *S, int i, int j, int t) {
  int u = j - i - 1;
  if (u < 3) return 0.0;
  int slot, kind;
  if (bf_special_hp(P, S, i, j, &slot, &kind))
    return kind == 4 ? BF_LDG(&P->x_tetra[slot]) : kind == 3 ? BF_LDG(&P->x_tri[slot]) : BF_LDG(&P->x_hexa[slot]);
  double w = (u <= 30) ? T.x_hairpin[u] : BF_LDG(&P->x_hp_big[min(u, BF_EXT_TAB - 1)]);
  if (u == 3) return (t > 2) ? w * T.x_TerminalAU : w;
  return w * T.x_mmH[t][S[i + 1]][S[j - 1]];
}

// ------------------------------------------------------------------ interior loops
// (i,j) outer pair of type t, inner pair (p,q); t2 = rtype[type(p,q)]; n1 = p-i-1, n2 = j-q-1
BF_HD int bf_e_intloop(const BfParams *__restrict__ P, const BfSmallI &T, int n1, int n2, int t, int t2,
                                            int si1, int sj1, int sp1, int sq1) {
  int nl = max(n1, n2), ns = min(n1, n2);
  if (nl == 0) return T.stack[t][t2];
  if (ns == 0) {
    int e = (nl <= BF_MAXLOOP) ? T.bulge[nl] : T.bulge[30] + BF_LDG(&P->ext_log[min(nl, BF_EXT_TAB - 1)]);
    if (nl == 1) e += T.stack[t][t2];
    else e += (t > 2 ? T.TerminalAU : 0) + (t2 > 2 ? T.TerminalAU : 0);
    return e;
  }
  if (ns == 1) {
    if (nl == 1) return BF_LDG(&P->int11[t][t2][si1][sj1]);
    if (nl == 2) return (n1 == 1) ? BF_LDG(&P->int21[t][t2][si1][sq1][sj1]) : BF_LDG(&P->int21[t2][t][sq1][si1][sp1]);
    int e = (nl + 1 <= BF_MAXLOOP) ? T.interior[nl + 1] : T.interior[30] + BF_LDG(&P->ext_log[min(nl + 1, BF_EXT_TAB - 1)]);
    e += min(T.ninio_max, (nl - ns) * T.ninio_m);
    return e + T.mm1nI[t][si1][sj1] + T.mm1nI[t2][sq1][sp1];
  }
  if (ns == 2) {
    if (nl == 2) return BF_LDG(&P->int22[t][t2][si1][sp1][sq1][sj1]);
    if (nl == 3) return T.interior[5] + T.ninio_m + T.mm23I[t][si1][sj1] + T.mm23I[t2][sq1][sp1];
  }
  int u = nl + ns;
  int e = (u <= BF_MAXLOOP) ? T.interior[u] : T.interior[30] + BF_LDG(&P->ext_log[min(u, BF_EXT_TAB - 1)]);
  e += min(T.ninio_max, (nl - ns) * T.ninio_m);
  return e + T.mmI[t][si1][sj1] + T.mmI[t2][sq1][sp1];
}

// Boltzmann weight of the same loop (u1+u2 <= MAXLOOP only: the PF never looks further)
__device__ __forceinline__ double bf_x_intloop(const BfParams *__restrict__ P, const BfSmallD &T, int n1, int n2, int t, int t2,
                                               int si1, int sj1, int sp1, int sq1) {
  int nl = max(n1, n2), ns = min(n1, n2);
  if (nl == 0) return T.x_stack[t][t2];
  if (ns == 0) {
    double w = T.x_bulge[nl];
    if (nl == 1) return w * T.x_stack[t][t2];
    if (t > 2) w *= T.x_TerminalAU;
    if (t2 > 2) w *= T.x_TerminalAU;
    return w;
  }
  if (ns == 1) {
    if (nl == 1) return BF_LDG(&P->x_int11[t][t2][si1][sj1]);
    if (nl == 2) return (n1 == 1) ? BF_LDG(&P->x_int21[t][t2][si1][sq1][sj1]) : BF_LDG(&P->x_int21[t2][t][sq1][si1][sp1]);
    return T.x_interior[nl + 1] * T.x_ninio[nl - ns] * T.x_mm1nI[t][si1][sj1] * T.x_mm1nI[t2][sq1][sp1];
  }
  if (ns == 2) {
    if (nl == 2) return BF_LDG(&P->x_int22[t][t2][si1][sp1][sq1][sj1]);
    if (nl == 3) return T.x_interior[5] * T.x_ninio[1] * T.x_mm23I[t][si1][sj1] * T.x_mm23I[t2][sq1][sp1];
  }
  return T.x_interior[nl + ns] * T.x_ninio[nl - ns] * T.x_mmI[t][si1][sj1] * T.x_mmI[t2][sq1][sp1];
}

// ------------------------------------------------------------------ stems in multi / exterior loops (a,b < 0: neighbour absent)
BF_HD int bf_e_mlstem(const BfSmallI &T, int t, int a, int b) {
  int e = T.MLintern + (t > 2 ? T.TerminalAU : 0);
  if (a >= 0 && b >= 0) e += T.mmM[t][a][b];
  else if (a >= 0) e += T.dangle5[t][a];
  else if (b >= 0) e += T.dangle3[t][b];
  return e;
}
BF_HD int bf_e_ext(const BfSmallI &T, int t, int a, int b) {
  int e = (t > 2 ? T.TerminalAU : 0);
  if (a >= 0 && b >= 0) e += T.mmE[t][a][b];
  else if (a >= 0) e += T.dangle5[t][a];
  else if (b >= 0) e += T.dangle3[t][b];
  return e;
}
__device__ __forceinline__ double bf_x_mlstem(const BfSmallD &T, int t, int a, int b) {
  double w = T.x_MLintern;
  if (t > 2) w *= T.x_TerminalAU;
  if (a >= 0 && b >= 0) w *= T.x_mmM[t][a][b];
  else if (a >= 0) w *= T.x_d5[t][a];
  else if (b >= 0) w *= T.x_d3[t][b];
  return w;
}
__device__ __forceinline__ double bf_x_ext(const BfSmallD &T, int t, int a, int b) {
  double w = (t > 2) ? T.x_TerminalAU : 1.0;
  if (a >= 0 && b >= 0) w *= T.x_mmE[t][a][b];
  else if (a >= 0) w *= T.x_d5[t][a];
  else if (b >= 0) w *= T.x_d3[t][b];
  return w;
}

// exterior stem (i,j): neighbours count only when present and on the same strand (A.7)
template <bool TWO>
__device__ __forceinline__ void bf_ext_nb(const BfCtx &X, int i, int j, int *a, int *b) {
  *a = (i > 1 && bf_same<TWO>(X, i - 1, i)) ? X.S[i - 1] : -1;
  *b = (j < X.n && bf_same<TWO>(X, j, j + 1)) ? X.S[j + 1] : -1;
}
// closing pair of a nick-containing loop, seen from inside
__device__ __forceinline__ void bf_nick_nb(const BfCtx &X, int i, int j, int *a, int *b) {
  *a = (j - 1 >= X.cp) ? X.S[j - 1] : -1;
  *b = (i + 1 < X.cp) ? X.S[i + 1] : -1;
}

// stage a POD struct from global into shared memory with the whole CTA
template <typename Tp>
__device__ __forceinline__ void bf_stage(Tp *dst, const Tp *__restrict__ src) {
  static_assert(sizeof(Tp) % 4 == 0, "word-sized struct expected");
  const uint32_t *s = reinterpret_cast<const uint32_t *>(src);
  uint32_t *d = reinterpret_cast<uint32_t *>(dst);
  for (int k = threadIdx.x; k < (int)(sizeof(Tp) / 4); k += blockDim.x) d[k] = BF_LDG(s + k);
}
