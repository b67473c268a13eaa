// bf_twobest.cu -- the energy of the SECOND-best secondary structure without enumerating the energy band (sm_100a).
//
// DesiRNA's negative design (`-nd on`) asks for the energy of the first suboptimal structure: it widens an energy band in
// 1 kcal/mol steps and lets ViennaRNA enumerate every structure in it (fc.subopt_cb with uniq_ML = 1,
// utils/energy_scores.py:453-488) only to read the second entry of the sorted list.  The same number is the second-best
// derivation of an UNAMBIGUOUS folding grammar, so one DP over (best, second best) pairs gives it:
//   alternatives of a cell are disjoint sets of structures  ->  merge their pairs, keep the two smallest
//   a concatenation A B                                      ->  (a1 + b1, min(a1 + b2, a2 + b1))
// The grammar is the partition function's (it has to count every structure once, SURVEY.md A.6): pair table c, fM1 (exactly one
// stem, starting at i, unpaired tail), fML (at least one stem: the last stem starts at u, before it either only unpaired bases
// or an fML), exterior f5; energies are the integer loop energies of the MFE kernels (A.3).  One CTA per sequence, a warp per
// cell -- this is a rare call (only for mutants that already fold into the target), not a throughput path.
//
// Two strands (TWO, some row has a cut): the grammar of the partition function's two-strand recursions, with the nick rules of
// bf_k_mfe<TWO>.  TURN applies within a strand only; a pair (i, j) with i < cp <= j closes the nick loop -- Ext of the reversed pair
// plus the exterior-style chains fcA2 over i+1..cp-1 and fcB2 over cp..j-1 (both unambiguous, one stem or one unpaired base at a
// time); unpaired stretches of interior loops, multiloops and fML never contain the nick; an exterior stem that spans the nick adds
// DuplexInit (one such stem at most, so a connected structure counts it once, as eval does).  Rows without a cut fold as single strands.
#include "bf_kernels.h"

#include <cstdlib>

#include "bf_device.cuh"

namespace {

constexpr int kNW2 = 8;

struct Two { int a, b; };   // a <= b, both clamped at BF_INF
__device__ __forceinline__ Two two_inf() { Two t; t.a = BF_INF; t.b = BF_INF; return t; }
__device__ __forceinline__ Two two_push(Two t, int v) {
  if (v < t.a) { t.b = t.a; t.a = v; }
  else if (v < t.b) t.b = v;
  return t;
}
__device__ __forceinline__ Two two_merge(Two x, Two y) { return two_push(two_push(x, y.a), y.b); }
__device__ __forceinline__ Two two_add(Two x, int e) {
  Two r;
  r.a = x.a < BF_INF ? min(x.a + e, BF_INF) : BF_INF;
  r.b = x.b < BF_INF ? min(x.b + e, BF_INF) : BF_INF;
  return r;
}
__device__ __forceinline__ Two two_cat(Two x, Two y) {   // concatenation of two independent parts
  Two r = two_inf();
  if (x.a < BF_INF && y.a < BF_INF) {
    r.a = min(x.a + y.a, BF_INF);
    int s = BF_INF;
    if (y.b < BF_INF) s = min(s, x.a + y.b);
    if (x.b < BF_INF) s = min(s, x.b + y.a);
    r.b = min(s, BF_INF);
  }
  return r;
}
__device__ __forceinline__ Two two_warp(Two t) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Two u;
    u.a = __shfl_xor_sync(BF_FULL, t.a, o);
    u.b = __shfl_xor_sync(BF_FULL, t.b, o);
    t = two_merge(t, u);
  }
  return t;
}

// tables per CTA in HBM: c, fML, fM1 as int2 (best, second), W x W each
template <bool TWO>
__global__ void __launch_bounds__(kNW2 * 32) bf_k_mfe2(const BfParams *__restrict__ P, BfBatchDev b, int2 *ws, size_t ws_slot, int W,
                                                       int *work_counter, int *out_e1, int *out_e2, const uint8_t *only) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallI T;
  __shared__ uint8_t cu1[BF_NCAND], cu2[BF_NCAND];
  __shared__ int s_seq;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  bf_stage(&T, &P->si);
  {
    int k = 0;   // candidates (u1, u2) ordered by size
    for (int sz = 0; sz <= BF_MAXLOOP; sz++)
      for (int a = 0; a <= sz; a++, k++)
        if ((k % (kNW2 * 32)) == tid) { cu1[k] = (uint8_t)a; cu2[k] = (uint8_t)(sz - a); }
  }
  const int nmax = W - 2;
  uint8_t *S = dyn;
  uint8_t *SP = S + (nmax + 2 + 15) / 16 * 16;
  int2 *f5 = reinterpret_cast<int2 *>(SP + (nmax + 2 + 15) / 16 * 16);
  int2 *fcA2 = f5 + (nmax + 4);    // TWO: chain over k..cp-1
  int2 *fcB2 = fcA2 + (nmax + 4);  // TWO: chain over cp..k
  int2 *c = ws + (size_t)blockIdx.x * ws_slot;
  int2 *fml = c + (size_t)W * W;
  int2 *fm1 = fml + (size_t)W * W;
#define C2_(i, j) c[(i) * W + (j)]
#define M2_(i, j) fml[(i) * W + (j)]
#define M1_(i, j) fm1[(i) * W + (j)]
  auto ld = [](const int2 &v) { Two t; t.a = v.x; t.b = v.y; return t; };
  auto st = [](Two t) { return make_int2(t.a, t.b); };

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int s = s_seq;
    if (s >= b.B) break;
    if (only && !only[s]) continue;   // (uniform: every thread reads the same flag)
    const int n = b.len[s];
    BfCtx X;
    X.n = n; X.W = W; X.S = S; X.SP = SP;
    {
      const int cut = (TWO && b.cut) ? b.cut[s] : 0;
      X.cp = (cut > 1 && cut <= n) ? cut : n + 1;
    }
    const int cp = X.cp;
    // pair type honoured by the recursions: TURN within a strand only
    auto ptype = [&](int i, int j) { return TWO ? bf_ptype<TWO>(X, i, j) : bf_ptype_bases(SP[i], SP[j]); };
    auto same = [&](int a, int c) { return bf_same<TWO>(X, a, c); };
    {
      const char *src = b.seq + (size_t)s * b.stride;
      const uint8_t *np = b.nopair ? b.nopair + (size_t)s * b.stride : nullptr;
      for (int k = tid; k <= n + 1; k += blockDim.x) {
        const int code = (k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0;
        S[k] = (uint8_t)code;
        SP[k] = (uint8_t)((np && k >= 1 && k <= n && np[k - 1]) ? 0 : code);
      }
    }
    // spans below the minimal hairpin (two strands: single bases): nothing
    const int d0 = TWO ? 1 : BF_TURN + 1;
    for (int k = tid; k < d0 * (n + 1); k += blockDim.x) {
      const int d = k / (n + 1), i = k % (n + 1) + 1, j = i + d;
      if (j <= n + 1 && i <= n) { C2_(i, j) = make_int2(BF_INF, BF_INF); M2_(i, j) = make_int2(BF_INF, BF_INF); M1_(i, j) = make_int2(BF_INF, BF_INF); }
    }
    if (TWO && tid == 0 && cp <= n) { fcA2[cp] = make_int2(0, BF_INF); fcB2[cp - 1] = make_int2(0, BF_INF); }
    __syncthreads();
    for (int d = d0; d <= n - 1; d++) {
      if (TWO && cp <= n) {
        // the chains next to the nick over segments of span d-1 (every c they read is final): fcA2[cp-d] (warp 0), fcB2[cp+d-1]
        // (warp 1).  A nick-spanning cell of diagonal d reads chains of span <= d-2.
        if (warp == 0 && cp - d >= 1) {
          const int k = cp - d;
          Two e = two_inf();
          for (int q = k + 1 + lane; q <= cp - 1; q += 32) {
            const int t = ptype(k, q);
            if (!t) continue;
            const Two cc = ld(C2_(k, q));
            if (cc.a >= BF_INF) continue;
            int a, bb; bf_ext_nb<TWO>(X, k, q, &a, &bb);
            e = two_merge(e, two_cat(two_add(cc, bf_e_ext(T, t, a, bb)), ld(fcA2[q + 1])));
          }
          e = two_warp(e);
          if (lane == 0) fcA2[k] = st(two_merge(e, ld(fcA2[k + 1])));
        } else if (warp == 1 && cp + d - 1 <= n) {
          const int k = cp + d - 1;
          Two e = two_inf();
          for (int p = cp + lane; p < k; p += 32) {
            const int t = ptype(p, k);
            if (!t) continue;
            const Two cc = ld(C2_(p, k));
            if (cc.a >= BF_INF) continue;
            int a, bb; bf_ext_nb<TWO>(X, p, k, &a, &bb);
            e = two_merge(e, two_cat(ld(fcB2[p - 1]), two_add(cc, bf_e_ext(T, t, a, bb))));
          }
          e = two_warp(e);
          if (lane == 0) fcB2[k] = st(two_merge(e, ld(fcB2[k - 1])));
        }
        __syncthreads();
      }
      for (int i = 1 + warp; i + d <= n; i += kNW2) {
        const int j = i + d;
        const int t = ptype(i, j);
        Two cij = two_inf();
        if (t) {
          const int si1 = S[i + 1], sj1 = S[j - 1];
          const bool nick = TWO && i < cp && j >= cp;
          if (lane == 0) {
            if (nick) {   // the nick loop closed by (i,j): Ext of the reversed pair, the chains on both sides
              int a, bb; bf_nick_nb(X, i, j, &a, &bb);
              cij = two_add(two_cat(ld(fcA2[i + 1]), ld(fcB2[j - 1])), bf_e_ext(T, bf_rtype(t), a, bb));
            } else {
              cij = two_push(cij, min(bf_e_hairpin(P, T, S, i, j, t), BF_INF));
            }
          }
          // the unpaired stretches of an interior loop may not contain the nick: p stays on i's strand, q on j's
          const int pmax = nick ? cp - 1 : n, qmin = nick ? cp : 0;
          const int smx = min(BF_MAXLOOP, TWO ? d - 3 : d - 2 - (BF_TURN + 1)), kmax = smx >= 0 ? (smx + 1) * (smx + 2) / 2 : 0;
          for (int k = lane; k < kmax; k += 32) {
            const int u1 = cu1[k], u2 = cu2[k];
            const int p = i + 1 + u1, q = j - 1 - u2;
            if (TWO ? (p > pmax || q < qmin) : (q - p <= BF_TURN)) continue;
            const int t2 = ptype(p, q);
            if (!t2) continue;
            const Two cc = ld(C2_(p, q));
            if (cc.a >= BF_INF) continue;
            cij = two_merge(cij, two_add(cc, bf_e_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1])));
          }
          // multiloop closed by (i,j): at least one stem in [i+1, u-1], exactly one stem starting at u in [u, j-1]
          if (!TWO || (same(i, i + 1) && same(j - 1, j))) {
            const int clos = T.MLclosing + bf_e_mlstem(T, bf_rtype(t), sj1, si1);
            const int ulo = TWO ? i + 2 : i + 2 + BF_TURN + 1, uhi = TWO ? j - 1 : j - 2 - BF_TURN;
            for (int u = ulo + lane; u <= uhi; u += 32) {
              if (TWO && !same(u - 1, u)) continue;
              const Two l = ld(M2_(i + 1, u - 1)), r = ld(M1_(u, j - 1));
              cij = two_merge(cij, two_add(two_cat(l, r), clos));
            }
          }
          cij = two_warp(cij);
        }
        // fM1(i,j): one stem starting at i, ending at j or before (unpaired tail)
        // (two strands: the tail may not contain the nick, the stem's outer neighbours are on its strands)
        Two m1 = two_add(ld(M1_(i, j - 1)), T.MLbase);
        if (TWO && !same(j - 1, j)) m1 = two_inf();
        if (t && cij.a < BF_INF && i > 1 && j < n && (!TWO || (same(i - 1, i) && same(j, j + 1))))
          m1 = two_merge(m1, two_add(cij, bf_e_mlstem(T, t, S[i - 1], S[j + 1])));
        // fML(i,j): the last stem starts at u; before it only unpaired bases, or an fML
        Two m = two_inf();
        for (int u = i + 1 + lane; u <= (TWO ? j : j - BF_TURN - 1); u += 32) {
          if (TWO && !same(u - 1, u)) continue;
          Two left = ld(M2_(i, u - 1));
          if (!TWO || same(i, u)) left = two_push(left, (u - i) * T.MLbase);
          m = two_merge(m, two_cat(left, ld(M1_(u, j))));
        }
        m = two_warp(m);
        m = two_merge(m, m1);   // u = i
        if (lane == 0) { C2_(i, j) = st(cij); M1_(i, j) = st(m1); M2_(i, j) = st(m); }
      }
      __syncthreads();
    }
    // exterior loop: f5(j) = f5(j-1) | f5(i-1) + c(i,j) + Ext  (the stem that ends at j starts at i)
    if (warp == 0) {
      if (lane == 0) f5[0] = make_int2(0, BF_INF);
      __syncwarp();
      for (int j = 1; j <= n; j++) {
        Two e = two_inf();
        for (int i = 1 + lane; i < (TWO ? j : j - BF_TURN); i += 32) {
          const int t = ptype(i, j);
          if (!t) continue;
          const Two cc = ld(C2_(i, j));
          if (cc.a >= BF_INF) continue;
          int a = (i > 1) ? S[i - 1] : -1, bb = (j < n) ? S[j + 1] : -1, dup = 0;
          if constexpr (TWO) {   // neighbours on the stem's strands only; the stem that spans the nick adds DuplexInit
            bf_ext_nb<TWO>(X, i, j, &a, &bb);
            if (!same(i, j)) dup = T.DuplexInit;
          }
          e = two_merge(e, two_cat(ld(f5[i - 1]), two_add(cc, bf_e_ext(T, t, a, bb) + dup)));
        }
        e = two_warp(e);
        if (lane == 0) f5[j] = st(two_merge(e, ld(f5[j - 1])));
        __syncwarp();
      }
      if (lane == 0) {
        out_e1[s] = n > 0 ? f5[n].x : 0;
        out_e2[s] = n > 0 ? f5[n].y : BF_INF;
      }
    }
  }
#undef C2_
#undef M2_
#undef M1_
}

size_t twobest_smem(int W, bool two) {
  const size_t nmax = W - 2;
  return 2 * ((nmax + 2 + 15) / 16 * 16) + (two ? 3 : 1) * (nmax + 4) * sizeof(int2);
}

template <bool TWO>
cudaError_t launch(const BfParams *dP, const BfBatchDev &b, int2 *ws, int wstride, int grid, int *work_counter, int *out_e1, int *out_e2,
                   cudaStream_t st, const uint8_t *only) {
  const size_t sm = twobest_smem(wstride, TWO);
  if (sm > 32 * 1024) { cudaError_t e = cudaFuncSetAttribute(bf_k_mfe2<TWO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); if (e != cudaSuccess) return e; }
  bf_k_mfe2<TWO><<<grid, kNW2 * 32, sm, st>>>(dP, b, ws, bf_twobest_slot(wstride), wstride, work_counter, out_e1, out_e2, only);
  return cudaGetLastError();
}

}  // namespace

size_t bf_twobest_slot(int wstride) { return (size_t)3 * wstride * wstride; }   // int2 entries per CTA

cudaError_t bf_launch_twobest(const BfParams *dP, const BfBatchDev &b, int2 *ws, int wstride, int grid, int *work_counter, int *out_e1, int *out_e2,
                              cudaStream_t st, const uint8_t *only, bool two) {
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  return two ? launch<true>(dP, b, ws, wstride, grid, work_counter, out_e1, out_e2, st, only)
             : launch<false>(dP, b, ws, wstride, grid, work_counter, out_e1, out_e2, st, only);
}
