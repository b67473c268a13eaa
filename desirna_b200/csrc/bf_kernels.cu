// bf_kernels.cu -- batched RNA folding kernels for sm_100a (B200).
//
// One persistent CTA folds one sequence at a time (sequences are pulled from an atomic
// work counter).  The O(N^2) tables are filled as an anti-diagonal wavefront: on
// diagonal d every cell (i, i+d) is independent, one warp owns a cell, the 32 lanes
// split the cell's candidates (interior loops, multiloop / fML split points) and the
// partial results meet in a warp reduction (redux.sync min for the MFE, shuffle tree
// for the partition function).  One __syncthreads() separates diagonals.
//
// What replaces what (reference = DesiRNA through ViennaRNA's SWIG API):
//   bf_k_mfe   <- fc.mfe() / fc.mfe_dimer() / RNA.fold()   energy_scores.py:151,156,354; sequence_utils.py:1183
//   bf_k_pf    <- fc.pf() / fc.pf_dimer()                  energy_scores.py:150,157; dimer_multichain_energy.py:47
//   bf_k_eval  <- fc.eval_structure()                      energy_scores.py:75,99
// Recurrences: SURVEY.md A.4 (fill), A.5 (backtrack order), A.6 (inside), A.7 (two strands), A.8 (eval).
#include "bf_kernels.h"

#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "bf_device.cuh"

namespace {

// (u1,u2) enumeration of interior-loop candidates, u1 major: consecutive lanes walk q downwards in one row of c
__constant__ uint8_t c_cand_u1[BF_NCAND];
__constant__ uint8_t c_cand_u2[BF_NCAND];
// the 487 decomposable candidates as three lists, each ordered by loop size: generic [0, 375), 1xn [375, 429), bulge [429, 487);
// c_list_cnt[t][s] = entries of list t with size <= s
constexpr int kNDecomp = 487, kListStart[4] = {0, 375, 429, 487};
__constant__ uint8_t c_list_u1[kNDecomp];
__constant__ uint8_t c_list_u2[kNDecomp];
__constant__ short c_list_cnt[3][32];

// the nine interior-loop shapes that are not decomposed (stack, bulge 1, 1x1, 1x2, 2x1, 2x2, 2x3, 3x2): their index in the size-ordered
// candidate list (size * (size + 1) / 2 + u1) and their (u1, u2)
__device__ constexpr int kSpecK[9] = {0, 1, 2, 4, 7, 8, 12, 17, 18};
__device__ constexpr int kSpecU1[9] = {0, 0, 1, 1, 1, 2, 2, 2, 3};
__device__ constexpr int kSpecU2[9] = {0, 1, 0, 1, 2, 1, 2, 3, 2};
constexpr int kPreArr = 15;   // sequence-only arrays per diagonal buffer (PRE variants)
constexpr int kPreArrD = 13;  // partition function: arrays of doubles per diagonal buffer
constexpr int kPreMax = 256;  // longest sequence (both strands) the PRE variants take

struct __align__(8) BfSector { short i, j; int kind; };  // kind: 0 exterior(f5 up to j) 1 multiloop part 2 pair 3 fcA from i 4 fcB up to j

__device__ __forceinline__ size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------- common per-sequence setup
template <bool TWO>
__device__ __forceinline__ void load_sequence(const BfBatchDev &b, int s, uint8_t *S, uint8_t *SP, BfCtx *X, int W) {
  const int n = b.len[s];
  const char *src = b.seq + (size_t)s * b.stride;
  const uint8_t *np = b.nopair ? b.nopair + (size_t)s * b.stride : nullptr;
  for (int k = threadIdx.x; k <= n + 1; k += blockDim.x) {
    int code = (k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0;
    S[k] = (uint8_t)code;
    SP[k] = (uint8_t)((np && k >= 1 && k <= n && np[k - 1]) ? 0 : code);
  }
  X->n = n;
  int cut = (TWO && b.cut) ? b.cut[s] : 0;
  X->cp = (cut > 1 && cut <= n) ? cut : n + 1;
  X->W = W;
  X->S = S;
  X->SP = SP;
}

// =====================================================================================================
//                                               MFE
// =====================================================================================================
// PRE (sequences up to kPreMax nt): two barriers per diagonal instead of four.  Everything of a cell that depends on the sequence only
// is computed ONE DIAGONAL AHEAD, as items of the long middle stage (its parameter-table reads in L2 then overlap the other warps'
// candidate work instead of sitting on the critical path), the nick-side recursions fcA / fcB are items of that stage too (what they
// write is first read a diagonal later), and the items are dealt to the warps through a shared counter.
template <bool TWO, int NWG, bool PRE>
__global__ void __launch_bounds__(NWG * 32) bf_k_mfe(const BfParams *__restrict__ P, BfBatchDev b, int *ws, size_t ws_slot_ints,
                                                       int wstride, int *work_counter, int *out_mfe, char *out_ss, int ss_stride,
                                                       unsigned tables_smem_off) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallI T;
  __shared__ int s_seq;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int W = wstride;  // row stride of the tables, >= n+2

  bf_stage(&T, &P->si);
  // decomposable interior-loop candidates: three size-ordered lists (generic, 1xn, bulge: the variant of c they read and the term of
  // the closing pair they add are constant within a list).  Entry: x = offset of the inner pair's table entry relative to cell
  // (i,j)'s (table + (1 + u1) rows - (1 + u2) columns), y = size penalty (16 bits) | u1 << 16 | u2 << 24 (the nick test)
  __shared__ int2 lst[kNDecomp];
  __shared__ short lcnt[3][32];
  __shared__ int spec21[32];   // the first 21 candidates by size: u1 | u2 << 8 | (shape + 1) << 24 for the nine shapes evaluated in full
  __syncthreads();
  for (int k = tid; k < kNDecomp; k += blockDim.x) {
    const int u1 = c_list_u1[k], u2 = c_list_u2[k], sz = u1 + u2, t = k < 375 ? 0 : k < 429 ? 1 : 2;
    const int pen = t == 2 ? T.bulge[sz] : t == 1 ? T.interior[sz] + min(T.ninio_max, (sz - 2) * T.ninio_m)
                           : T.interior[sz] + min(T.ninio_max, abs(u1 - u2) * T.ninio_m);
    lst[k] = make_int2((3 + t) * W * W + (1 + u1) * W - (1 + u2), (min(pen, 32767) & 0xffff) | u1 << 16 | u2 << 24);
  }
  for (int k = tid; k < 96; k += blockDim.x) lcnt[k >> 5][k & 31] = c_list_cnt[k >> 5][k & 31];
  if (tid < 32) {
    int shape = 0;
    for (int q = 0; q < 9; q++) if (kSpecK[q] == tid) shape = q + 1;
    spec21[tid] = tid < 21 ? (c_cand_u1[tid] | c_cand_u2[tid] << 8 | shape << 24) : 0;
  }

  // dynamic smem carve-up
  const int nmax = W - 2;
  uint8_t *S = dyn;
  uint8_t *SP = S + align_up(nmax + 2, 16);
  int *f5 = reinterpret_cast<int *>(SP + align_up(nmax + 2, 16));
  int *fcA = f5 + (nmax + 4);
  int *fcB = fcA + (nmax + 4);
  BfSector *stk = reinterpret_cast<BfSector *>(fcB + (nmax + 4));
  // per-cell arrays of the diagonal in work (index = i)
  const int NA = nmax + 4;
  int *cbase = reinterpret_cast<int *>(stk + (2 * nmax + 16));
  // !PRE: cT cE0 cMMO cMM1O cMLC cEC cMS cLIST.   PRE: cEC cMS, then two buffers (diagonal parity) of the kPreArr sequence-only arrays
  // cT cE0 cMMO cMM1O cMLC cLIST cE9[9] (the nine interior-loop shapes that are evaluated in full, INF where the inner pair is impossible)
  int *cT = cbase, *cE0 = cT + NA, *cMMO = cE0 + NA, *cMM1O = cMMO + NA, *cMLC = cMM1O + NA;
  int *cEC = PRE ? cbase : cMLC + NA, *cMS = cEC + NA, *cLIST = cMS + NA;
  int *pre0 = cbase + 2 * NA;
  __shared__ int s_np, s_np2[2], s_next;
  if (tid == 0) { s_np = 0; s_np2[0] = s_np2[1] = 0; s_next = 0; }

  // short sequences: the three tables live in shared memory behind the per-sequence arrays (offset passed by the host), else in HBM
  int *c = tables_smem_off ? reinterpret_cast<int *>(dyn + tables_smem_off) : ws + (size_t)blockIdx.x * ws_slot_ints;
  int *fml = c + (size_t)W * W;
  int *fmlT = fml + (size_t)W * W;
  // c with the inner-pair term of a decomposable interior loop folded in (generic: + mismatchI, 1xn: + mismatch1nI, bulge: + terminalAU)
  int *cG = fmlT + (size_t)W * W, *c1 = cG + (size_t)W * W, *cB = c1 + (size_t)W * W;
#define CG_(i, j) cG[(i) * W + (j)]
#define C1_(i, j) c1[(i) * W + (j)]
#define CB_(i, j) cB[(i) * W + (j)]
#define C_(i, j) c[(i) * W + (j)]
#define M_(i, j) fml[(i) * W + (j)]
#define MT_(j, i) fmlT[(j) * W + (i)]

  // the decomposable interior-loop candidates of cell (i,j) up to loop size smx, this lane's share: per candidate one list entry, one
  // table value, add + min; four (generic) / two in flight per round.  A cell that spans the nick tests u1 <= a, u2 <= bq (p stays
  // on i's strand, q on j's); for every other cell the test is vacuous
  auto decomp = [&](int i, int j, int smx, bool span, int a, int bq, int mmO, int mm1O, int tauO) -> int {
    int e = BF_INF;
    if (smx < 0) return e;
    const int *cij = c + i * W + j;
    auto run = [&](auto uc, auto tc, int outer) {
      constexpr int U = decltype(uc)::value, t = decltype(tc)::value, first = kListStart[t], last = kListStart[t + 1] - 1;
      const int cnt = lcnt[t][smx];
      for (int k0 = first + lane; k0 < first + cnt; k0 += 32 * U) {
        int2 cd[U];
        int cc[U];
#pragma unroll
        for (int u = 0; u < U; u++) cd[u] = lst[min(k0 + 32 * u, last)];
#pragma unroll
        for (int u = 0; u < U; u++) {
          bool ok = k0 + 32 * u < first + cnt;
          if (TWO && span) ok = ok && ((cd[u].y >> 16) & 255) <= a && ((cd[u].y >> 24) & 255) <= bq;
          cc[u] = ok ? cij[cd[u].x] : BF_INF;
        }
#pragma unroll
        for (int u = 0; u < U; u++)
          if (cc[u] < BF_INF) e = min(e, cc[u] + (int)(short)(cd[u].y & 0xffff) + outer);
      }
    };
    run(std::integral_constant<int, 4>(), std::integral_constant<int, 0>(), mmO);
    run(std::integral_constant<int, 2>(), std::integral_constant<int, 1>(), mm1O);
    run(std::integral_constant<int, 2>(), std::integral_constant<int, 2>(), tauO);
    return e;
  };

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int s = s_seq;
    if (s >= b.B) break;
    BfCtx X;
    load_sequence<TWO>(b, s, S, SP, &X, W);
    const int n = X.n, cp = X.cp;
    // spans that are never computed must read as INF
    const int d0 = TWO ? 1 : BF_TURN + 1;
    for (int k = tid; k < d0 * (n + 1); k += blockDim.x) {
      int d = k / (n + 1), i = k % (n + 1) + 1, j = i + d;
      if (j <= n + 1 && i <= n) { M_(i, j) = BF_INF; MT_(j, i) = BF_INF; C_(i, j) = BF_INF; CG_(i, j) = BF_INF; C1_(i, j) = BF_INF; CB_(i, j) = BF_INF; }
    }
    for (int k = tid; k <= n + 2; k += blockDim.x) { fcA[k] = 0; fcB[k] = 0; }
    __syncthreads();

    if constexpr (PRE) {
      // sequence-only terms of diagonal dd into buffer bf: ten tasks per cell (0: pair type, hairpin / nick term, closing-pair terms and
      // the list of pairable cells; 1..9: the shapes evaluated in full), lanes = tasks [32 * chunk, 32 * chunk + 32)
      auto setup = [&](int dd, int chunk, int bf) {
        int *q = pre0 + (size_t)bf * kPreArr * NA;
        const int g = chunk * 32 + lane, i = g / 10 + 1, task = g - (i - 1) * 10, j = i + dd;
        if (i > n - dd) return;
        const int t = bf_ptype<TWO>(X, i, j);
        if (!t) { if (task == 0) q[i] = 0; return; }
        const int si1 = S[i + 1], sj1 = S[j - 1];
        if (task == 0) {
          q[i] = t;
          int e0;
          if (TWO && i < cp && j >= cp) { int a, bb; bf_nick_nb(X, i, j, &a, &bb); e0 = bf_e_ext(T, bf_rtype(t), a, bb); }   // + fcA[i+1] + fcB[j-1] when the cell is computed
          else e0 = bf_e_hairpin(P, T, S, i, j, t);
          q[NA + i] = e0; q[2 * NA + i] = T.mmI[t][si1][sj1]; q[3 * NA + i] = T.mm1nI[t][si1][sj1];
          q[4 * NA + i] = (!TWO || (bf_same<TWO>(X, i, i + 1) && bf_same<TWO>(X, j - 1, j))) ? T.MLclosing + bf_e_mlstem(T, bf_rtype(t), sj1, si1) : BF_INF;
          q[5 * NA + atomicAdd(&s_np2[bf], 1)] = i;
        } else {
          const int pmax = (TWO && i < cp) ? cp - 1 : n, qmin = (TWO && j >= cp) ? cp : 0;
          const int sh = task - 1, u1 = kSpecU1[sh], u2 = kSpecU2[sh], p = i + 1 + u1, qq = j - 1 - u2;
          int e9 = BF_INF;
          if (qq > p && p <= pmax && qq >= qmin) {
            const int t2 = bf_ptype<TWO>(X, p, qq);
            if (t2) e9 = bf_e_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S[p - 1], S[qq + 1]);
          }
          q[(6 + sh) * NA + i] = e9;
        }
      };
      for (int ch = warp; ch * 32 < (n - d0) * 10; ch += NWG) setup(d0, ch, d0 & 1);
      __syncthreads();
      for (int d = d0; d <= n - 1; d++) {
        const int bf = d & 1;
        const int *q = pre0 + (size_t)bf * kPreArr * NA;
        const int *qT = q, *qE0 = q + NA, *qMMO = q + 2 * NA, *qMM1O = q + 3 * NA, *qMLC = q + 4 * NA, *qLIST = q + 5 * NA, *qE9 = q + 6 * NA;
        const int ncell = n - d, np = s_np2[bf];
        const int nfc = (TWO && cp <= n) ? 2 : 0, nset = d + 1 <= n - 1 ? ((n - d - 1) * 10 + 31) / 32 : 0;
        const int total = nfc + nset + np + ncell;
        for (;;) {
          int it = 0;
          if (lane == 0) it = atomicAdd(&s_next, 1);
          it = __shfl_sync(BF_FULL, it, 0);
          if (it >= total) break;
          if (it < nfc) {
            // exterior-style decompositions next to the nick: fcA[k] for segment k..cp-1, fcB[k] for cp..k.  Segment span is d-1, so
            // every c it needs is final; the cells of this diagonal read fcA / fcB at indices written on earlier diagonals only.
            if (it == 0) {
              const int k = cp - d;
              if (k >= 1) {
                int e = BF_INF;
                for (int qq = k + 1 + lane; qq <= cp - 1; qq += 32) {
                  const int t = bf_ptype<TWO>(X, k, qq);
                  if (t) {
                    const int cc = C_(k, qq);
                    if (cc < BF_INF) { int a, bb; bf_ext_nb<TWO>(X, k, qq, &a, &bb); e = min(e, cc + bf_e_ext(T, t, a, bb) + fcA[qq + 1]); }
                  }
                }
                e = bf_warp_min(e);
                if (lane == 0) fcA[k] = min(e, fcA[k + 1]);
              }
            } else {
              const int k = cp + d - 1;
              if (k <= n) {
                int e = BF_INF;
                for (int p = cp + lane; p < k; p += 32) {
                  const int t = bf_ptype<TWO>(X, p, k);
                  if (t) {
                    const int cc = C_(p, k);
                    if (cc < BF_INF) { int a, bb; bf_ext_nb<TWO>(X, p, k, &a, &bb); e = min(e, fcB[p - 1] + cc + bf_e_ext(T, t, a, bb)); }
                  }
                }
                e = bf_warp_min(e);
                if (lane == 0) fcB[k] = min(e, fcB[k - 1]);
              }
            }
          } else if (it < nfc + nset) {
            setup(d + 1, it - nfc, bf ^ 1);
          } else if (it < nfc + nset + np) {
            const int i = qLIST[it - nfc - nset], j = i + d, t = qT[i];
            const int mmO = qMMO[i], mm1O = qMM1O[i], tauO = t > 2 ? T.TerminalAU : 0, mlc = qMLC[i];
            const int smx = min(BF_MAXLOOP, d - 3), kmax = smx >= 0 ? (smx + 1) * (smx + 2) / 2 : 0;   // candidates are ordered by size
            // the unpaired stretches of a regular loop may not contain the nick: p stays on i's strand, q on j's
            const int pmax = (TWO && i < cp) ? cp - 1 : n, qmin = (TWO && j >= cp) ? cp : 0;
            int e = decomp(i, j, smx, TWO && i < cp && j >= cp, pmax - i - 1, j - 1 - qmin, mmO, mm1O, tauO);
            if (lane < min(kmax, 21)) {   // the shapes evaluated in full sit among the first 21 candidates
              const int x = spec21[lane], sh = x >> 24;
              const int p = i + 1 + (x & 255), qq = j - 1 - ((x >> 8) & 255);
              if (sh && p <= pmax && qq >= qmin) {
                const int e9 = qE9[(sh - 1) * NA + i];
                if (e9 < BF_INF) {
                  const int cc = C_(p, qq);
                  if (cc < BF_INF) e = min(e, cc + e9);
                }
              }
            }
            if (mlc < BF_INF) {   // multiloop closed by (i,j)
              int dec = BF_INF;
              const int *rowL = &M_(i + 1, 0);
              const int *rowR = &MT_(j - 1, 0);
              const int ulo = TWO ? i + 2 : i + 2 + BF_TURN + 1, uhi = TWO ? j - 1 : j - 2 - BF_TURN;
              for (int u = ulo + lane; u <= uhi; u += 32) {
                if (TWO && !bf_same<TWO>(X, u - 1, u)) continue;
                dec = min(dec, rowL[u - 1] + rowR[u]);
              }
              if (dec < BF_INF) e = min(e, dec + mlc);
            }
            e = bf_warp_min(e);
            if (lane == 0) {
              int e0 = qE0[i];
              if (TWO && i < cp && j >= cp) e0 += fcA[i + 1] + fcB[j - 1];
              cEC[i] = min(min(e, e0), BF_INF);
            }
          } else {
            const int i = it - nfc - nset - np + 1, j = i + d;
            int m = BF_INF;
            const int *rowL = &M_(i, 0);
            const int *rowR = &MT_(j, 0);
            const int ulo = TWO ? i + 1 : i + 1 + BF_TURN + 1, uhi = TWO ? j : j - 1 - BF_TURN;
            for (int u = ulo + lane; u <= uhi; u += 32) {
              if (TWO && !bf_same<TWO>(X, u - 1, u)) continue;
              m = min(m, rowL[u - 1] + rowR[u]);
            }
            m = bf_warp_min(m);
            if (lane == 0) cMS[i] = m;
          }
        }
        __syncthreads();
        for (int i = 1 + tid; i <= ncell; i += blockDim.x) {
          const int j = i + d, t = qT[i];
          const int e = t ? cEC[i] : BF_INF;
          int m = cMS[i];
          if (e < BF_INF && i > 1 && j < n && bf_same<TWO>(X, i - 1, i) && bf_same<TWO>(X, j, j + 1))
            m = min(m, e + bf_e_mlstem(T, t, S[i - 1], S[j + 1]));
          if (bf_same<TWO>(X, i, i + 1)) m = min(m, M_(i + 1, j) + T.MLbase);
          if (bf_same<TWO>(X, j - 1, j)) m = min(m, M_(i, j - 1) + T.MLbase);
          m = min(m, BF_INF);
          C_(i, j) = e; M_(i, j) = m; MT_(j, i) = m;
          if (e < BF_INF) {
            const int tr = bf_rtype(t), a = S[j + 1], bb = S[i - 1];
            CG_(i, j) = e + T.mmI[tr][a][bb]; C1_(i, j) = e + T.mm1nI[tr][a][bb]; CB_(i, j) = e + (t > 2 ? T.TerminalAU : 0);
          } else {
            CG_(i, j) = BF_INF; C1_(i, j) = BF_INF; CB_(i, j) = BF_INF;
          }
        }
        if (tid == 0) { s_np2[bf] = 0; s_next = 0; }
        __syncthreads();
      }
    } else {
    for (int d = d0; d <= n - 1; d++) {
      if (TWO && cp <= n) {
        // exterior-style decompositions next to the nick: fcA[k] for segment k..cp-1, fcB[k] for cp..k.
        // Segment span is d-1, so every c it needs is final.
        if (warp == 0) {
          int k = cp - d;
          if (k >= 1) {
            int e = BF_INF;
            for (int q = k + 1 + lane; q <= cp - 1; q += 32) {
              int t = bf_ptype<TWO>(X, k, q);
              if (t) {
                int cc = C_(k, q);
                if (cc < BF_INF) { int a, bb; bf_ext_nb<TWO>(X, k, q, &a, &bb); e = min(e, cc + bf_e_ext(T, t, a, bb) + fcA[q + 1]); }
              }
            }
            e = bf_warp_min(e);
            if (lane == 0) fcA[k] = min(e, fcA[k + 1]);
          }
        } else if (warp == 1) {
          int k = cp + d - 1;
          if (k <= n) {
            int e = BF_INF;
            for (int p = cp + lane; p < k; p += 32) {
              int t = bf_ptype<TWO>(X, p, k);
              if (t) {
                int cc = C_(p, k);
                if (cc < BF_INF) { int a, bb; bf_ext_nb<TWO>(X, p, k, &a, &bb); e = min(e, fcB[p - 1] + cc + bf_e_ext(T, t, a, bb)); }
              }
            }
            e = bf_warp_min(e);
            if (lane == 0) fcB[k] = min(e, fcB[k - 1]);
          }
        }
        __syncthreads();
      }
      // Three stages per diagonal.  A (lanes = cells): everything of a cell that depends on the sequence only -- pair type, the hairpin
      // or nick-loop term, the closing pair's terms -- and the list of pairable cells.  B (a warp per item): interior-loop candidates
      // (all but nine shapes decomposed: one table value + a size penalty + a term of the closing pair, as in bf_fill3.cu) and the
      // multiloop-closing split of every pairable cell; the fML split of every cell.  C (lanes = cells): c, fML and the three variants.
      const int ncell = n - d;
      for (int i = 1 + tid; i <= ncell; i += blockDim.x) {
        const int j = i + d;
        const int t = bf_ptype<TWO>(X, i, j);
        cT[i] = t;
        if (t) {
          const int si1 = S[i + 1], sj1 = S[j - 1];
          int e0;
          if (TWO && i < cp && j >= cp) {
            int a, bb; bf_nick_nb(X, i, j, &a, &bb);
            e0 = bf_e_ext(T, bf_rtype(t), a, bb) + fcA[i + 1] + fcB[j - 1];
          } else {
            e0 = bf_e_hairpin(P, T, S, i, j, t);
          }
          cE0[i] = e0; cMMO[i] = T.mmI[t][si1][sj1]; cMM1O[i] = T.mm1nI[t][si1][sj1];
          cMLC[i] = (!TWO || (bf_same<TWO>(X, i, i + 1) && bf_same<TWO>(X, j - 1, j))) ? T.MLclosing + bf_e_mlstem(T, bf_rtype(t), sj1, si1) : BF_INF;
          cLIST[atomicAdd(&s_np, 1)] = i;
        }
      }
      __syncthreads();
      const int np = s_np;
      for (int it = warp; it < np + ncell; it += NWG) {
        if (it < np) {
          const int i = cLIST[it], j = i + d, t = cT[i];
          const int si1 = S[i + 1], sj1 = S[j - 1];
          const int mmO = cMMO[i], mm1O = cMM1O[i], tauO = t > 2 ? T.TerminalAU : 0, mlc = cMLC[i];
          const int smx = min(BF_MAXLOOP, d - 3), kmax = smx >= 0 ? (smx + 1) * (smx + 2) / 2 : 0;   // candidates are ordered by size
          // the unpaired stretches of a regular loop may not contain the nick: p stays on i's strand, q on j's
          const int pmax = (TWO && i < cp) ? cp - 1 : n, qmin = (TWO && j >= cp) ? cp : 0;
          int e = decomp(i, j, smx, TWO && i < cp && j >= cp, pmax - i - 1, j - 1 - qmin, mmO, mm1O, tauO);
          if (lane < min(kmax, 21)) {   // the shapes evaluated in full sit among the first 21 candidates
            const int x = spec21[lane], u1 = x & 255, u2 = (x >> 8) & 255;
            const int p = i + 1 + u1, q = j - 1 - u2;
            if ((x >> 24) && p <= pmax && q >= qmin) {
              const int t2 = bf_ptype<TWO>(X, p, q);
              const int cc = t2 ? C_(p, q) : BF_INF;
              if (cc < BF_INF) e = min(e, cc + bf_e_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1]));
            }
          }
          if (mlc < BF_INF) {   // multiloop closed by (i,j)
            int dec = BF_INF;
            const int *rowL = &M_(i + 1, 0);
            const int *rowR = &MT_(j - 1, 0);
            const int ulo = TWO ? i + 2 : i + 2 + BF_TURN + 1, uhi = TWO ? j - 1 : j - 2 - BF_TURN;
            for (int u = ulo + lane; u <= uhi; u += 32) {
              if (TWO && !bf_same<TWO>(X, u - 1, u)) continue;
              dec = min(dec, rowL[u - 1] + rowR[u]);
            }
            if (dec < BF_INF) e = min(e, dec + mlc);
          }
          e = bf_warp_min(e);
          if (lane == 0) cEC[i] = min(min(e, cE0[i]), BF_INF);
        } else {
          const int i = it - np + 1, j = i + d;
          int m = BF_INF;
          const int *rowL = &M_(i, 0);
          const int *rowR = &MT_(j, 0);
          const int ulo = TWO ? i + 1 : i + 1 + BF_TURN + 1, uhi = TWO ? j : j - 1 - BF_TURN;
          for (int u = ulo + lane; u <= uhi; u += 32) {
            if (TWO && !bf_same<TWO>(X, u - 1, u)) continue;
            m = min(m, rowL[u - 1] + rowR[u]);
          }
          m = bf_warp_min(m);
          if (lane == 0) cMS[i] = m;
        }
      }
      __syncthreads();
      for (int i = 1 + tid; i <= ncell; i += blockDim.x) {
        const int j = i + d, t = cT[i];
        const int e = t ? cEC[i] : BF_INF;
        int m = cMS[i];
        if (e < BF_INF && i > 1 && j < n && bf_same<TWO>(X, i - 1, i) && bf_same<TWO>(X, j, j + 1))
          m = min(m, e + bf_e_mlstem(T, t, S[i - 1], S[j + 1]));
        if (bf_same<TWO>(X, i, i + 1)) m = min(m, M_(i + 1, j) + T.MLbase);
        if (bf_same<TWO>(X, j - 1, j)) m = min(m, M_(i, j - 1) + T.MLbase);
        m = min(m, BF_INF);
        C_(i, j) = e; M_(i, j) = m; MT_(j, i) = m;
        if (e < BF_INF) {
          const int tr = bf_rtype(t), a = S[j + 1], bb = S[i - 1];
          CG_(i, j) = e + T.mmI[tr][a][bb]; C1_(i, j) = e + T.mm1nI[tr][a][bb]; CB_(i, j) = e + (t > 2 ? T.TerminalAU : 0);
        } else {
          CG_(i, j) = BF_INF; C1_(i, j) = BF_INF; CB_(i, j) = BF_INF;
        }
      }
      if (tid == 0) s_np = 0;
      __syncthreads();
    }

    }

    // ---- exterior loop f5 (warp 0), then backtrack (warp 0)
    if (warp == 0) {
      if (lane == 0) f5[0] = 0;
      __syncwarp();
      for (int j = 1; j <= n; j++) {
        int e = BF_INF;
        for (int i = 1 + lane; i < j; i += 32) {
          int t = bf_ptype<TWO>(X, i, j);
          if (!t) continue;
          int cc = C_(i, j);
          if (cc >= BF_INF) continue;
          int a, bb; bf_ext_nb<TWO>(X, i, j, &a, &bb);
          e = min(e, f5[i - 1] + cc + bf_e_ext(T, t, a, bb) + (bf_same<TWO>(X, i, j) ? 0 : T.DuplexInit));
        }
        e = bf_warp_min(e);
        if (lane == 0) f5[j] = min(e, f5[j - 1]);
        __syncwarp();
      }
      if (lane == 0 && out_mfe) out_mfe[s] = f5[n];
    }
    if (out_ss) {
      char *ss = out_ss + (size_t)s * ss_stride;
      for (int k = tid; k < ss_stride; k += blockDim.x) ss[k] = (k < n) ? '.' : 0;
    }
    __syncthreads();
    if (warp == 0 && out_ss) {
      char *ss = out_ss + (size_t)s * ss_stride;
      int sp = 0;
      if (lane == 0) { stk[0].i = 1; stk[0].j = (short)n; stk[0].kind = 0; }
      sp = 1;
      __syncwarp();
      int guard = 0;
      while (sp > 0 && guard++ < 8 * n + 64) {
        BfSector sec = stk[--sp];
        __syncwarp();
        int i = sec.i, j = sec.j;
        bool to_pair = false;
        if (sec.kind == 0) {
          while (j > 0 && f5[j] == f5[j - 1]) j--;
          if (j <= 1) continue;
          int fu = 0;
          for (int base = j - 1; base >= 1 && !fu; base -= 32) {
            int u = base - lane;
            bool ok = false;
            if (u >= 1) {
              int t = bf_ptype<TWO>(X, u, j);
              if (t) {
                int cc = C_(u, j);
                if (cc < BF_INF) {
                  int a, bb; bf_ext_nb<TWO>(X, u, j, &a, &bb);
                  ok = f5[j] == f5[u - 1] + cc + bf_e_ext(T, t, a, bb) + (bf_same<TWO>(X, u, j) ? 0 : T.DuplexInit);
                }
              }
            }
            unsigned mk = __ballot_sync(BF_FULL, ok);
            if (mk) fu = base - (__ffs(mk) - 1);
          }
          if (!fu) break;  // cannot happen for a consistent fill
          if (lane == 0) { stk[sp].i = 1; stk[sp].j = (short)(fu - 1); stk[sp].kind = 0; }
          sp++;
          __syncwarp();
          i = fu; to_pair = true;
        } else if (TWO && sec.kind == 3) {
          while (i < cp && fcA[i] == fcA[i + 1]) i++;
          if (i >= cp) continue;
          int fq = 0;
          for (int base = i + 1; base <= cp - 1 && !fq; base += 32) {
            int q = base + lane;
            bool ok = false;
            if (q <= cp - 1) {
              int t = bf_ptype<TWO>(X, i, q);
              if (t) {
                int cc = C_(i, q);
                if (cc < BF_INF) { int a, bb; bf_ext_nb<TWO>(X, i, q, &a, &bb); ok = fcA[i] == cc + bf_e_ext(T, t, a, bb) + fcA[q + 1]; }
              }
            }
            unsigned mk = __ballot_sync(BF_FULL, ok);
            if (mk) fq = base + (__ffs(mk) - 1);
          }
          if (!fq) break;
          if (lane == 0) { stk[sp].i = (short)(fq + 1); stk[sp].j = 0; stk[sp].kind = 3; }
          sp++;
          __syncwarp();
          j = fq; to_pair = true;
        } else if (TWO && sec.kind == 4) {
          while (j >= cp && fcB[j] == fcB[j - 1]) j--;
          if (j < cp) continue;
          int fp = 0;
          for (int base = j - 1; base >= cp && !fp; base -= 32) {
            int p = base - lane;
            bool ok = false;
            if (p >= cp) {
              int t = bf_ptype<TWO>(X, p, j);
              if (t) {
                int cc = C_(p, j);
                if (cc < BF_INF) { int a, bb; bf_ext_nb<TWO>(X, p, j, &a, &bb); ok = fcB[j] == fcB[p - 1] + cc + bf_e_ext(T, t, a, bb); }
              }
            }
            unsigned mk = __ballot_sync(BF_FULL, ok);
            if (mk) fp = base - (__ffs(mk) - 1);
          }
          if (!fp) break;
          if (lane == 0) { stk[sp].i = 0; stk[sp].j = (short)(fp - 1); stk[sp].kind = 4; }
          sp++;
          __syncwarp();
          i = fp; to_pair = true;
        } else if (sec.kind == 1) {
          while (j > i && bf_same<TWO>(X, j - 1, j) && M_(i, j) == M_(i, j - 1) + T.MLbase) j--;
          while (i < j && bf_same<TWO>(X, i, i + 1) && M_(i, j) == M_(i + 1, j) + T.MLbase) i++;
          const int mij = M_(i, j);
          const int t = bf_ptype<TWO>(X, i, j);
          if (t && C_(i, j) < BF_INF && i > 1 && j < n && bf_same<TWO>(X, i - 1, i) && bf_same<TWO>(X, j, j + 1) &&
              mij == C_(i, j) + bf_e_mlstem(T, t, S[i - 1], S[j + 1])) {
            to_pair = true;
          } else {
            int fu = 0;
            for (int base = i + 1; base <= j && !fu; base += 32) {
              int u = base + lane;
              bool ok = false;
              if (u <= j && bf_same<TWO>(X, u - 1, u)) {
                int l = M_(i, u - 1), r = MT_(j, u);
                ok = l < BF_INF && r < BF_INF && mij == l + r;
              }
              unsigned mk = __ballot_sync(BF_FULL, ok);
              if (mk) fu = base + (__ffs(mk) - 1);
            }
            if (!fu) break;
            if (lane == 0) {
              stk[sp].i = (short)i; stk[sp].j = (short)(fu - 1); stk[sp].kind = 1;
              stk[sp + 1].i = (short)fu; stk[sp + 1].j = (short)j; stk[sp + 1].kind = 1;
            }
            sp += 2;
            __syncwarp();
          }
        } else {
          to_pair = true;  // kind 2
        }
        if (!to_pair) continue;
        // ---- pair (i,j): follow interior loops downwards
        for (;;) {
          if (lane == 0) { ss[i - 1] = '('; ss[j - 1] = ')'; }
          const int t = bf_ptype<TWO>(X, i, j), cij = C_(i, j);
          const int si1 = S[i + 1], sj1 = S[j - 1];
          if (TWO && i < cp && j >= cp) {
            int a, bb; bf_nick_nb(X, i, j, &a, &bb);
            if (cij == bf_e_ext(T, bf_rtype(t), a, bb)) break;  // hairpin-like loop around the nick
          } else if (cij == bf_e_hairpin(P, T, S, i, j, t)) break;
          int fp = 0, fq = 0;
          const int pmax = min(j - 2, i + BF_MAXLOOP + 1);
          for (int p = i + 1; p <= pmax && !fp; p++) {
            if (TWO && !bf_same<TWO>(X, i, p)) break;
            const int minq = max(p + 1, j - i + p - BF_MAXLOOP - 2);
            const int q = j - 1 - lane;
            bool ok = false;
            if (q >= minq && bf_same<TWO>(X, q, j)) {
              int t2 = bf_ptype<TWO>(X, p, q);
              if (t2) {
                int cc = C_(p, q);
                ok = cc < BF_INF && cij == cc + bf_e_intloop(P, T, p - i - 1, j - q - 1, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1]);
              }
            }
            unsigned mk = __ballot_sync(BF_FULL, ok);
            if (mk) { fp = p; fq = j - 1 - (__ffs(mk) - 1); }
          }
          if (fp) { i = fp; j = fq; continue; }
          // multiloop
          int fu = 0;
          if (!TWO || (bf_same<TWO>(X, i, i + 1) && bf_same<TWO>(X, j - 1, j))) {
            const int en = cij - T.MLclosing - bf_e_mlstem(T, bf_rtype(t), sj1, si1);
            for (int base = i + 2; base <= j - 1 && !fu; base += 32) {
              int u = base + lane;
              bool ok = false;
              if (u <= j - 1 && bf_same<TWO>(X, u - 1, u)) {
                int l = M_(i + 1, u - 1), r = MT_(j - 1, u);
                ok = l < BF_INF && r < BF_INF && en == l + r;
              }
              unsigned mk = __ballot_sync(BF_FULL, ok);
              if (mk) fu = base + (__ffs(mk) - 1);
            }
          }
          if (fu) {
            if (lane == 0) {
              stk[sp].i = (short)(i + 1); stk[sp].j = (short)(fu - 1); stk[sp].kind = 1;
              stk[sp + 1].i = (short)fu; stk[sp + 1].j = (short)(j - 1); stk[sp + 1].kind = 1;
            }
            sp += 2;
            __syncwarp();
          } else if (TWO && i < cp && j >= cp) {
            // loop around the nick with stems inside: tried last (tie order pinned by the G5 goldens)
            if (lane == 0) {
              stk[sp].i = (short)(i + 1); stk[sp].j = 0; stk[sp].kind = 3;
              stk[sp + 1].i = 0; stk[sp + 1].j = (short)(j - 1); stk[sp + 1].kind = 4;
            }
            sp += 2;
            __syncwarp();
          }
          break;
        }
      }
    }
  }
#undef C_
#undef M_
#undef MT_
}

// =====================================================================================================
//                                     partition function (inside)
// =====================================================================================================
template <bool TWO, int NWG, bool PRE>
__global__ void __launch_bounds__(NWG * 32) bf_k_pf(const BfParams *__restrict__ P, BfBatchDev b, double *ws, size_t ws_slot_dbl,
                                                      int wstride, int *work_counter, const int *mfe_for_scale, double *out5,
                                                      unsigned tables_smem_off) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallD T;
  __shared__ int s_seq;
  __shared__ double s_lnscale;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int W = wstride;
  bf_stage(&T, &P->sd);
  // decomposable interior-loop candidates in three size-ordered lists as in bf_k_mfe: x = table-entry offset relative to the cell's,
  // y = u1 << 16 | u2 << 24; the weight of an entry, scale included, is rebuilt for every sequence (lw)
  __shared__ int2 lst[kNDecomp];
  __shared__ double lw[kNDecomp];
  __shared__ short lcnt[3][32];
  __shared__ int spec21[32];
  for (int k = tid; k < kNDecomp; k += blockDim.x) {
    const int u1 = c_list_u1[k], u2 = c_list_u2[k], t = k < 375 ? 0 : k < 429 ? 1 : 2;
    lst[k] = make_int2((3 + t) * W * W + (1 + u1) * W - (1 + u2), u1 << 16 | u2 << 24);
  }
  for (int k = tid; k < 96; k += blockDim.x) lcnt[k >> 5][k & 31] = c_list_cnt[k >> 5][k & 31];
  if (tid < 32) {
    int shape = 0;
    for (int q = 0; q < 9; q++) if (kSpecK[q] == tid) shape = q + 1;
    spec21[tid] = tid < 21 ? (c_cand_u1[tid] | c_cand_u2[tid] << 8 | shape << 24) : 0;
  }

  const int nmax = W - 2;
  double *scl = reinterpret_cast<double *>(dyn);  // scale^-k
  double *bu = scl + (nmax + 4);                   // (B(MLbase)/scale)^k
  double *q5 = bu + (nmax + 4);
  double *qA = q5 + (nmax + 4);
  double *qB = qA + (nmax + 4);
  // per-cell arrays of the diagonal in work (index = i)
  // !PRE: cB0 cXMMO cXMM1O cXMLC cQBr cQS | cT cLIST | S SP.   PRE (see bf_k_mfe): cQBr cQS, two buffers of kPreArrD arrays of doubles
  // cB0 cXMMO cXMM1O cXMLC cXE9[9] | two buffers of cT cLIST | S SP
  const int NA = nmax + 4;
  double *dbase = qB + NA;
  double *cB0 = dbase, *cXMMO = cB0 + NA, *cXMM1O = cXMMO + NA, *cXMLC = cXMM1O + NA;
  double *cQBr = PRE ? dbase : cXMLC + NA, *cQS = cQBr + NA;
  double *pre0 = dbase + 2 * NA;
  int *ibase = reinterpret_cast<int *>(PRE ? pre0 + (size_t)2 * kPreArrD * NA : cQS + NA);
  int *cT = ibase, *cLIST = cT + NA;
  uint8_t *S = reinterpret_cast<uint8_t *>(ibase + (PRE ? 4 : 2) * NA);
  uint8_t *SP = S + align_up(nmax + 2, 16);
  __shared__ int s_np, s_np2[2], s_next;
  if (tid == 0) { s_np = 0; s_np2[0] = s_np2[1] = 0; s_next = 0; }

  double *qb = tables_smem_off ? reinterpret_cast<double *>(dyn + tables_smem_off) : ws + (size_t)blockIdx.x * ws_slot_dbl;
  double *qm = qb + (size_t)W * W;
  double *qm1T = qm + (size_t)W * W;  // qm1T[j][i] = qm1[i][j]
  double *qG = qm1T + (size_t)W * W, *q1 = qG + (size_t)W * W, *qBB = q1 + (size_t)W * W;   // qb x inner-pair factor (see bf_k_mfe)
#define QG_(i, j) qG[(i) * W + (j)]
#define Q1_(i, j) q1[(i) * W + (j)]
#define QBB_(i, j) qBB[(i) * W + (j)]
#define QB_(i, j) qb[(i) * W + (j)]
#define QM_(i, j) qm[(i) * W + (j)]
#define QM1T_(j, i) qm1T[(j) * W + (i)]

  // the decomposable interior-loop candidates of cell (i,j) up to loop size smx, this lane's share (see bf_k_mfe); the closing pair's
  // factor multiplies the sum of a list once
  auto decomp = [&](int i, int j, int smx, bool span, int a, int bq, double xmmO, double xmm1O, double xtauO) -> double {
    double acc = 0.0;
    if (smx < 0) return acc;
    const double *qij = qb + i * W + j;
    auto run = [&](auto uc, auto tc, double outer) {
      constexpr int U = decltype(uc)::value, t = decltype(tc)::value, first = kListStart[t], last = kListStart[t + 1] - 1;
      const int cnt = lcnt[t][smx];
      double part = 0.0;
      for (int k0 = first + lane; k0 < first + cnt; k0 += 32 * U) {
        int2 cd[U];
        double cw[U], v[U];
#pragma unroll
        for (int u = 0; u < U; u++) { const int kk = min(k0 + 32 * u, last); cd[u] = lst[kk]; cw[u] = lw[kk]; }
#pragma unroll
        for (int u = 0; u < U; u++) {
          bool ok = k0 + 32 * u < first + cnt;
          if (TWO && span) ok = ok && ((cd[u].y >> 16) & 255) <= a && ((cd[u].y >> 24) & 255) <= bq;
          v[u] = ok ? qij[cd[u].x] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < U; u++) part = fma(v[u], cw[u], part);
      }
      acc = fma(part, outer, acc);
    };
    run(std::integral_constant<int, 4>(), std::integral_constant<int, 0>(), xmmO);
    run(std::integral_constant<int, 2>(), std::integral_constant<int, 1>(), xmm1O);
    run(std::integral_constant<int, 2>(), std::integral_constant<int, 2>(), xtauO);
    return acc;
  };

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int s = s_seq;
    if (s >= b.B) break;
    BfCtx X;
    load_sequence<TWO>(b, s, S, SP, &X, W);
    const int n = X.n, cp = X.cp;
    if (tid == 0) {
      // per-nucleotide scale: from the MFE when available (ViennaRNA exp_params_rescale, sfact 1.07),
      // else ViennaRNA's default estimate of -185 cal/mol per nucleotide
      double lns = 185.0 / T.kT;
      if (mfe_for_scale && n > 0) {
        double m = (double)mfe_for_scale[s] * 10.0;  // cal/mol
        if (m < 0.0) lns = -1.07 * m / T.kT / (double)n;
        if (lns < 185.0 / T.kT * 0.25) lns = 185.0 / T.kT * 0.25;
      }
      s_lnscale = lns;
      const double sc = exp(-lns), bs = T.x_MLbase * sc;
      scl[0] = 1.0; bu[0] = 1.0;
      for (int k = 1; k <= n + 2; k++) { scl[k] = scl[k - 1] * sc; bu[k] = bu[k - 1] * bs; }
    }
    const int d0 = TWO ? 1 : BF_TURN + 1;
    for (int k = tid; k < d0 * (n + 1); k += blockDim.x) {
      int d = k / (n + 1), i = k % (n + 1) + 1, j = i + d;
      if (j <= n + 1 && i <= n) { QB_(i, j) = 0.0; QM_(i, j) = 0.0; QM1T_(j, i) = 0.0; QG_(i, j) = 0.0; Q1_(i, j) = 0.0; QBB_(i, j) = 0.0; }
    }
    for (int k = tid; k <= n + 2; k += blockDim.x) { qA[k] = 0.0; qB[k] = 0.0; }
    __syncthreads();
    for (int k = tid; k < kNDecomp; k += blockDim.x) {   // weights of the decomposable candidates at this sequence's scale
      const int u1 = (lst[k].y >> 16) & 255, u2 = (lst[k].y >> 24) & 255, sz = u1 + u2;
      const double w = k >= 429 ? T.x_bulge[sz] : k >= 375 ? T.x_interior[sz] * T.x_ninio[sz - 2] : T.x_interior[sz] * T.x_ninio[abs(u1 - u2)];
      lw[k] = w * exp(-s_lnscale * (sz + 2));
    }
    if (TWO && cp <= n && tid == 0) { qA[cp] = 1.0; qB[cp - 1] = 1.0; }
    __syncthreads();

    if constexpr (PRE) {
      auto setup = [&](int dd, int chunk, int bf) {   // ten tasks per cell, lanes = tasks (see bf_k_mfe)
        double *q = pre0 + (size_t)bf * kPreArrD * NA;
        int *qi = ibase + (size_t)bf * 2 * NA;
        const int g = chunk * 32 + lane, i = g / 10 + 1, task = g - (i - 1) * 10, j = i + dd;
        if (i > n - dd) return;
        const int t = bf_ptype<TWO>(X, i, j);
        if (!t) { if (task == 0) qi[i] = 0; return; }
        const int si1 = S[i + 1], sj1 = S[j - 1];
        if (task == 0) {
          qi[i] = t;
          double b0;
          if (TWO && i < cp && j >= cp) { int a, bb; bf_nick_nb(X, i, j, &a, &bb); b0 = bf_x_ext(T, bf_rtype(t), a, bb) * scl[2]; }   // x qA[i+1] x qB[j-1] when the cell is computed
          else b0 = bf_x_hairpin(P, T, S, i, j, t) * scl[dd + 1];
          q[i] = b0; q[NA + i] = T.x_mmI[t][si1][sj1]; q[2 * NA + i] = T.x_mm1nI[t][si1][sj1];
          q[3 * NA + i] = (!TWO || (bf_same<TWO>(X, i, i + 1) && bf_same<TWO>(X, j - 1, j))) ? T.x_MLclosing * bf_x_mlstem(T, bf_rtype(t), sj1, si1) * scl[2] : 0.0;
          qi[NA + atomicAdd(&s_np2[bf], 1)] = i;
        } else {
          const int pmax = (TWO && i < cp) ? cp - 1 : n, qmin = (TWO && j >= cp) ? cp : 0;
          const int sh = task - 1, u1 = kSpecU1[sh], u2 = kSpecU2[sh], p = i + 1 + u1, qq = j - 1 - u2;
          double x9 = 0.0;
          if (qq > p && p <= pmax && qq >= qmin) {
            const int t2 = bf_ptype<TWO>(X, p, qq);
            if (t2) x9 = bf_x_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S[p - 1], S[qq + 1]) * scl[u1 + u2 + 2];
          }
          q[(4 + sh) * NA + i] = x9;
        }
      };
      for (int ch = warp; ch * 32 < (n - d0) * 10; ch += NWG) setup(d0, ch, d0 & 1);
      __syncthreads();
      for (int d = d0; d <= n - 1; d++) {
        const int bf = d & 1;
        const double *q = pre0 + (size_t)bf * kPreArrD * NA;
        const double *qB0 = q, *qXMMO = q + NA, *qXMM1O = q + 2 * NA, *qXMLC = q + 3 * NA, *qXE9 = q + 4 * NA;
        const int *qT = ibase + (size_t)bf * 2 * NA, *qLIST = qT + NA;
        const int ncell = n - d, np = s_np2[bf];
        const int nfc = (TWO && cp <= n) ? 2 : 0, nset = d + 1 <= n - 1 ? ((n - d - 1) * 10 + 31) / 32 : 0;
        const int total = nfc + nset + np + ncell;
        for (;;) {
          int it = 0;
          if (lane == 0) it = atomicAdd(&s_next, 1);
          it = __shfl_sync(BF_FULL, it, 0);
          if (it >= total) break;
          if (it < nfc) {
            if (it == 0) {
              const int k = cp - d;
              if (k >= 1) {
                double sum = 0.0;
                for (int qq = k + 1 + lane; qq <= cp - 1; qq += 32) {
                  const int t = bf_ptype<TWO>(X, k, qq);
                  if (t) { int a, bb; bf_ext_nb<TWO>(X, k, qq, &a, &bb); sum += QB_(k, qq) * bf_x_ext(T, t, a, bb) * qA[qq + 1]; }
                }
                sum = bf_warp_sum(sum);
                if (lane == 0) qA[k] = sum + qA[k + 1] * scl[1];
              }
            } else {
              const int k = cp + d - 1;
              if (k <= n) {
                double sum = 0.0;
                for (int p = cp + lane; p < k; p += 32) {
                  const int t = bf_ptype<TWO>(X, p, k);
                  if (t) { int a, bb; bf_ext_nb<TWO>(X, p, k, &a, &bb); sum += qB[p - 1] * QB_(p, k) * bf_x_ext(T, t, a, bb); }
                }
                sum = bf_warp_sum(sum);
                if (lane == 0) qB[k] = sum + qB[k - 1] * scl[1];
              }
            }
          } else if (it < nfc + nset) {
            setup(d + 1, it - nfc, bf ^ 1);
          } else if (it < nfc + nset + np) {
            const int i = qLIST[it - nfc - nset], j = i + d, t = qT[i];
            const double xmmO = qXMMO[i], xmm1O = qXMM1O[i], xtauO = t > 2 ? T.x_TerminalAU : 1.0, xmlc = qXMLC[i];
            const int smx = min(BF_MAXLOOP, d - 3), kmax = smx >= 0 ? (smx + 1) * (smx + 2) / 2 : 0;   // candidates are ordered by size
            const int pmax = (TWO && i < cp) ? cp - 1 : n, qmin = (TWO && j >= cp) ? cp : 0;
            double acc = decomp(i, j, smx, TWO && i < cp && j >= cp, pmax - i - 1, j - 1 - qmin, xmmO, xmm1O, xtauO);
            if (lane < min(kmax, 21)) {   // the shapes evaluated in full sit among the first 21 candidates
              const int x = spec21[lane], sh = x >> 24;
              const int p = i + 1 + (x & 255), qq = j - 1 - ((x >> 8) & 255);
              if (sh && p <= pmax && qq >= qmin) acc += QB_(p, qq) * qXE9[(sh - 1) * NA + i];
            }
            if (xmlc != 0.0) {
              double dec = 0.0;
              const double *rowL = &QM_(i + 1, 0);
              const double *rowR = &QM1T_(j - 1, 0);
              const int ulo = TWO ? i + 2 : i + 2 + BF_TURN + 1, uhi = TWO ? j - 1 : j - 2 - BF_TURN;
              for (int u = ulo + lane; u <= uhi; u += 32) {
                if (TWO && !bf_same<TWO>(X, u - 1, u)) continue;
                dec += rowL[u - 1] * rowR[u];
              }
              acc += dec * xmlc;
            }
            acc = bf_warp_sum(acc);
            if (lane == 0) {
              double b0 = qB0[i];
              if (TWO && i < cp && j >= cp) b0 *= qA[i + 1] * qB[j - 1];
              cQBr[i] = acc + b0;
            }
          } else {
            // qm[i][j] - qm1[i][j] = sum_u (bu[u-i] + qm[i][u-1]) * qm1[u][j]
            const int i = it - nfc - nset - np + 1, j = i + d;
            double sum = 0.0;
            const double *rowL = &QM_(i, 0);
            const double *rowR = &QM1T_(j, 0);
            const int uhi = TWO ? j : j - BF_TURN - 1;
            for (int u = i + 1 + lane; u <= uhi; u += 32) {
              double left = 0.0;
              if (!TWO || bf_same<TWO>(X, i, u)) left = bu[u - i];
              if (!TWO || bf_same<TWO>(X, u - 1, u)) left += rowL[u - 1];
              sum += left * rowR[u];
            }
            sum = bf_warp_sum(sum);
            if (lane == 0) cQS[i] = sum;
          }
        }
        __syncthreads();
        for (int i = 1 + tid; i <= ncell; i += blockDim.x) {
          const int j = i + d, t = qT[i];
          const double qbij = t ? cQBr[i] : 0.0;
          // qm1[i][j]: exactly one stem, starting at i, unpaired tail up to j
          double qm1ij = 0.0;
          if (bf_same<TWO>(X, j - 1, j)) qm1ij = QM1T_(j - 1, i) * bu[1];
          if (t && i > 1 && j < n && bf_same<TWO>(X, i - 1, i) && bf_same<TWO>(X, j, j + 1)) qm1ij += qbij * bf_x_mlstem(T, t, S[i - 1], S[j + 1]);
          QB_(i, j) = qbij; QM_(i, j) = cQS[i] + qm1ij; QM1T_(j, i) = qm1ij;
          if (t) {
            const int tr = bf_rtype(t), a = S[j + 1], bb = S[i - 1];
            QG_(i, j) = qbij * T.x_mmI[tr][a][bb]; Q1_(i, j) = qbij * T.x_mm1nI[tr][a][bb]; QBB_(i, j) = qbij * (t > 2 ? T.x_TerminalAU : 1.0);
          } else {
            QG_(i, j) = 0.0; Q1_(i, j) = 0.0; QBB_(i, j) = 0.0;
          }
        }
        if (tid == 0) { s_np2[bf] = 0; s_next = 0; }
        __syncthreads();
      }
    } else {
    for (int d = d0; d <= n - 1; d++) {
      if (TWO && cp <= n) {
        if (warp == 0) {
          int k = cp - d;
          if (k >= 1) {
            double sum = 0.0;
            for (int q = k + 1 + lane; q <= cp - 1; q += 32) {
              int t = bf_ptype<TWO>(X, k, q);
              if (t) { int a, bb; bf_ext_nb<TWO>(X, k, q, &a, &bb); sum += QB_(k, q) * bf_x_ext(T, t, a, bb) * qA[q + 1]; }
            }
            sum = bf_warp_sum(sum);
            if (lane == 0) qA[k] = sum + qA[k + 1] * scl[1];
          }
        } else if (warp == 1) {
          int k = cp + d - 1;
          if (k <= n) {
            double sum = 0.0;
            for (int p = cp + lane; p < k; p += 32) {
              int t = bf_ptype<TWO>(X, p, k);
              if (t) { int a, bb; bf_ext_nb<TWO>(X, p, k, &a, &bb); sum += qB[p - 1] * QB_(p, k) * bf_x_ext(T, t, a, bb); }
            }
            sum = bf_warp_sum(sum);
            if (lane == 0) qB[k] = sum + qB[k - 1] * scl[1];
          }
        }
        __syncthreads();
      }
      // the three stages of bf_k_mfe, with sums of Boltzmann weights
      const int ncell = n - d;
      for (int i = 1 + tid; i <= ncell; i += blockDim.x) {
        const int j = i + d;
        const int t = bf_ptype<TWO>(X, i, j);
        cT[i] = t;
        if (t) {
          const int si1 = S[i + 1], sj1 = S[j - 1];
          double b0;
          if (TWO && i < cp && j >= cp) {
            int a, bb; bf_nick_nb(X, i, j, &a, &bb);
            b0 = bf_x_ext(T, bf_rtype(t), a, bb) * qA[i + 1] * qB[j - 1] * scl[2];
          } else {
            b0 = bf_x_hairpin(P, T, S, i, j, t) * scl[d + 1];
          }
          cB0[i] = b0; cXMMO[i] = T.x_mmI[t][si1][sj1]; cXMM1O[i] = T.x_mm1nI[t][si1][sj1];
          cXMLC[i] = (!TWO || (bf_same<TWO>(X, i, i + 1) && bf_same<TWO>(X, j - 1, j))) ? T.x_MLclosing * bf_x_mlstem(T, bf_rtype(t), sj1, si1) * scl[2] : 0.0;
          cLIST[atomicAdd(&s_np, 1)] = i;
        }
      }
      __syncthreads();
      const int np = s_np;
      for (int it = warp; it < np + ncell; it += NWG) {
        if (it < np) {
          const int i = cLIST[it], j = i + d, t = cT[i];
          const int si1 = S[i + 1], sj1 = S[j - 1];
          const double xmmO = cXMMO[i], xmm1O = cXMM1O[i], xtauO = t > 2 ? T.x_TerminalAU : 1.0, xmlc = cXMLC[i];
          const int smx = min(BF_MAXLOOP, d - 3), kmax = smx >= 0 ? (smx + 1) * (smx + 2) / 2 : 0;   // candidates are ordered by size
          const int pmax = (TWO && i < cp) ? cp - 1 : n, qmin = (TWO && j >= cp) ? cp : 0;
          double acc = decomp(i, j, smx, TWO && i < cp && j >= cp, pmax - i - 1, j - 1 - qmin, xmmO, xmm1O, xtauO);
          if (lane < min(kmax, 21)) {   // the shapes evaluated in full sit among the first 21 candidates
            const int x = spec21[lane], u1 = x & 255, u2 = (x >> 8) & 255;
            const int p = i + 1 + u1, q = j - 1 - u2;
            if ((x >> 24) && p <= pmax && q >= qmin) {
              const int t2 = bf_ptype<TWO>(X, p, q);
              if (t2) acc += QB_(p, q) * bf_x_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1]) * scl[u1 + u2 + 2];
            }
          }
          if (xmlc != 0.0) {
            double dec = 0.0;
            const double *rowL = &QM_(i + 1, 0);
            const double *rowR = &QM1T_(j - 1, 0);
            const int ulo = TWO ? i + 2 : i + 2 + BF_TURN + 1, uhi = TWO ? j - 1 : j - 2 - BF_TURN;
            for (int u = ulo + lane; u <= uhi; u += 32) {
              if (TWO && !bf_same<TWO>(X, u - 1, u)) continue;
              dec += rowL[u - 1] * rowR[u];
            }
            acc += dec * xmlc;
          }
          acc = bf_warp_sum(acc);
          if (lane == 0) cQBr[i] = acc + cB0[i];
        } else {
          // qm[i][j] - qm1[i][j] = sum_u (bu[u-i] + qm[i][u-1]) * qm1[u][j]
          const int i = it - np + 1, j = i + d;
          double sum = 0.0;
          const double *rowL = &QM_(i, 0);
          const double *rowR = &QM1T_(j, 0);
          const int uhi = TWO ? j : j - BF_TURN - 1;
          for (int u = i + 1 + lane; u <= uhi; u += 32) {
            double left = 0.0;
            if (!TWO || bf_same<TWO>(X, i, u)) left = bu[u - i];
            if (!TWO || bf_same<TWO>(X, u - 1, u)) left += rowL[u - 1];
            sum += left * rowR[u];
          }
          sum = bf_warp_sum(sum);
          if (lane == 0) cQS[i] = sum;
        }
      }
      __syncthreads();
      for (int i = 1 + tid; i <= ncell; i += blockDim.x) {
        const int j = i + d, t = cT[i];
        const double qbij = t ? cQBr[i] : 0.0;
        // qm1[i][j]: exactly one stem, starting at i, unpaired tail up to j
        double qm1ij = 0.0;
        if (bf_same<TWO>(X, j - 1, j)) qm1ij = QM1T_(j - 1, i) * bu[1];
        if (t && i > 1 && j < n && bf_same<TWO>(X, i - 1, i) && bf_same<TWO>(X, j, j + 1)) qm1ij += qbij * bf_x_mlstem(T, t, S[i - 1], S[j + 1]);
        QB_(i, j) = qbij; QM_(i, j) = cQS[i] + qm1ij; QM1T_(j, i) = qm1ij;
        if (t) {
          const int tr = bf_rtype(t), a = S[j + 1], bb = S[i - 1];
          QG_(i, j) = qbij * T.x_mmI[tr][a][bb]; Q1_(i, j) = qbij * T.x_mm1nI[tr][a][bb]; QBB_(i, j) = qbij * (t > 2 ? T.x_TerminalAU : 1.0);
        } else {
          QG_(i, j) = 0.0; Q1_(i, j) = 0.0; QBB_(i, j) = 0.0;
        }
      }
      if (tid == 0) s_np = 0;
      __syncthreads();
    }

    }

    if (warp == 0) {
      if (lane == 0) q5[0] = 1.0;
      __syncwarp();
      for (int j = 1; j <= n; j++) {
        double sum = 0.0;
        for (int i = 1 + lane; i < j; i += 32) {
          int t = bf_ptype<TWO>(X, i, j);
          if (!t) continue;
          int a, bb; bf_ext_nb<TWO>(X, i, j, &a, &bb);
          sum += q5[i - 1] * QB_(i, j) * bf_x_ext(T, t, a, bb);
        }
        sum = bf_warp_sum(sum);
        if (lane == 0) q5[j] = sum + q5[j - 1] * scl[1];
        __syncwarp();
      }
      if (lane == 0 && out5) {
        const double kT = T.kT, lns = s_lnscale;
        double *o = out5 + (size_t)s * 5;
        o[0] = o[1] = o[2] = o[3] = 0.0;
        o[4] = -kT * (log(q5[n]) + n * lns) / 1000.0;
        if (TWO && cp <= n) {
          const int nA = cp - 1, nB = n - cp + 1;
          const double QA = qA[1], QBv = qB[n];
          double QAB = (q5[n] - QA * QBv) * T.x_DuplexInit;
          bool sym = (nA == nB);
          for (int k = 1; sym && k <= nA; k++) sym = (S[k] == S[nA + k]);
          if (sym) QAB *= 0.5;
          const double QT = QA * QBv + QAB;
          o[0] = -kT * (log(QA) + nA * lns) / 1000.0;
          o[1] = -kT * (log(QBv) + nB * lns) / 1000.0;
          o[2] = (QAB > 1e-17) ? -kT * (log(QAB) + n * lns) / 1000.0 : 999.0;
          o[3] = -kT * (log(QT) + n * lns) / 1000.0;
        }
      }
    }
  }
#undef QB_
#undef QM_
#undef QM1T_
}

// =====================================================================================================
//                                        eval_structure
// =====================================================================================================
// One CTA per (sequence, target).  Thread 0 matches brackets, then every thread scores the loops
// closed by the pairs it owns; a block reduction adds them up.
__global__ void __launch_bounds__(128) bf_k_eval(const BfParams *__restrict__ P, BfBatchDev b, const char *targets, int n_targets,
                                                 int tstride, int *out_e) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallI T;
  __shared__ int s_bad, s_sum;
  const int s = blockIdx.x / n_targets, k = blockIdx.x % n_targets;
  if (s >= b.B) return;
  const int tid = threadIdx.x;
  const int nmax = b.stride;
  short *pt = reinterpret_cast<short *>(dyn);
  short *stk = pt + (nmax + 4);
  uint8_t *S = reinterpret_cast<uint8_t *>(stk + (nmax + 4));
  uint8_t *SP = S + align_up(nmax + 2, 16);
  bf_stage(&T, &P->si);
  BfCtx X;
  load_sequence<true>(b, s, S, SP, &X, nmax + 2);
  const int n = X.n, cp = X.cp;
  const char *db = targets + ((size_t)s * n_targets + k) * tstride;
  for (int i = tid; i <= n + 1; i += blockDim.x) pt[i] = 0;
  if (tid == 0) { s_bad = 0; s_sum = 0; }
  __syncthreads();
  if (tid == 0) {
    int sp = 0;
    for (int i = 1; i <= n; i++) {
      char ch = db[i - 1];
      if (ch == '(') stk[sp++] = (short)i;
      else if (ch == ')') {
        if (!sp) { s_bad = 1; break; }
        int o = stk[--sp];
        pt[o] = (short)i; pt[i] = (short)o;
      }
    }
    if (sp) s_bad = 1;
  }
  __syncthreads();
  if (s_bad) { if (tid == 0) out_e[(size_t)s * n_targets + k] = BF_INF; return; }
  int e = 0;
  if (tid == 0) {
    // exterior loop
    bool connected = false;
    for (int i = 1; i <= n; i++) {
      int j = pt[i];
      if (j > i) {
        int t = bf_ptype_bases(S[i], S[j]); if (!t) t = 7;
        int a, bb; bf_ext_nb<true>(X, i, j, &a, &bb);
        e += bf_e_ext(T, t, a, bb);
        i = j;
      }
    }
    for (int i = 1; i < cp && !connected; i++) if (pt[i] >= cp) connected = true;
    if (connected && cp <= n) e += T.DuplexInit;
  }
  for (int i = 1 + tid; i <= n; i += blockDim.x) {
    const int j = pt[i];
    if (j <= i) continue;
    int t = bf_ptype_bases(S[i], S[j]); if (!t) t = 7;
    int nstem = 0, p1 = 0, q1 = 0, mlsum = 0, extsum = 0, unp = 0, prev = i;
    bool nick = false;
    for (int x = i + 1; x < j;) {
      if (pt[x] > x) {
        const int p = x, q = pt[x];
        int t2 = bf_ptype_bases(S[p], S[q]); if (!t2) t2 = 7;
        if (prev < cp && p >= cp) nick = true;
        if (!nstem) { p1 = p; q1 = q; }
        nstem++;
        mlsum += bf_e_mlstem(T, t2, S[p - 1], S[q + 1]);
        int a, bb; bf_ext_nb<true>(X, p, q, &a, &bb);
        extsum += bf_e_ext(T, t2, a, bb);
        prev = q; x = q + 1;
      } else { unp++; x++; }
    }
    if (prev < cp && j >= cp) nick = true;
    if (nick) {
      int a, bb; bf_nick_nb(X, i, j, &a, &bb);
      e += bf_e_ext(T, bf_rtype(t), a, bb) + extsum;
    } else if (nstem == 0) {
      e += bf_e_hairpin(P, T, S, i, j, t);
    } else if (nstem == 1) {
      int t2 = bf_ptype_bases(S[q1], S[p1]); if (!t2) t2 = 7;
      e += bf_e_intloop(P, T, p1 - i - 1, j - q1 - 1, t, t2, S[i + 1], S[j - 1], S[p1 - 1], S[q1 + 1]);
    } else {
      e += T.MLclosing + bf_e_mlstem(T, bf_rtype(t), S[j - 1], S[i + 1]) + mlsum + unp * T.MLbase;
    }
  }
  // INF-safe block sum: clamp each partial so that a forbidden loop (hairpin < 3) stays recognisable
  e = __reduce_add_sync(BF_FULL, e);
  if ((tid & 31) == 0) atomicAdd(&s_sum, e);
  __syncthreads();
  if (tid == 0) out_e[(size_t)s * n_targets + k] = s_sum;
}

}  // namespace

// =====================================================================================================
//                                        host-side launchers
// =====================================================================================================
static bool g_cand_uploaded = false;

cudaError_t bf_upload_constants() {
  if (g_cand_uploaded) return cudaSuccess;
  uint8_t u1[BF_NCAND], u2[BF_NCAND];
  int k = 0;
  // ordered by loop size u1 + u2: a cell of span d only has candidates up to size d - 3, i.e. the first (d-2)(d-1)/2 entries
  for (int sz = 0; sz <= BF_MAXLOOP; sz++)
    for (int a = 0; a <= sz; a++) { u1[k] = (uint8_t)a; u2[k] = (uint8_t)(sz - a); k++; }
  cudaError_t e = cudaMemcpyToSymbol(c_cand_u1, u1, sizeof u1);
  if (e != cudaSuccess) return e;
  e = cudaMemcpyToSymbol(c_cand_u2, u2, sizeof u2);
  if (e != cudaSuccess) return e;
  // the decomposable candidates by kind, each list ordered by size (kinds as in the kernels: the nine special shapes are left out)
  uint8_t l1[kNDecomp], l2[kNDecomp];
  short cnt[3][32];
  int pos[3] = {kListStart[0], kListStart[1], kListStart[2]};
  for (int sz = 0; sz <= BF_MAXLOOP; sz++) {
    for (int a = 0; a <= sz; a++) {
      const int b = sz - a;
      const bool special = sz <= 1 || (a == 1 && b == 1) || (sz == 3 && a >= 1 && b >= 1) || (a == 2 && b == 2) || (sz == 5 && (a == 2 || a == 3));
      if (special) continue;
      const int t = (a == 0 || b == 0) ? 2 : (a == 1 || b == 1) ? 1 : 0;
      if (pos[t] >= kListStart[t + 1]) return cudaErrorInvalidValue;
      l1[pos[t]] = (uint8_t)a; l2[pos[t]] = (uint8_t)b; pos[t]++;
    }
    for (int t = 0; t < 3; t++) cnt[t][sz] = (short)(pos[t] - kListStart[t]);
  }
  for (int t = 0; t < 3; t++) { if (pos[t] != kListStart[t + 1]) return cudaErrorInvalidValue; cnt[t][31] = cnt[t][30]; }
  e = cudaMemcpyToSymbol(c_list_u1, l1, sizeof l1);
  if (e != cudaSuccess) return e;
  e = cudaMemcpyToSymbol(c_list_u2, l2, sizeof l2);
  if (e != cudaSuccess) return e;
  e = cudaMemcpyToSymbol(c_list_cnt, cnt, sizeof cnt);
  if (e == cudaSuccess) g_cand_uploaded = true;
  return e;
}

static size_t bf_mfe_slot_ints(int wstride) { return (size_t)6 * wstride * wstride; }      // c, fML, fML^T + the three inner-term variants of c
static size_t bf_pf_slot_doubles(int wstride) { return (size_t)6 * wstride * wstride; }   // qb, qm, qm1^T + the three variants of qb

// The generic kernels (two strands; any length the fill path does not cover) keep three W x W tables per CTA.  Short sequences --
// the reference's two-strand examples are 17 & 18 nt -- fit in shared memory next to the per-sequence arrays, which takes the L2
// round trip out of every table access.  Capped so that at least two CTAs share an SM.
static bool gen_wide(int B, int sms, const BfOpts &o) { return B > 0 && B <= sms && o.wide != 0; }
// the two-barrier variants: batches that leave SMs idle, i.e. latency matters (measured: 17 & 18 nt x 64 MFE 0.164 -> 0.150 ms, but
// 50 & 50 nt x 4096 16.7 -> 25.5 ms)
static bool gen_pre(int wstride, bool wide) { return wide && wstride - 2 <= kPreMax; }
static size_t mfe_smem(int wstride, bool pre) {
  size_t nmax = wstride - 2;
  const size_t arrays = pre ? 3 + 2 + 2 * kPreArr : 3 + 8;
  return 2 * ((nmax + 2 + 15) / 16 * 16) + arrays * (nmax + 4) * sizeof(int) + (2 * nmax + 16) * sizeof(BfSector);
}
static size_t pf_smem(int wstride, bool pre) {
  size_t nmax = wstride - 2;
  return (pre ? 5 + 2 + 2 * kPreArrD : 5 + 6) * (nmax + 4) * sizeof(double) + (pre ? 4 : 2) * (nmax + 4) * sizeof(int) + 2 * ((nmax + 2 + 15) / 16 * 16);
}
static const size_t kGenTablesCap = 100 * 1024;
static unsigned mfe_tables_off(int wstride, bool pre) {   // 0: tables in HBM
  const size_t base = (mfe_smem(wstride, pre) + 15) / 16 * 16;
  return base + bf_mfe_slot_ints(wstride) * sizeof(int) <= kGenTablesCap ? (unsigned)base : 0u;
}
static unsigned pf_tables_off(int wstride, bool pre) {
  const size_t base = (pf_smem(wstride, pre) + 15) / 16 * 16;
  return base + bf_pf_slot_doubles(wstride) * sizeof(double) <= kGenTablesCap ? (unsigned)base : 0u;
}
static size_t mfe_smem_total(int wstride, bool pre) { const unsigned o = mfe_tables_off(wstride, pre); return o ? o + bf_mfe_slot_ints(wstride) * sizeof(int) : mfe_smem(wstride, pre); }
static size_t pf_smem_total(int wstride, bool pre) { const unsigned o = pf_tables_off(wstride, pre); return o ? o + bf_pf_slot_doubles(wstride) * sizeof(double) : pf_smem(wstride, pre); }
// the 48 KB a launch gets without opting in cover static + dynamic shared memory; the generic kernels hold 10-18 KB of static arrays
static const size_t kOptIn = 16 * 1024;
static size_t eval_smem(int stride) { return 2 * (stride + 4) * sizeof(short) + 2 * ((stride + 2 + 15) / 16 * 16); }

using MfeKernel = void (*)(const BfParams *, BfBatchDev, int *, size_t, int, int *, int *, char *, int, unsigned);
using PfKernel = void (*)(const BfParams *, BfBatchDev, double *, size_t, int, int *, const int *, double *, unsigned);
template <bool PRE>
static MfeKernel mfe_kernel_p(bool two, bool wide) {
  return two ? (wide ? bf_k_mfe<true, 16, PRE> : bf_k_mfe<true, BF_WARPS, PRE>) : (wide ? bf_k_mfe<false, 16, PRE> : bf_k_mfe<false, BF_WARPS, PRE>);
}
template <bool PRE>
static PfKernel pf_kernel_p(bool two, bool wide) {
  return two ? (wide ? bf_k_pf<true, 16, PRE> : bf_k_pf<true, BF_WARPS, PRE>) : (wide ? bf_k_pf<false, 16, PRE> : bf_k_pf<false, BF_WARPS, PRE>);
}
static MfeKernel mfe_kernel(bool two, bool wide, bool pre) { return pre ? mfe_kernel_p<true>(two, wide) : mfe_kernel_p<false>(two, wide); }
static PfKernel pf_kernel(bool two, bool wide, bool pre) { return pre ? pf_kernel_p<true>(two, wide) : pf_kernel_p<false>(two, wide); }

// CTAs per SM of the 8-warp build: what sizes the grid of a large batch (1 when the query fails)
template <typename K>
static int gen_occupancy(K kern, size_t sm) {
  int nb = 0;
  if (sm > kOptIn) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, BF_THREADS, sm) != cudaSuccess) return 1;
  return nb < 1 ? 1 : nb;
}

// key: two | wide << 1 | pre << 2.  A warp per cell: with few sequences (a CTA owns its SM) 16 warps per CTA halve the rounds per
// diagonal.  The grid keeps the per-CTA workspace within a sane share of HBM (48 GB MFE, 64 GB PF).
cudaError_t bf_gen_mfe_plan(int stride, int B, bool two, const BfOpts &o, int sms, BfPlan *p) {
  const int wstride = stride + 2;
  const bool wide = gen_wide(B, sms, o), pre = gen_pre(wstride, wide);
  p->family = BF_FAM_GENERIC;
  p->key = (two ? 1 : 0) | (wide ? 2 : 0) | (pre ? 4 : 0);
  p->smem = mfe_smem_total(wstride, pre);
  p->tables_off = mfe_tables_off(wstride, pre);
  p->ws = bf_mfe_slot_ints(wstride);
  p->grid = std::min(B, sms * gen_occupancy(mfe_kernel(two, false, false), mfe_smem_total(wstride, false)));
  while (p->grid > sms && (size_t)p->grid * p->ws * sizeof(int) > ((size_t)48 << 30)) p->grid -= sms;
  return cudaSuccess;
}

cudaError_t bf_gen_pf_plan(int stride, int B, bool two, const BfOpts &o, int sms, BfPlan *p) {
  const int wstride = stride + 2;
  const bool wide = gen_wide(B, sms, o), pre = gen_pre(wstride, wide);
  p->family = BF_FAM_GENERIC;
  p->key = (two ? 1 : 0) | (wide ? 2 : 0) | (pre ? 4 : 0);
  p->smem = pf_smem_total(wstride, pre);
  p->tables_off = pf_tables_off(wstride, pre);
  p->ws = bf_pf_slot_doubles(wstride);
  p->grid = std::min(B, sms * gen_occupancy(pf_kernel(two, false, false), pf_smem_total(wstride, false)));
  while (p->grid > sms && (size_t)p->grid * p->ws * sizeof(double) > ((size_t)64 << 30)) p->grid -= sms;
  return cudaSuccess;
}

cudaError_t bf_launch_mfe(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, int *ws, int *work_counter, int *out_mfe, char *out_ss,
                          int ss_stride, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  const bool wide = p.key & 2;
  auto kern = mfe_kernel(p.key & 1, wide, p.key & 4);
  if (p.smem > kOptIn) { e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem); if (e != cudaSuccess) return e; }
  kern<<<p.grid, (wide ? 16 : BF_WARPS) * 32, p.smem, st>>>(dP, b, ws, p.ws, b.stride + 2, work_counter, out_mfe, out_ss, ss_stride, p.tables_off);
  return cudaGetLastError();
}

cudaError_t bf_launch_pf(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, double *ws, int *work_counter, const int *mfe_for_scale,
                         double *out5, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  const bool wide = p.key & 2;
  auto kern = pf_kernel(p.key & 1, wide, p.key & 4);
  if (p.smem > kOptIn) { e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem); if (e != cudaSuccess) return e; }
  kern<<<p.grid, (wide ? 16 : BF_WARPS) * 32, p.smem, st>>>(dP, b, ws, p.ws, b.stride + 2, work_counter, mfe_for_scale, out5, p.tables_off);
  return cudaGetLastError();
}

cudaError_t bf_launch_eval(const BfParams *dP, const BfBatchDev &b, const char *targets, int n_targets, int tstride, int *out_e,
                           cudaStream_t st) {
  if (b.B * n_targets == 0) return cudaSuccess;
  size_t sm = eval_smem(b.stride);
  if (sm > kOptIn) { cudaError_t e = cudaFuncSetAttribute(bf_k_eval, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); if (e != cudaSuccess) return e; }
  bf_k_eval<<<b.B * n_targets, 128, sm, st>>>(dP, b, targets, n_targets, tstride, out_e);
  return cudaGetLastError();
}
