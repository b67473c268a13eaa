// bf_fill.cu -- diagonal-major wavefront kernels for single-strand folds (sm_100a).
//
// This is the throughput path behind score_sequence()'s fc.mfe() / fc.pf() calls
// (utils/energy_scores.py:150-151 in the reference; recurrences: SURVEY.md A.4-A.6).
//
// Layout.  Every O(N^2) table is stored by anti-diagonal: entry (i,j), d = j-i >= 4, lives at
// off(d) + i-1 with off(d) = sum_{x=4}^{d-1} (n-x).  With the 32 lanes of a warp running along
// a diagonal, every operand of every recurrence is a stride-1 access:
//   interior loops   c[p][q],  p = i+1+u1, q = j-1-u2  ->  diagonal d-2-(u1+u2), index i+1+u1
//   fML / qm splits  fml[i][u-1] + fml[u][j]            ->  diagonal k-1 index i, diagonal d-k index i+k
// so shared-memory reads are conflict-free and HBM reads/writes are coalesced.
//
// Interior loops look back at most 32 diagonals (u1+u2 <= 30), so only a 32-deep RING of the pair
// table is kept on chip.  The ring is stored three times with the inner pair's sequence-dependent
// term already folded in (generic: + mismatchI, 1xn: + mismatch1nI, bulge: + terminalAU), which
// turns every decomposable candidate into load + add-min (MFE) or load + fma (PF) against a
// warp-uniform length penalty.  The nine non-decomposable candidates (stack, bulge-1, 1x1, 1x2,
// 2x1, 2x2, 2x3, 3x2) are evaluated once per cell.
//
// The multiloop closing term of c(i,j) is the split part of fML(i+1,j-1), produced two diagonals
// earlier: it is kept in a 4-deep ring instead of being recomputed.
//
// One persistent CTA folds one sequence at a time.  Per diagonal: all warps accumulate partial
// minima / sums for (32-cell chunk, loop-size) work units, one barrier, one thread per cell
// combines them and writes the new diagonal, one barrier.  The exterior loop (f5 / q5) and the
// backtrack run afterwards in one-warp-per-sequence kernels on the tables written to HBM.
#include "bf_kernels.h"

#include <cstdlib>
#include <type_traits>

#include "bf_device.cuh"

namespace {

constexpr int kRing = 32;
constexpr int kInfThr = BF_INF / 2;

__device__ __forceinline__ size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// tile-major copy of a triangular table (blocked split): 4x4 tiles, tile (I,J) at tile_off(NT,I) + J-I, entry a*4+b
__host__ __device__ __forceinline__ int tile_off(int NT, int I) { return I * NT - I * (I - 1) / 2; }
__host__ __device__ __forceinline__ size_t tile_table_entries(int nmax) {
  const size_t nt = (nmax + 3) / 4;
  return nt * (nt + 1) / 2 * 16;
}

__device__ __forceinline__ int ptype_sp(const uint8_t *SP, int i, int j) { return bf_ptype_bases(SP[i], SP[j]); }

// ---------------------------------------------------------------------------------------------
// shared-memory plans (identical arithmetic on host and device)
// ---------------------------------------------------------------------------------------------
// placement flags of the MFE fill: where the tables that are re-read every diagonal live
constexpr int kMfeFmSmem = 1;   // packed fML table on chip (else: the per-sequence HBM copy, L2-resident while in use)
constexpr int kMfeRgSmem = 2;   // the three 32-deep pair rings on chip (else: per-CTA HBM workspace)

struct MfePlan {
  int rs;  // ring row stride (ints)
  size_t o_S, o_SP, o_toff, o_pg, o_pb, o_p1, o_fm, o_ring, o_dml, o_pi, o_ps, o_list, o_sa, o_f5, total;
};
__host__ __device__ inline MfePlan mfe_plan(int nmax, int nw, int pl, bool blk = false, bool atom = false) {
  MfePlan p;
  p.rs = (nmax + 8 + 3) / 4 * 4;
  size_t o = 0;
  p.o_S = o; o += (nmax + 2 + 15) / 16 * 16;
  p.o_SP = o; o += (nmax + 2 + 15) / 16 * 16;
  p.o_toff = o; o += (size_t)(nmax + 4) / 4 * 4 * sizeof(int);
  p.o_pg = o; o += 31 * 32 * sizeof(int);
  p.o_pb = o; o += 32 * sizeof(int);
  p.o_p1 = o; o += 32 * sizeof(int);
  p.o_fm = o; o += (pl & kMfeFmSmem) ? (tri_size(nmax) + 4) * sizeof(int) : 0;
  p.o_ring = o; o += (pl & kMfeRgSmem) ? (size_t)3 * kRing * p.rs * sizeof(int) : 0;
  p.o_dml = o; o += (size_t)4 * p.rs * sizeof(int);
  const int nbuf = atom ? 1 : nw;   // double-buffered partial minima: one buffer per warp, or one shared by all warps (atomicMin)
  p.o_pi = o; o += (size_t)2 * nbuf * p.rs * sizeof(int);
  p.o_ps = o; o += (size_t)2 * nbuf * p.rs * sizeof(int);
  p.o_list = o; o += (size_t)2 * p.rs * sizeof(unsigned short);  // pairable cells of a diagonal, double-buffered
  o = (o + 15) / 16 * 16;
  p.o_sa = o; o += blk ? (size_t)3 * ((nmax + 3) / 4) * 16 * sizeof(int) : 0;  // blocked-split minima of three tile-diagonals
  p.o_f5 = o; o += nw == 16 ? (size_t)(nmax + 8) * sizeof(int) : 0;   // exterior recursion inside the fill (16-warp variants)
  p.total = o;
  return p;
}

// Compact the pairable cells of diagonal d into list[0..count): one warp, ballot + popc prefix.
__device__ __forceinline__ int build_pair_list(const uint8_t *SP, int n, int d, unsigned short *list, int lane) {
  int count = 0;
  for (int base = 1; base <= n - d; base += 32) {
    const int i = base + lane;
    const bool ok = (i <= n - d) && bf_ptype_bases(SP[i], SP[i + d]) != 0;
    const unsigned mk = __ballot_sync(BF_FULL, ok);
    if (ok) list[count + __popc(mk & ((1u << lane) - 1))] = (unsigned short)i;
    count += __popc(mk);
  }
  return count;
}

// strided share of the loop sizes s = smax .. 2 with the long and the short ones alternating between warps
// (idx = 0 is s = smax; warp w takes idx = w, 2NW-1-w, 2NW+w, 4NW-1-w, ...)
#define BF_FOR_MY_S(NW, warp, smax, s)                                                          \
  for (int idx_ = (warp), flip_ = 0, s = (smax) - idx_; s >= 2;                                  \
       idx_ += flip_ ? 2 * (warp) + 1 : 2 * ((NW) - 1 - (warp)) + 1, flip_ ^= 1, s = (smax) - idx_)

// =====================================================================================================
//                                           MFE fill
// =====================================================================================================
// ctri / ftri: per-sequence tables in HBM (slot s at s * tri_slot), read later by bf_k_trace.
// Phase d of the diagonal loop: every warp first combines the partial minima of diagonal d-1 for the cells
// it owns (-> c, fML, ring rows of d-1), then accumulates partial minima for diagonal d.  The heavy part of
// diagonal d only reads diagonals <= d-2 (interior loops) and <= d-5 (fML splits), so one barrier per
// diagonal is enough; the partial buffers are double-buffered.
//
// BLK (blocked split): the bulk of  min_u fML[i][u-1] + fML[u][j]  is taken out of the per-diagonal loop.  fML is mirrored
// TILE-MAJOR (4x4 tiles) in the per-CTA workspace; for the tiles of tile-diagonal D' = J-I the products over the intermediate
// tiles K = I+3 .. J-3 only need diagonals <= 4D'-9, so they are computed as 4x4 register-tiled (min,+) block products
// (8 x 128-bit loads per 64 relaxations, lanes = 4 tiles x 8 K-slices) during the four phases d = 4D'-7 .. 4D'-4, one quarter
// of the tiles per phase, into SA[D' % 3].  The per-diagonal loop keeps only the <= 15 candidates next to either end.
// ATOM: the warps share one partial buffer per kind and merge with atomicMin (shared memory): smaller footprint, more CTAs per SM
// where the per-warp buffers were what limited occupancy (short sequences with the rings on chip, long sequences).
template <int NW, int PL, bool BLK = false, bool ATOM = false>
__global__ void __launch_bounds__(NW * 32) bf_k_mfe_fill(const BfParams *__restrict__ P, BfBatchDev b, int *ctri, int *ftri,
                                                         size_t tri_slot, int *ws, size_t ws_slot, int *work_counter, int *f5_out) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq, s_np[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  const MfePlan pl = mfe_plan(nmax, NW, PL, BLK, ATOM);
  constexpr int NBUF = ATOM ? 1 : NW;
  const int RS = pl.rs;
  uint8_t *S = dyn + pl.o_S;
  uint8_t *SP = dyn + pl.o_SP;
  int *toff = reinterpret_cast<int *>(dyn + pl.o_toff);
  int *SA = reinterpret_cast<int *>(dyn + pl.o_sa);
  const int NTS = (nmax + 3) / 4;  // tiles per side at the batch stride (SA row length)
  // tile-major fML mirror: last part of this CTA's workspace slot
  int *FMT = BLK ? ws + (size_t)blockIdx.x * ws_slot + (ws_slot - (tile_table_entries(nmax) + 7) / 8 * 8) : nullptr;
  int *pg = reinterpret_cast<int *>(dyn + pl.o_pg);   // [s][k], k = u1-2: interior[s] + ninio(|s-2u1|)
  int *pb = reinterpret_cast<int *>(dyn + pl.o_pb);   // bulge[s]
  int *p1 = reinterpret_cast<int *>(dyn + pl.o_p1);   // 1xn: interior[s] + ninio(s-2)
  int *fms = reinterpret_cast<int *>(dyn + pl.o_fm);
  int *ring = (PL & kMfeRgSmem) ? reinterpret_cast<int *>(dyn + pl.o_ring) : ws + (size_t)blockIdx.x * ws_slot;
  int *CG = ring, *C1 = ring + kRing * RS, *CB = ring + 2 * kRing * RS;
  int *DML = reinterpret_cast<int *>(dyn + pl.o_dml);
  int *PI = reinterpret_cast<int *>(dyn + pl.o_pi);
  int *PS = reinterpret_cast<int *>(dyn + pl.o_ps);
  unsigned short *LST = reinterpret_cast<unsigned short *>(dyn + pl.o_list);

  for (int k = tid; k < (int)(pl.total / 4); k += blockDim.x) reinterpret_cast<int *>(dyn)[k] = 0;
  __syncthreads();
  const BfSmallI &T = P->si;
  for (int k = tid; k < 31 * 32; k += blockDim.x) {
    const int s = k >> 5, u1 = (k & 31) + 2;
    int v = BF_INF;
    if (s >= 6 && u1 <= s - 2) v = T.interior[s] + min(T.ninio_max, abs(s - 2 * u1) * T.ninio_m);
    pg[k] = v;
  }
  if (tid < 32) {
    pb[tid] = (tid >= 2 && tid <= 30) ? T.bulge[tid] : BF_INF;
    p1[tid] = (tid >= 4 && tid <= 30) ? T.interior[tid] + min(T.ninio_max, (tid - 2) * T.ninio_m) : BF_INF;
  }
  for (int k = tid; k < 3 * kRing * RS; k += blockDim.x) ring[k] = BF_INF;
  if (ATOM) for (int k = tid; k < 2 * RS; k += blockDim.x) { PI[k] = BF_INF; PS[k] = BF_INF; }

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int sq = s_seq;
    if (sq >= b.B) break;
    const int n = b.len[sq];
    {
      const char *src = b.seq + (size_t)sq * b.stride;
      const uint8_t *np = b.nopair ? b.nopair + (size_t)sq * b.stride : nullptr;
      for (int k = tid; k <= n + 1; k += blockDim.x) {
        int code = (k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0;
        S[k] = (uint8_t)code;
        SP[k] = (uint8_t)((np && k >= 1 && k <= n && np[k - 1]) ? 0 : code);
      }
    }
    for (int k = tid; k <= n; k += blockDim.x) toff[k] = (k >= 4) ? tri_off(n, k) : 0;
    for (int k = tid; k < 4 * RS; k += blockDim.x) DML[k] = BF_INF;
    const int NT = (n + 3) >> 2;
    if (BLK) {
      for (int k = tid; k < (NT * (NT + 1) / 2) * 16; k += blockDim.x) FMT[k] = BF_INF;
      for (int k = tid; k < 3 * NTS * 16; k += blockDim.x) SA[k] = BF_INF;
    }
    int *cg_out = ctri + (size_t)sq * tri_slot;
    int *fg_out = ftri + (size_t)sq * tri_slot;
    int *FM = (PL & kMfeFmSmem) ? fms : fg_out;
    // 16-warp variants: the exterior recursion f5 (bf_k_trace) advances inside the fill, one column per phase on warp NW-2 --
    // f5[j] needs the diagonals up to j-1, complete and visible from phase j+1 on; bf_k_trace then only backtracks
    constexpr bool EXTF = (NW == 16);
    int *f5s = reinterpret_cast<int *>(dyn + pl.o_f5);
    int f5_next = 1;
    if (EXTF && f5_out && tid == (NW - 2) * 32) f5s[0] = 0;
    auto f5_step = [&](int j) {
      int e = BF_INF;
      for (int i = 1 + lane; i < j - BF_TURN; i += 32) {
        const int t = ptype_sp(SP, i, j);
        if (!t) continue;
        const int cc = cg_out[toff[j - i] + i - 1];
        if (cc >= BF_INF) continue;
        e = min(e, f5s[i - 1] + cc + bf_e_ext(T, t, i > 1 ? (int)S[i - 1] : -1, j < n ? (int)S[j + 1] : -1));
      }
      e = bf_warp_min(e);
      if (lane == 0) f5s[j] = min(e, f5s[j - 1]);
      __syncwarp();
    };
    __syncthreads();
    if (warp == 0 && n > BF_TURN + 1) {
      const int cnt = build_pair_list(SP, n, BF_TURN + 1, LST + ((BF_TURN + 1) & 1) * RS, lane);
      if (lane == 0) s_np[(BF_TURN + 1) & 1] = cnt;
    }
    __syncthreads();

    for (int d = BF_TURN + 1; d <= n; d++) {
      // ------------------------------------------------------------ pairable cells of the next diagonal
      if (warp == NW - 1 && d + 1 <= n - 1) {
        const int cnt = build_pair_list(SP, n, d + 1, LST + ((d + 1) & 1) * RS, lane);
        if (lane == 0) s_np[(d + 1) & 1] = cnt;
      }
      if (EXTF && f5_out && warp == NW - 2)
        while (f5_next <= d - 1) f5_step(f5_next++);
      // ------------------------------------------------------------ combine diagonal d-1
      if (d > BF_TURN + 1) {
        const int dd = d - 1, ncell = n - dd, buf = dd & 1;
        int *pi = PI + buf * NBUF * RS, *ps = PS + buf * NBUF * RS;
        for (int cell = tid; cell < ncell; cell += blockDim.x) {
          const int i = cell + 1, j = i + dd;
          const int t = ptype_sp(SP, i, j);
          int e = BF_INF, sp = BF_INF;
          if (ATOM) { sp = ps[cell]; ps[cell] = BF_INF; }   // the buffer is used again two phases later
          else {
#pragma unroll
            for (int w = 0; w < NW; w++) sp = min(sp, ps[w * RS + cell]);
          }
          if (t) {
            if (ATOM) { e = pi[cell]; pi[cell] = BF_INF; }
            else {
#pragma unroll
              for (int w = 0; w < NW; w++) e = min(e, pi[w * RS + cell]);
            }
            const int dm = DML[((dd - 2) & 3) * RS + i + 1];
            if (dm < kInfThr) e = min(e, dm + T.MLclosing + bf_e_mlstem(T, bf_rtype(t), S[j - 1], S[i + 1]));
            if (e >= kInfThr) e = BF_INF;
          }
          const int tI = (i - 1) >> 2, tJ = (j - 1) >> 2, tab = ((i - 1) & 3) * 4 + ((j - 1) & 3);
          if (BLK && tJ - tI >= 6) sp = min(sp, SA[((tJ - tI) % 3) * NTS * 16 + tI * 16 + tab]);
          if (sp >= kInfThr) sp = BF_INF;
          int m = sp;
          if (e < BF_INF && i > 1 && j < n) m = min(m, e + bf_e_mlstem(T, t, S[i - 1], S[j + 1]));
          if (dd > BF_TURN + 1) {
            const int o = toff[dd - 1] + i - 1;
            m = min(m, min(FM[o + 1], FM[o]) + T.MLbase);
          }
          if (m >= kInfThr) m = BF_INF;
          const int o = toff[dd] + i - 1;
          cg_out[o] = e;
          fg_out[o] = m;
          if (BLK) FMT[(size_t)(tile_off(NT, tI) + tJ - tI) * 16 + tab] = m;
          if (PL & kMfeFmSmem) fms[o] = m;
          DML[(dd & 3) * RS + i] = sp;
          const int row = (dd & (kRing - 1)) * RS + i;
          int eg = BF_INF, e1 = BF_INF, eb = BF_INF;
          if (e < BF_INF) {
            const int t2 = bf_rtype(t), a = S[j + 1], bb = S[i - 1];  // as an inner pair: sq1 = S[q+1], sp1 = S[p-1]
            eg = e + T.mmI[t2][a][bb];
            e1 = e + T.mm1nI[t2][a][bb];
            eb = e + (t > 2 ? T.TerminalAU : 0);
          }
          CG[row] = eg; C1[row] = e1; CB[row] = eb;
        }
      }
      // ------------------------------------------------------------ partial minima of diagonal d
      if (d <= n - 1) {
        const int ncell = n - d, buf = d & 1;
        int *pi = PI + (buf * NBUF + (ATOM ? 0 : warp)) * RS, *ps = PS + (buf * NBUF + (ATOM ? 0 : warp)) * RS;
        const int smax = min(BF_MAXLOOP, d - 6);  // inner diagonal d-2-s >= 4
        // ---- pair-only work on the compacted list: interior loops, hairpin
        const int np = s_np[buf];
        const unsigned short *list = LST + buf * RS;
        for (int c = 0; c < np; c += 32) {
          const int kk = c + lane;
          const int i = list[min(kk, np - 1)];      // idle lanes repeat the last pairable cell and are dropped at the store
          const int j = i + d;
          const int t = ptype_sp(SP, i, j);
          const int si1 = S[i + 1], sj1 = S[j - 1];
          int accg = BF_INF, acc1 = BF_INF, accb = BF_INF;
          constexpr bool kBatchR2 = (NW >= 8 && PL == 0 && BLK);  // long-sequence configuration: every ring is read through L2
          if (kBatchR2) {
            // bulge and 1xn candidates of this warp's (at most four) loop sizes: all sixteen loads first
            int sv[4], ns = 0;
            BF_FOR_MY_S(NW, warp, smax, s) { if (ns < 4) sv[ns] = s; ns++; }
            int b0[4], b1[4], o0[4], o1[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
              const int s = u < ns ? sv[u] : 2;
              const int row = ((d - 2 - s) & (kRing - 1)) * RS + i;
              b0[u] = CB[row + 1]; b1[u] = CB[row + 1 + s];
              o0[u] = C1[row + 2]; o1[u] = C1[row + s];
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
              if (u < ns) {
                accb = min(accb, min(b0[u], b1[u]) + pb[sv[u]]);
                if (sv[u] >= 4) acc1 = min(acc1, min(o0[u], o1[u]) + p1[sv[u]]);
              }
            }
          }
          BF_FOR_MY_S(NW, warp, smax, s) {
            const int row = ((d - 2 - s) & (kRing - 1)) * RS + i;
            if (!kBatchR2) {
              accb = min(accb, min(CB[row + 1], CB[row + 1 + s]) + pb[s]);
              if (s >= 4) acc1 = min(acc1, min(C1[row + 2], C1[row + s]) + p1[s]);
            }
            if (s >= 6) {
              const int *cgp = CG + row + 3;
              const int *pen = pg + (s << 5);
              const int kn = s - 3;
              if (PL & kMfeRgSmem) {
#pragma unroll 4
                for (int k = 0; k < kn; k++) accg = min(accg, cgp[k] + pen[k]);
              } else {  // ring rows come from L2: keep more loads in flight
#pragma unroll 8
                for (int k = 0; k < kn; k++) accg = min(accg, cgp[k] + pen[k]);
              }
            }
          }
          int tot = min(accg + T.mmI[t][si1][sj1], min(acc1 + T.mm1nI[t][si1][sj1], accb + (t > 2 ? T.TerminalAU : 0)));
          // the hairpin and the nine non-decomposable interior candidates, dealt round-robin to the warps
          for (int k = (warp + c + d) % NW; k < 10; k += NW) {
            if (k == 9) { tot = min(tot, bf_e_hairpin(P, T, S, i, j, t)); continue; }
            const int u1 = (0x322211100ull >> (4 * k)) & 15, u2 = (0x232121010ull >> (4 * k)) & 15;
            const int p = i + 1 + u1, q = j - 1 - u2;
            if (q - p <= BF_TURN) continue;
            int cc = CB[((q - p) & (kRing - 1)) * RS + p];  // c + terminalAU(inner pair)
            if (cc >= kInfThr) continue;
            const int t2 = ptype_sp(SP, p, q);
            if (t2 > 2) cc -= T.TerminalAU;
            tot = min(tot, cc + bf_e_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1]));
          }
          if (kk < np) { if (ATOM) { if (tot < kInfThr) atomicMin(&pi[i - 1], tot); } else pi[i - 1] = tot; }
        }
        // ---- fML split for every cell: k = u - i in [5, d-4]
        if (!BLK) {
        for (int c = 0; c < ncell; c += 32) {
          const int cell = c + lane;
          const int i = min(cell, ncell - 1) + 1;
          int accs = BF_INF;
          const int *left = FM + (i - 1);
          // operands come from L2 unless the table is on chip: deep unrolling keeps many loads in flight on long diagonals
          if (d - 8 >= 16 * NW) {
#pragma unroll 8
            for (int k = 5 + warp; k <= d - 4; k += NW) accs = min(accs, left[toff[k - 1]] + left[toff[d - k] + k]);
          } else {
#pragma unroll 4
            for (int k = 5 + warp; k <= d - 4; k += NW) accs = min(accs, left[toff[k - 1]] + left[toff[d - k] + k]);
          }
          if (cell < ncell) { if (ATOM) { if (accs < kInfThr) atomicMin(&ps[cell], accs); } else ps[cell] = accs; }
        }
        } else {
        // blocked split: only the candidates next to either end stay here -- k in [5, 12] and [d-10, d-4] minus what the
        // block products of tiles K = I+3 .. J-3 cover (left column x+k-1 inside those tiles).  Four chunks of 32 cells are
        // handled together so that eight operand pairs are in flight per thread.
        for (int c = 0; c < ncell; c += 128) {
          int xs[4], klo[4], khi[4], accs[4];
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const int x = min(c + 32 * u + lane, ncell - 1);
            const int tI = x >> 2, tJ = (x + d) >> 2;
            xs[u] = x;
            klo[u] = (tJ - tI >= 6) ? 4 * (tI + 3) - x + 1 : 1 << 30;  // covered k range
            khi[u] = 4 * (tJ - 3) + 3 - x + 1;
            accs[u] = BF_INF;
          }
          for (int slot = warp; slot < 15; slot += NW) {
            const int k = slot < 8 ? 5 + slot : d - 18 + slot;  // 5..12, d-10..d-4
            if (k < 5 || k > d - 4 || (slot >= 8 && k <= 12)) continue;  // warp-uniform
            const int o1 = toff[k - 1], o2 = toff[d - k] + k;
            int va[4], vb[4];
#pragma unroll
            for (int u = 0; u < 4; u++) { va[u] = FM[xs[u] + o1]; vb[u] = FM[xs[u] + o2]; }
#pragma unroll
            for (int u = 0; u < 4; u++)
              if (k < klo[u] || k > khi[u]) accs[u] = min(accs[u], va[u] + vb[u]);
          }
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const int cell = c + 32 * u + lane;
            if (cell < ncell) { if (ATOM) { if (accs[u] < kInfThr) atomicMin(&ps[cell], accs[u]); } else ps[cell] = accs[u]; }
          }
        }
        // block products for tile-diagonal D' = (d+7)/4, quarter q = (d+7)%4 of its tiles
        {
          const int Dp = (d + 7) >> 2, q = (d + 7) & 3;
          if (Dp >= 6 && Dp < NT) {
            const int Tn = NT - Dp;
            int *dst = SA + (Dp % 3) * NTS * 16;
            for (int g = warp; q + 16 * g < Tn; g += NW) {
              const int I = q + 4 * (4 * g + (lane >> 3)), J = I + Dp, sl = lane & 7;
              int acc[16];
#pragma unroll
              for (int k = 0; k < 16; k++) acc[k] = BF_INF;
              if (I < Tn) {
                const int *rowI = FMT + (size_t)tile_off(NT, I) * 16;
                for (int K = I + 3 + sl; K <= J - 3; K += 8) {
                  const int4 *lp = reinterpret_cast<const int4 *>(rowI + (K - I) * 16);
                  const int4 *rp = reinterpret_cast<const int4 *>(FMT + (size_t)(tile_off(NT, K) + J - K) * 16);
                  const int4 *rq = reinterpret_cast<const int4 *>(FMT + (size_t)(tile_off(NT, K + 1) + J - K - 1) * 16);
                  const int4 r0 = rp[1], r1 = rp[2], r2 = rp[3], r3 = rq[0];  // rows u = 4K+c+1, c = 0..3 (0-based)
#pragma unroll
                  for (int a = 0; a < 4; a++) {
                    const int4 l = lp[a];  // fML[4I+a][4K+c], c = 0..3
                    acc[a * 4 + 0] = min(acc[a * 4 + 0], min(min(l.x + r0.x, l.y + r1.x), min(l.z + r2.x, l.w + r3.x)));
                    acc[a * 4 + 1] = min(acc[a * 4 + 1], min(min(l.x + r0.y, l.y + r1.y), min(l.z + r2.y, l.w + r3.y)));
                    acc[a * 4 + 2] = min(acc[a * 4 + 2], min(min(l.x + r0.z, l.y + r1.z), min(l.z + r2.z, l.w + r3.z)));
                    acc[a * 4 + 3] = min(acc[a * 4 + 3], min(min(l.x + r0.w, l.y + r1.w), min(l.z + r2.w, l.w + r3.w)));
                  }
                }
              }
#pragma unroll
              for (int o = 4; o > 0; o >>= 1) {
#pragma unroll
                for (int k = 0; k < 16; k++) acc[k] = min(acc[k], __shfl_xor_sync(BF_FULL, acc[k], o));
              }
              if (I < Tn && sl == 0) {
                int4 *d4 = reinterpret_cast<int4 *>(dst + I * 16);
                d4[0] = make_int4(acc[0], acc[1], acc[2], acc[3]);
                d4[1] = make_int4(acc[4], acc[5], acc[6], acc[7]);
                d4[2] = make_int4(acc[8], acc[9], acc[10], acc[11]);
                d4[3] = make_int4(acc[12], acc[13], acc[14], acc[15]);
              }
            }
          }
        }
        }
      }
      __syncthreads();
    }
    if (EXTF && f5_out && warp == NW - 2) {
      while (f5_next <= n) f5_step(f5_next++);
      for (int k = lane; k <= n; k += 32) f5_out[(size_t)sq * (nmax + 4) + k] = f5s[k];
    }
  }
}

// =====================================================================================================
//                    exterior loop + backtrack: one warp per sequence, tables in HBM
// =====================================================================================================
struct __align__(8) Sector { short i, j; int kind; };  // 0 exterior (f5 up to j), 1 multiloop part, 2 pair

template <int WPB>
__global__ void __launch_bounds__(WPB * 32) bf_k_trace(const BfParams *__restrict__ P, BfBatchDev b, const int *__restrict__ ctri,
                                                       const int *__restrict__ ftri, size_t tri_slot, int *out_mfe, char *out_ss,
                                                       int ss_stride, const int *__restrict__ f5_in) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallI T;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  bf_stage(&T, &P->si);
  __syncthreads();
  const int sq = blockIdx.x * WPB + warp;
  if (sq >= b.B) return;
  // per-warp carve-up
  const size_t per_warp = align_up(2 * align_up(nmax + 2, 16) + (nmax + 4) * sizeof(int) + (2 * nmax + 16) * sizeof(Sector), 16);
  unsigned char *base = dyn + per_warp * warp;
  uint8_t *S = base;
  uint8_t *SP = S + align_up(nmax + 2, 16);
  int *f5 = reinterpret_cast<int *>(SP + align_up(nmax + 2, 16));
  Sector *stk = reinterpret_cast<Sector *>(f5 + (nmax + 4));
  const int n = b.len[sq];
  {
    const char *src = b.seq + (size_t)sq * b.stride;
    const uint8_t *np = b.nopair ? b.nopair + (size_t)sq * b.stride : nullptr;
    for (int k = lane; k <= n + 1; k += 32) {
      int code = (k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0;
      S[k] = (uint8_t)code;
      SP[k] = (uint8_t)((np && k >= 1 && k <= n && np[k - 1]) ? 0 : code);
    }
  }
  __syncwarp();
  const int *c = ctri + (size_t)sq * tri_slot;
  const int *fm = ftri + (size_t)sq * tri_slot;
  auto C_ = [&](int i, int j) -> int { return (j - i > BF_TURN) ? __ldg(c + tri_off(n, j - i) + i - 1) : BF_INF; };
  auto M_ = [&](int i, int j) -> int { return (j - i > BF_TURN) ? __ldg(fm + tri_off(n, j - i) + i - 1) : BF_INF; };
  auto ext_e = [&](int i, int j, int t) -> int {
    const int a = (i > 1) ? S[i - 1] : -1, bb = (j < n) ? S[j + 1] : -1;
    return bf_e_ext(T, t, a, bb);
  };

  if (lane == 0) f5[0] = 0;
  __syncwarp();
  // f5[j] = min(f5[j-1], min_i f5[i-1] + c(i,j) + Ext(i,j)): a serial chain over j whose table look-ups do not depend on f5.
  // The table entries of column j+PD are fetched while column j is reduced (PD columns of look-ups in flight: one column's
  // reduction is far shorter than a table load that misses in L2), the exterior terms are added when the column is reduced;
  // K = 32-wide chunks of i per lane.
  auto chain = [&](auto kc) {
    constexpr int K = decltype(kc)::value, PD = 16 / K;
    int cc[PD][K];
    auto fetch = [&](int j, int *v) {
#pragma unroll
      for (int c = 0; c < K; c++) {
        const int i = 1 + lane + 32 * c;
        v[c] = (j <= n && i < j - BF_TURN && ptype_sp(SP, i, j)) ? C_(i, j) : BF_INF;
      }
    };
#pragma unroll
    for (int p = 0; p < PD; p++) fetch(1 + p, cc[p]);
    for (int j0 = 1; j0 <= n; j0 += PD) {
#pragma unroll
      for (int p = 0; p < PD; p++) {
        const int j = j0 + p;
        if (j > n) break;
        int e = BF_INF;
#pragma unroll
        for (int c = 0; c < K; c++) {
          const int i = 1 + lane + 32 * c;
          if (cc[p][c] < BF_INF) {   // set only for i < j - TURN with a pair type
            const int v = cc[p][c] + ext_e(i, j, ptype_sp(SP, i, j));
            if (v < BF_INF) e = min(e, f5[i - 1] + v);
          }
        }
        fetch(j + PD, cc[p]);
        e = bf_warp_min(e);
        if (lane == 0) f5[j] = min(e, f5[j - 1]);
        __syncwarp();
      }
    }
  };
  if (f5_in) {   // the 16-warp fill already ran the recursion
    for (int k = lane; k <= n; k += 32) f5[k] = __ldg(f5_in + (size_t)sq * (nmax + 4) + k);
    __syncwarp();
  }
  else if (n <= 64) chain(std::integral_constant<int, 2>());
  else if (n <= 128) chain(std::integral_constant<int, 4>());
  else if (n <= 256) chain(std::integral_constant<int, 8>());
  else
  for (int j = 1; j <= n; j++) {
    int e = BF_INF;
    for (int i = 1 + lane; i < j - BF_TURN; i += 32) {
      const int t = ptype_sp(SP, i, j);
      if (!t) continue;
      const int cc = C_(i, j);
      if (cc >= BF_INF) continue;
      e = min(e, f5[i - 1] + cc + ext_e(i, j, t));
    }
    e = bf_warp_min(e);
    if (lane == 0) f5[j] = min(e, f5[j - 1]);
    __syncwarp();
  }
  if (lane == 0 && out_mfe) out_mfe[sq] = f5[n];
  if (!out_ss) return;
  char *ss = out_ss + (size_t)sq * ss_stride;
  for (int k = lane; k < ss_stride; k += 32) ss[k] = (k < n) ? '.' : 0;
  __syncwarp();

  // backtrack: same order of choices as the fill-independent rule of SURVEY.md A.5
  int sp = 0;
  if (lane == 0) { stk[0].i = 1; stk[0].j = (short)n; stk[0].kind = 0; }
  sp = 1;
  __syncwarp();
  int guard = 0;
  while (sp > 0 && guard++ < 8 * n + 64) {
    Sector sec = stk[--sp];
    __syncwarp();
    int i = sec.i, j = sec.j;
    bool to_pair = false;
    if (sec.kind == 0) {
      while (j > 0 && f5[j] == f5[j - 1]) j--;
      if (j <= 1) continue;
      int fu = 0;
      for (int bs = j - 1; bs >= 1 && !fu; bs -= 32) {
        const int u = bs - lane;
        bool ok = false;
        if (u >= 1) {
          const int t = ptype_sp(SP, u, j);
          if (t) {
            const int cc = C_(u, j);
            if (cc < BF_INF) ok = f5[j] == f5[u - 1] + cc + ext_e(u, j, t);
          }
        }
        const unsigned mk = __ballot_sync(BF_FULL, ok);
        if (mk) fu = bs - (__ffs(mk) - 1);
      }
      if (!fu) break;
      if (lane == 0) { stk[sp].i = 1; stk[sp].j = (short)(fu - 1); stk[sp].kind = 0; }
      sp++;
      __syncwarp();
      i = fu; to_pair = true;
    } else if (sec.kind == 1) {
      // unpaired ends of the multiloop part: `while (M(i,j) == M(i,j-1) + MLbase) j--`, then the same from the left -- 32 positions
      // per table round trip instead of one (the run of positions that satisfy the test, counted from the current end)
      for (;;) {
        const int jj = j - lane;
        const bool ok = jj > i && M_(i, jj) == M_(i, jj - 1) + T.MLbase;
        const unsigned mk = __ballot_sync(BF_FULL, ok);
        if (mk == BF_FULL) { j -= 32; continue; }
        j -= __ffs(~mk) - 1;
        break;
      }
      for (;;) {
        const int ii = i + lane;
        const bool ok = ii < j && M_(ii, j) == M_(ii + 1, j) + T.MLbase;
        const unsigned mk = __ballot_sync(BF_FULL, ok);
        if (mk == BF_FULL) { i += 32; continue; }
        i += __ffs(~mk) - 1;
        break;
      }
      const int mij = M_(i, j);
      const int t = ptype_sp(SP, i, j);
      const int cij = C_(i, j);
      if (t && cij < BF_INF && i > 1 && j < n && mij == cij + bf_e_mlstem(T, t, S[i - 1], S[j + 1])) {
        to_pair = true;
      } else {
        int fu = 0;
        for (int bs = i + 1; bs <= j && !fu; bs += 32) {
          const int u = bs + lane;
          bool ok = false;
          if (u <= j) {
            const int l = M_(i, u - 1), r = M_(u, j);
            ok = l < BF_INF && r < BF_INF && mij == l + r;
          }
          const unsigned mk = __ballot_sync(BF_FULL, ok);
          if (mk) fu = bs + (__ffs(mk) - 1);
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
      to_pair = true;
    }
    if (!to_pair) continue;
    for (;;) {
      if (lane == 0) { ss[i - 1] = '('; ss[j - 1] = ')'; }
      {
        // a helix in one table round trip: lane k asks whether pair (i+k, j-k) -- a pair of the structure if all lanes before it say
        // yes -- continues with the stacked pair (i+k+1, j-k-1).  That is the walk's own first choice for a pair that is not an
        // optimal hairpin closing (hairpin test first, then inner pairs by p ascending, q descending: the stack comes first)
        const int ik = i + lane, jk = j - lane;
        bool stacked = false;
        if (jk - ik > 2) {
          const int tk = ptype_sp(SP, ik, jk), t2 = ptype_sp(SP, ik + 1, jk - 1);
          if (tk && t2) {
            const int ck = C_(ik, jk), cc = C_(ik + 1, jk - 1);
            stacked = ck < BF_INF && cc < BF_INF && ck == cc + bf_e_intloop(P, T, 0, 0, tk, bf_rtype(t2), S[ik + 1], S[jk - 1], S[ik], S[jk]) &&
                      ck != bf_e_hairpin(P, T, S, ik, jk, tk);
          }
        }
        const unsigned mk = __ballot_sync(BF_FULL, stacked);
        const int run = mk == BF_FULL ? 32 : __ffs(~mk) - 1;
        if (run > 0) {
          if (lane < run) { ss[ik - 1] = '('; ss[jk - 1] = ')'; }
          __syncwarp();
          i += run; j -= run;
          continue;
        }
      }
      const int t = ptype_sp(SP, i, j), cij = C_(i, j);
      const int si1 = S[i + 1], sj1 = S[j - 1];
      if (cij == bf_e_hairpin(P, T, S, i, j, t)) break;
      int fp = 0, fq = 0;
      const int pmax = min(j - 2, i + BF_MAXLOOP + 1);
      // inner pairs in the order p ascending, q descending (lanes = q).  The first row alone (a stacked pair or a bulge on the 3' side:
      // most steps end here), the others four rows per round so that their table reads are in flight together -- a pair that closes a
      // multiloop walks all 31 rows before the split is tried
      {
        const int p = i + 1, q = j - 1 - lane;
        bool ok = false;
        if (p <= pmax && q >= max(p + 1, j - i + p - BF_MAXLOOP - 2)) {
          const int t2 = ptype_sp(SP, p, q);
          if (t2) {
            const int cc = C_(p, q);
            ok = cc < BF_INF && cij == cc + bf_e_intloop(P, T, 0, j - q - 1, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1]);
          }
        }
        const unsigned mk = __ballot_sync(BF_FULL, ok);
        if (mk) { fp = p; fq = j - 1 - (__ffs(mk) - 1); }
      }
      for (int p0 = i + 2; p0 <= pmax && !fp; p0 += 4) {
        const int q = j - 1 - lane;
        int cc[4], t2[4];
#pragma unroll
        for (int r = 0; r < 4; r++) {
          const int p = p0 + r;
          const bool in = p <= pmax && q >= max(p + 1, j - i + p - BF_MAXLOOP - 2);
          t2[r] = in ? ptype_sp(SP, p, q) : 0;
          cc[r] = t2[r] ? C_(p, q) : BF_INF;
        }
#pragma unroll
        for (int r = 0; r < 4; r++) {
          const int p = p0 + r;
          const bool ok = cc[r] < BF_INF && cij == cc[r] + bf_e_intloop(P, T, p - i - 1, j - q - 1, t, bf_rtype(t2[r]), si1, sj1, S[p - 1], S[q + 1]);
          const unsigned mk = __ballot_sync(BF_FULL, ok);
          if (mk && !fp) { fp = p; fq = j - 1 - (__ffs(mk) - 1); }
        }
      }
      if (fp) { i = fp; j = fq; continue; }
      int fu = 0;
      const int en = cij - T.MLclosing - bf_e_mlstem(T, bf_rtype(t), sj1, si1);
      for (int bs = i + 2; bs <= j - 1 && !fu; bs += 32) {
        const int u = bs + lane;
        bool ok = false;
        if (u <= j - 1) {
          const int l = M_(i + 1, u - 1), r = M_(u, j - 1);
          ok = l < BF_INF && r < BF_INF && en == l + r;
        }
        const unsigned mk = __ballot_sync(BF_FULL, ok);
        if (mk) fu = bs + (__ffs(mk) - 1);
      }
      if (fu) {
        if (lane == 0) {
          stk[sp].i = (short)(i + 1); stk[sp].j = (short)(fu - 1); stk[sp].kind = 1;
          stk[sp + 1].i = (short)fu; stk[sp + 1].j = (short)(j - 1); stk[sp + 1].kind = 1;
        }
        sp += 2;
        __syncwarp();
      }
      break;
    }
  }
}

// =====================================================================================================
//                                   partition function (inside) fill
// =====================================================================================================
constexpr int kPfQmSmem = 1;   // packed qm and qm1 tables on chip (else: per-CTA HBM workspace)
constexpr int kPfQgSmem = 4;   // the generic-interior ring on chip (the 1xn and bulge rings are always in the workspace)

struct PfPlan {
  int rs;
  size_t o_S, o_toff, o_wg, o_wb, o_w1, o_scl, o_bu, o_qm, o_qm1, o_qg, o_qms, o_au, o_pi, o_ps, o_list, o_q5, total;
};
__host__ __device__ inline PfPlan pf_plan(int nmax, int nw, int pl, bool half = false) {
  PfPlan p;
  p.rs = (nmax + 8 + 3) / 4 * 4;
  size_t o = 0;
  p.o_wg = o; o += 31 * 32 * sizeof(double);
  p.o_wb = o; o += 32 * sizeof(double);
  p.o_w1 = o; o += 32 * sizeof(double);
  p.o_scl = o; o += (size_t)(nmax + 8) * sizeof(double);
  p.o_bu = o; o += (size_t)(nmax + 8) * sizeof(double);
  p.o_qm = o; o += (pl & kPfQmSmem) ? (tri_size(nmax) + 4) * sizeof(double) : 0;
  p.o_qm1 = o; o += (pl & kPfQmSmem) ? (tri_size(nmax) + 4) * sizeof(double) : 0;
  p.o_qg = o; o += (pl & kPfQgSmem) ? (size_t)kRing * p.rs * sizeof(double) : 0;
  p.o_qms = o; o += (size_t)4 * p.rs * sizeof(double);
  p.o_au = o; o += (size_t)2 * p.rs * sizeof(double);
  const int nb = half ? nw / 2 : nw;  // per-warp partial buffers; half: two warps share one (see bf_k_pf_fill)
  p.o_pi = o; o += (size_t)2 * nb * p.rs * sizeof(double);
  p.o_ps = o; o += (size_t)2 * nb * p.rs * sizeof(double);
  p.o_list = o; o += (size_t)2 * p.rs * sizeof(unsigned short);
  p.o_toff = o; o += (size_t)(nmax + 4) / 4 * 4 * sizeof(int);
  p.o_S = o; o += (nmax + 2 + 15) / 16 * 16;
  p.o_q5 = o; o += nw == 16 ? (size_t)(nmax + 8) * sizeof(double) : 0;   // exterior recursion inside the fill (16-warp variants)
  p.total = o;
  return p;
}
// doubles of per-CTA HBM workspace for the tables that are not on chip
__host__ __device__ inline size_t pf_ws_doubles(int nmax, int pl) {
  const size_t rs = (nmax + 8 + 3) / 4 * 4;
  size_t o = 2 * kRing * rs;
  if (!(pl & kPfQmSmem)) o += 2 * ((tri_size(nmax) + 7) / 8 * 8);
  if (!(pl & kPfQgSmem)) o += kRing * rs;
  return (o + 7) / 8 * 8;
}

// named barrier of a warp pair (ids 1..8; id 0 is __syncthreads)
__device__ __forceinline__ void pair_barrier(int k) {
  asm volatile("bar.sync %0, 64;" ::"r"(k + 1) : "memory");
}

// qbtri: per-sequence qb table in HBM (for the exterior pass).  Same phase structure as bf_k_mfe_fill.
// qm(i,j) = qm1(i,j) + A(i,j) + sum_k qm[i][i+k-1] qm1[i+k][j] with A(i,j) = sum_{k>=1} bu^k qm1(i+k,j)
//         = bu (qm1(i+1,j) + A(i+1,j)): the unpaired-prefix part is carried along the diagonals in O(1) per cell.
// HALF: warps w and w + NW/2 share one partial buffer.  The first of the pair does the interior part, then the split part; the
// second does them in the opposite order; between the two halves the pair meets at a named barrier, after which each ADDS onto
// what the other stored.  Halves the reduction buffers (two CTAs per SM at L = 400) at the cost of one 64-thread barrier.
// BLK: blocked split as in bf_k_mfe_fill.  qm and qm1 are mirrored tile-major in the workspace; the products over tiles
// K = I+3 .. J-3 of tile-diagonal D' are accumulated during phases d = 4D'-7 .. 4D'-4 (lanes = 4 tiles x 4 K-slices x 2 column
// halves, 12 x 128-bit loads per 32 DFMA and 4 B of operand traffic per relaxation instead of 16) into SA[D' % 3] (workspace).
// MINB: CTAs per SM the build is capped for (__launch_bounds__; 0 = the compiler's choice).  The compiler takes 128 registers when
// it may; 80 (3 CTAs) or 64 (4 CTAs) cost a few bytes of spill and buy occupancy where shared memory and L2 capacity allow it.
template <int NW, int PL, bool HALF = false, bool BLK = false, int MINB = 0>
__global__ void __launch_bounds__(NW * 32, MINB) bf_k_pf_fill(const BfParams *__restrict__ P, BfBatchDev b, double *qbtri, size_t tri_slot,
                                                        double *ws, size_t ws_slot, double *qm_perseq, const int *mfe_for_scale,
                                                        double *lnscale_out, int *work_counter, double *out5) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq, s_np[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  constexpr int NB = HALF ? NW / 2 : NW;
  const PfPlan pl = pf_plan(nmax, NW, PL, HALF);
  const int RS = pl.rs;
  uint8_t *S = dyn + pl.o_S;
  int *toff = reinterpret_cast<int *>(dyn + pl.o_toff);
  double *wg = reinterpret_cast<double *>(dyn + pl.o_wg);
  double *wb = reinterpret_cast<double *>(dyn + pl.o_wb);
  double *w1 = reinterpret_cast<double *>(dyn + pl.o_w1);
  double *scl = reinterpret_cast<double *>(dyn + pl.o_scl);
  double *bu = reinterpret_cast<double *>(dyn + pl.o_bu);
  double *QMS = reinterpret_cast<double *>(dyn + pl.o_qms);
  double *AU = reinterpret_cast<double *>(dyn + pl.o_au);
  double *PI = reinterpret_cast<double *>(dyn + pl.o_pi);
  double *PS = reinterpret_cast<double *>(dyn + pl.o_ps);
  unsigned short *LST = reinterpret_cast<unsigned short *>(dyn + pl.o_list);
  double *wsp = ws + (size_t)blockIdx.x * ws_slot;
  double *QM, *QM1, *QG, *Q1, *QBB;
  if (PL & kPfQmSmem) {
    QM = reinterpret_cast<double *>(dyn + pl.o_qm);
    QM1 = reinterpret_cast<double *>(dyn + pl.o_qm1);
  } else {
    QM = wsp; QM1 = wsp + (tri_size(nmax) + 7) / 8 * 8; wsp += 2 * ((tri_size(nmax) + 7) / 8 * 8);
  }
  if (PL & kPfQgSmem) QG = reinterpret_cast<double *>(dyn + pl.o_qg);
  else { QG = wsp; wsp += kRing * RS; }
  Q1 = wsp; QBB = wsp + kRing * RS;
  // blocked split: tile-major mirrors of qm / qm1 and the block-product sums of three tile-diagonals, at the end of the slot
  const int NTS = (nmax + 3) / 4;
  const size_t tt = (tile_table_entries(nmax) + 7) / 8 * 8;
  double *QMT = BLK ? ws + (size_t)blockIdx.x * ws_slot + (ws_slot - (2 * tt + (size_t)3 * NTS * 16)) : nullptr;
  double *QM1T = BLK ? QMT + tt : nullptr;
  double *SA = BLK ? QM1T + tt : nullptr;

  for (int k = tid; k < (int)(pl.total / 4); k += blockDim.x) reinterpret_cast<int *>(dyn)[k] = 0;
  __syncthreads();
  const BfSmallD &T = P->sd;
  for (int k = tid; k < kRing * RS; k += blockDim.x) { QG[k] = 0.0; Q1[k] = 0.0; QBB[k] = 0.0; }

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int sq = s_seq;
    if (sq >= b.B) break;
    const int n = b.len[sq];
    {
      const char *src = b.seq + (size_t)sq * b.stride;
      for (int k = tid; k <= n + 1; k += blockDim.x) S[k] = (uint8_t)((k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0);
    }
    for (int k = tid; k <= n; k += blockDim.x) toff[k] = (k >= 4) ? tri_off(n, k) : 0;
    // per-nucleotide scale (ViennaRNA exp_params_rescale, sfact 1.07; default estimate -185 cal/mol/nt)
    double lns = 185.0 / T.kT;
    if (mfe_for_scale && n > 0) {
      const double m = (double)mfe_for_scale[sq] * 10.0;
      if (m < 0.0) lns = -1.07 * m / T.kT / (double)n;
      if (lns < 185.0 / T.kT * 0.25) lns = 185.0 / T.kT * 0.25;
    }
    {
      const double bl = log(T.x_MLbase) - lns;
      for (int k = tid; k <= n + 2; k += blockDim.x) { scl[k] = exp(-lns * k); bu[k] = exp(bl * k); }
    }
    if (tid == 0 && lnscale_out) lnscale_out[sq] = lns;
    // 16-warp variants (a CTA owns its SM, latency is what counts): the exterior recursion q5 (bf_k_pf_ext) advances inside the
    // fill, one column per phase on warp NW-2 -- q5[j] needs the diagonals up to j-1, complete and visible from phase j+1 on
    constexpr bool EXTQ = (NW == 16);
    double *q5s = reinterpret_cast<double *>(dyn + pl.o_q5);
    const double *qb_out_ext = qbtri + (size_t)sq * tri_slot;
    if (EXTQ && out5 && tid == (NW - 2) * 32) q5s[0] = 1.0;
    const double sc1 = exp(-lns);
    int q5_next = 1;
    auto q5_step = [&](int j) {
      double sum = 0.0;
      for (int i = 1 + lane; i < j - BF_TURN; i += 32) {
        const int t = bf_ptype_bases(S[i], S[j]);
        if (!t) continue;
        const int a = (i > 1) ? S[i - 1] : -1, bb = (j < n) ? S[j + 1] : -1;
        sum += q5s[i - 1] * qb_out_ext[toff[j - i] + i - 1] * bf_x_ext(T, t, a, bb);
      }
      sum = bf_warp_sum(sum);
      if (lane == 0) q5s[j] = sum + q5s[j - 1] * sc1;
      __syncwarp();
    };
    for (int k = tid; k < 4 * RS; k += blockDim.x) QMS[k] = 0.0;
    for (int k = tid; k < 2 * RS; k += blockDim.x) AU[k] = 0.0;
    const int NT = (n + 3) >> 2;
    if (BLK) {
      for (int k = tid; k < (NT * (NT + 1) / 2) * 16; k += blockDim.x) { QMT[k] = 0.0; QM1T[k] = 0.0; }
      for (int k = tid; k < 3 * NTS * 16; k += blockDim.x) SA[k] = 0.0;
    }
    __syncthreads();
    for (int k = tid; k < 31 * 32; k += blockDim.x) {
      const int s = k >> 5, u1 = (k & 31) + 2;
      wg[k] = (s >= 6 && u1 <= s - 2) ? T.x_interior[s] * T.x_ninio[abs(s - 2 * u1)] * scl[s + 2] : 0.0;
    }
    if (tid < 32) {
      wb[tid] = (tid >= 2 && tid <= 30) ? T.x_bulge[tid] * scl[tid + 2] : 0.0;
      w1[tid] = (tid >= 4 && tid <= 30) ? T.x_interior[tid] * T.x_ninio[tid - 2] * scl[tid + 2] : 0.0;
    }
    double *qb_out = qbtri + (size_t)sq * tri_slot;
    if (qm_perseq) {  // the outside pass needs qm and qm1 of every sequence: keep them per sequence instead of per CTA
      QM = qm_perseq + (size_t)sq * 2 * tri_slot;
      QM1 = QM + tri_slot;
    }
    const double bu1 = exp(log(T.x_MLbase) - lns);
    const double xtau = T.x_TerminalAU, inv_tau = 1.0 / xtau;
    const double xclose = T.x_MLclosing * exp(-2.0 * lns);
    if (warp == 0 && n > BF_TURN + 1) {
      const int cnt = build_pair_list(S, n, BF_TURN + 1, LST + ((BF_TURN + 1) & 1) * RS, lane);
      if (lane == 0) s_np[(BF_TURN + 1) & 1] = cnt;
    }
    __syncthreads();

    for (int d = BF_TURN + 1; d <= n; d++) {
      if (warp == NW - 1 && d + 1 <= n - 1) {
        const int cnt = build_pair_list(S, n, d + 1, LST + ((d + 1) & 1) * RS, lane);
        if (lane == 0) s_np[(d + 1) & 1] = cnt;
      }
      if (EXTQ && out5 && warp == NW - 2)
        while (q5_next <= d - 1) q5_step(q5_next++);
      // ------------------------------------------------------------ combine diagonal d-1
      if (d > BF_TURN + 1) {
        const int dd = d - 1, ncell = n - dd, buf = dd & 1;
        const double *pi = PI + buf * NB * RS, *ps = PS + buf * NB * RS;
        for (int cell = tid; cell < ncell; cell += blockDim.x) {
          const int i = cell + 1, j = i + dd;
          const int t = bf_ptype_bases(S[i], S[j]);
          double qms = 0.0, qb = 0.0;
#pragma unroll
          for (int w = 0; w < NB; w++) qms += ps[w * RS + cell];
          const int tI = (i - 1) >> 2, tJ = (j - 1) >> 2, tab = ((i - 1) & 3) * 4 + ((j - 1) & 3);
          if (BLK && tJ - tI >= 6) qms += SA[((tJ - tI) % 3) * NTS * 16 + tI * 16 + tab];
          if (t) {
#pragma unroll
            for (int w = 0; w < NB; w++) qb += pi[w * RS + cell];
            qb += QMS[((dd - 2) & 3) * RS + i + 1] * (xclose * bf_x_mlstem(T, bf_rtype(t), S[j - 1], S[i + 1]));
          }
          double qm1 = 0.0, au = 0.0;
          if (dd > BF_TURN + 1) {
            const int o = toff[dd - 1] + i - 1;
            qm1 = QM1[o] * bu1;                                        // (i, j-1) plus one unpaired base
            au = bu1 * (QM1[o + 1] + AU[((dd - 1) & 1) * RS + i + 1]);  // stems starting right of i
          }
          if (t && i > 1 && j < n) qm1 += qb * bf_x_mlstem(T, t, S[i - 1], S[j + 1]);
          const double qm = qms + au + qm1;
          const int o = toff[dd] + i - 1;
          qb_out[o] = qb;
          QM[o] = qm;
          QM1[o] = qm1;
          if (BLK) {
            const size_t to = (size_t)(tile_off(NT, tI) + tJ - tI) * 16 + tab;
            QMT[to] = qm;
            QM1T[to] = qm1;
          }
          QMS[(dd & 3) * RS + i] = qms;
          AU[(dd & 1) * RS + i] = au;
          const int row = (dd & (kRing - 1)) * RS + i;
          double g = 0.0, g1 = 0.0, gb = 0.0;
          if (t) {
            const int t2 = bf_rtype(t), a = S[j + 1], bb = S[i - 1];
            g = qb * T.x_mmI[t2][a][bb];
            g1 = qb * T.x_mm1nI[t2][a][bb];
            gb = (t > 2) ? qb * xtau : qb;
          }
          QG[row] = g; Q1[row] = g1; QBB[row] = gb;
        }
      }
      // ------------------------------------------------------------ partial sums of diagonal d
      if (d <= n - 1) {
        const int ncell = n - d, buf = d & 1;
        double *pi = PI + (buf * NB + warp % NB) * RS, *ps = PS + (buf * NB + warp % NB) * RS;
        const int smax = min(BF_MAXLOOP, d - 6);
        const int np = s_np[buf];
        const unsigned short *list = LST + buf * RS;
        auto do_interior = [&](const bool add) {
        for (int c = 0; c < np; c += 32) {
          const int kk = c + lane;
          const int i = list[min(kk, np - 1)];
          const int j = i + d;
          const int t = bf_ptype_bases(S[i], S[j]);
          const int si1 = S[i + 1], sj1 = S[j - 1];
          double accg = 0.0, acc1 = 0.0, accb = 0.0;
          constexpr bool kBatchR2 = (NW >= 8 && PL == 0);  // long-sequence configuration: every ring is read through L2
          if (kBatchR2) {
            // bulge and 1xn candidates of this warp's (at most four) loop sizes: all sixteen loads first
            int sv[4], ns = 0;
            BF_FOR_MY_S(NW, warp, smax, s) { if (ns < 4) sv[ns] = s; ns++; }
            double b0[4], b1[4], o0[4], o1[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
              const int s = u < ns ? sv[u] : 2;
              const int row = ((d - 2 - s) & (kRing - 1)) * RS + i;
              b0[u] = QBB[row + 1]; b1[u] = QBB[row + 1 + s];
              o0[u] = Q1[row + 2]; o1[u] = Q1[row + s];
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
              if (u < ns) {
                accb += (b0[u] + b1[u]) * wb[sv[u]];
                if (sv[u] >= 4) acc1 += (o0[u] + o1[u]) * w1[sv[u]];
              }
            }
          }
          BF_FOR_MY_S(NW, warp, smax, s) {
            const int row = ((d - 2 - s) & (kRing - 1)) * RS + i;
            if (!kBatchR2) {
              accb += (QBB[row + 1] + QBB[row + 1 + s]) * wb[s];
              if (s >= 4) acc1 += (Q1[row + 2] + Q1[row + s]) * w1[s];
            }
            if (s >= 6) {
              const double *qp = QG + row + 3;
              const double *w = wg + (s << 5);
              const int kn = s - 3;
              double a0 = 0.0, a1 = 0.0;
              int k = 0;
              if (!(PL & kPfQgSmem)) {  // ring rows come from L2: eight loads in flight
                for (; k + 7 < kn; k += 8) {
                  const double q0 = qp[k], q1 = qp[k + 1], q2 = qp[k + 2], q3 = qp[k + 3], q4 = qp[k + 4], q5 = qp[k + 5], q6 = qp[k + 6], q7 = qp[k + 7];
                  a0 = fma(q0, w[k], a0); a1 = fma(q1, w[k + 1], a1); a0 = fma(q2, w[k + 2], a0); a1 = fma(q3, w[k + 3], a1);
                  a0 = fma(q4, w[k + 4], a0); a1 = fma(q5, w[k + 5], a1); a0 = fma(q6, w[k + 6], a0); a1 = fma(q7, w[k + 7], a1);
                }
              }
              for (; k + 1 < kn; k += 2) { a0 = fma(qp[k], w[k], a0); a1 = fma(qp[k + 1], w[k + 1], a1); }
              if (k < kn) a0 = fma(qp[k], w[k], a0);
              accg += a0 + a1;
            }
          }
          double tot = accg * T.x_mmI[t][si1][sj1] + acc1 * T.x_mm1nI[t][si1][sj1] + accb * (t > 2 ? xtau : 1.0);
          for (int k = (warp + c + d) % NW; k < 10; k += NW) {
            if (k == 9) { tot += bf_x_hairpin(P, T, S, i, j, t) * scl[d + 1]; continue; }
            const int u1 = (0x322211100ull >> (4 * k)) & 15, u2 = (0x232121010ull >> (4 * k)) & 15;
            const int p = i + 1 + u1, q = j - 1 - u2;
            if (q - p <= BF_TURN) continue;
            const int t2 = bf_ptype_bases(S[p], S[q]);
            if (!t2) continue;
            double qv = QBB[((q - p) & (kRing - 1)) * RS + p];  // qb * terminalAU(t2): undo the factor
            if (t2 > 2) qv *= inv_tau;
            tot += qv * bf_x_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1]) * scl[u1 + u2 + 2];
          }
          if (kk < np) pi[i - 1] = add ? pi[i - 1] + tot : tot;
        }
        };
        // ---- qm split for every cell: k = u - i in [5, d-4] (qm on diagonal k-1 >= 4, qm1 on diagonal d-k >= 4)
        auto do_split = [&](const bool add) {
        if (!BLK) {
        for (int c = 0; c < ncell; c += 32) {
          const int cell = c + lane;
          const int i = min(cell, ncell - 1) + 1;
          double accs = 0.0;
          const double *left = QM + (i - 1), *right = QM1 + (i - 1);
          if (d - 8 >= 16 * NW) {
#pragma unroll 8
            for (int k = 5 + warp; k <= d - 4; k += NW) accs = fma(left[toff[k - 1]], right[toff[d - k] + k], accs);
          } else {
#pragma unroll 4
            for (int k = 5 + warp; k <= d - 4; k += NW) accs = fma(left[toff[k - 1]], right[toff[d - k] + k], accs);
          }
          if (cell < ncell) ps[cell] = add ? ps[cell] + accs : accs;
        }
        } else {
        // only the candidates next to either end stay here: k in [5, 12] and [d-10, d-4] minus what the block products cover.
        // Four chunks of 32 cells are handled together so that eight operand pairs are in flight per thread.
        for (int c = 0; c < ncell; c += 128) {
          int xs[4], klo[4], khi[4];
          double accs[4];
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const int x = min(c + 32 * u + lane, ncell - 1);
            const int tI = x >> 2, tJ = (x + d) >> 2;
            xs[u] = x;
            klo[u] = (tJ - tI >= 6) ? 4 * (tI + 3) - x + 1 : 1 << 30;  // covered k range
            khi[u] = 4 * (tJ - 3) + 3 - x + 1;
            accs[u] = 0.0;
          }
          for (int slot = warp; slot < 15; slot += NW) {
            const int k = slot < 8 ? 5 + slot : d - 18 + slot;  // 5..12, d-10..d-4
            if (k < 5 || k > d - 4 || (slot >= 8 && k <= 12)) continue;  // warp-uniform
            const int o1 = toff[k - 1], o2 = toff[d - k] + k;
            double va[4], vb[4];
#pragma unroll
            for (int u = 0; u < 4; u++) { va[u] = QM[xs[u] + o1]; vb[u] = QM1[xs[u] + o2]; }
#pragma unroll
            for (int u = 0; u < 4; u++)
              if (k < klo[u] || k > khi[u]) accs[u] += va[u] * vb[u];
          }
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const int cell = c + 32 * u + lane;
            if (cell < ncell) ps[cell] = add ? ps[cell] + accs[u] : accs[u];
          }
        }
        // block products for tile-diagonal D' = (d+7)/4, quarter q = (d+7)%4 of its tiles
        const int Dp = (d + 7) >> 2, q = (d + 7) & 3;
        if (Dp >= 6 && Dp < NT) {
          const int Tn = NT - Dp;
          double *dst = SA + (Dp % 3) * NTS * 16;
          for (int g = warp; q + 16 * g < Tn; g += NW) {
            const int I = q + 4 * (4 * g + (lane >> 3)), J = I + Dp, sl = (lane >> 1) & 3, hb = (lane & 1) * 2;  // columns hb, hb+1
            double acc[8];
#pragma unroll
            for (int k = 0; k < 8; k++) acc[k] = 0.0;
            if (I < Tn) {
              const double *rowI = QMT + (size_t)tile_off(NT, I) * 16;
              for (int K = I + 3 + sl; K <= J - 3; K += 4) {
                const double *lp = rowI + (K - I) * 16;
                const double *rp = QM1T + (size_t)(tile_off(NT, K) + J - K) * 16 + hb;
                const double *rq = QM1T + (size_t)(tile_off(NT, K + 1) + J - K - 1) * 16 + hb;
                const double2 r0 = *reinterpret_cast<const double2 *>(rp + 4), r1 = *reinterpret_cast<const double2 *>(rp + 8),
                              r2 = *reinterpret_cast<const double2 *>(rp + 12), r3 = *reinterpret_cast<const double2 *>(rq);
#pragma unroll
                for (int a = 0; a < 4; a++) {
                  const double2 l01 = *reinterpret_cast<const double2 *>(lp + a * 4), l23 = *reinterpret_cast<const double2 *>(lp + a * 4 + 2);
                  acc[a * 2 + 0] = fma(l01.x, r0.x, fma(l01.y, r1.x, fma(l23.x, r2.x, fma(l23.y, r3.x, acc[a * 2 + 0]))));
                  acc[a * 2 + 1] = fma(l01.x, r0.y, fma(l01.y, r1.y, fma(l23.x, r2.y, fma(l23.y, r3.y, acc[a * 2 + 1]))));
                }
              }
            }
#pragma unroll
            for (int o = 4; o > 1; o >>= 1) {
#pragma unroll
              for (int k = 0; k < 8; k++) acc[k] += __shfl_xor_sync(BF_FULL, acc[k], o);
            }
            if (I < Tn && sl == 0) {
#pragma unroll
              for (int a = 0; a < 4; a++) *reinterpret_cast<double2 *>(dst + I * 16 + a * 4 + hb) = make_double2(acc[a * 2], acc[a * 2 + 1]);
            }
          }
        }
        }
        };
        if (!HALF) {
          do_interior(false);
          do_split(false);
        } else if (warp < NB) {
          do_interior(false);
          pair_barrier(warp % NB);
          do_split(true);
        } else {
          do_split(false);
          pair_barrier(warp % NB);
          do_interior(true);
        }
      }
      __syncthreads();
    }
    if (EXTQ && out5 && warp == NW - 2) {
      while (q5_next <= n) q5_step(q5_next++);
      if (lane == 0) {
        double *o = out5 + (size_t)sq * 5;
        o[0] = o[1] = o[2] = o[3] = 0.0;
        o[4] = (n > 0) ? -T.kT * (log(q5s[n]) + n * lns) / 1000.0 : 0.0;
      }
    }
  }
}

// exterior pass of the partition function: one warp per sequence on the qb table in HBM
template <int WPB>
__global__ void __launch_bounds__(WPB * 32) bf_k_pf_ext(const BfParams *__restrict__ P, BfBatchDev b, const double *__restrict__ qbtri,
                                                        size_t tri_slot, const double *__restrict__ lnscale, double *out5) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallD T;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  bf_stage(&T, &P->sd);
  __syncthreads();
  const int sq = blockIdx.x * WPB + warp;
  if (sq >= b.B) return;
  const size_t per_warp = align_up((nmax + 4) * sizeof(double) + align_up(nmax + 2, 16), 16);
  unsigned char *base = dyn + per_warp * warp;
  double *q5 = reinterpret_cast<double *>(base);
  uint8_t *S = reinterpret_cast<uint8_t *>(q5 + (nmax + 4));
  const int n = b.len[sq];
  const char *src = b.seq + (size_t)sq * b.stride;
  for (int k = lane; k <= n + 1; k += 32) S[k] = (uint8_t)((k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0);
  const double lns = lnscale[sq], sc1 = exp(-lns);
  const double *qb = qbtri + (size_t)sq * tri_slot;
  if (lane == 0) q5[0] = 1.0;
  __syncwarp();
  // q5[j] = q5[j-1] * scale + sum_i q5[i-1] * qb(i,j) * xExt(i,j): as in bf_k_trace the weights of column j+1 are fetched while
  // column j is reduced.  The products are formed in the order of the plain loop (q5 * qb, then * xExt): same bits.
  auto chain = [&](auto kc) {
    constexpr int K = decltype(kc)::value;
    double curq[K], curx[K], nxtq[K], nxtx[K];
    auto fetch = [&](int j, double *vq, double *vx) {
#pragma unroll
      for (int c = 0; c < K; c++) {
        const int i = 1 + lane + 32 * c;
        double q = 0.0, x = 0.0;
        if (i < j - BF_TURN) {
          const int t = bf_ptype_bases(S[i], S[j]);
          if (t) {
            const int a = (i > 1) ? S[i - 1] : -1, bb = (j < n) ? S[j + 1] : -1;
            q = __ldg(qb + tri_off(n, j - i) + i - 1);
            x = bf_x_ext(T, t, a, bb);
          }
        }
        vq[c] = q; vx[c] = x;
      }
    };
    fetch(1, curq, curx);
    for (int j = 1; j <= n; j++) {
      if (j < n) fetch(j + 1, nxtq, nxtx);
      double sum = 0.0;
#pragma unroll
      for (int c = 0; c < K; c++)
        if (curx[c] != 0.0) sum += q5[lane + 32 * c] * curq[c] * curx[c];
      sum = bf_warp_sum(sum);
      if (lane == 0) q5[j] = sum + q5[j - 1] * sc1;
      __syncwarp();
#pragma unroll
      for (int c = 0; c < K; c++) { curq[c] = nxtq[c]; curx[c] = nxtx[c]; }
    }
  };
  if (n <= 64) chain(std::integral_constant<int, 2>());
  else if (n <= 128) chain(std::integral_constant<int, 4>());
  else if (n <= 256) chain(std::integral_constant<int, 8>());
  else
  for (int j = 1; j <= n; j++) {
    double sum = 0.0;
    for (int i = 1 + lane; i < j - BF_TURN; i += 32) {
      const int t = bf_ptype_bases(S[i], S[j]);
      if (!t) continue;
      const int a = (i > 1) ? S[i - 1] : -1, bb = (j < n) ? S[j + 1] : -1;
      sum += q5[i - 1] * __ldg(qb + tri_off(n, j - i) + i - 1) * bf_x_ext(T, t, a, bb);
    }
    sum = bf_warp_sum(sum);
    if (lane == 0) q5[j] = sum + q5[j - 1] * sc1;
    __syncwarp();
  }
  if (lane == 0 && out5) {
    double *o = out5 + (size_t)sq * 5;
    o[0] = o[1] = o[2] = o[3] = 0.0;
    o[4] = (n > 0) ? -T.kT * (log(q5[n]) + n * lns) / 1000.0 : 0.0;
  }
}

constexpr int kTraceWPB = 4;

size_t trace_smem(int nmax) {
  size_t a = (nmax + 2 + 15) / 16 * 16;
  size_t per_warp = (2 * a + (nmax + 4) * sizeof(int) + (2 * nmax + 16) * sizeof(Sector) + 15) / 16 * 16;
  return per_warp * kTraceWPB;
}
size_t pfext_smem(int nmax) {
  size_t a = (nmax + 2 + 15) / 16 * 16;
  size_t per_warp = ((nmax + 4) * sizeof(double) + a + 15) / 16 * 16;
  return per_warp * kTraceWPB;
}

template <typename K>
cudaError_t set_smem(K kern, size_t sm) {
  return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sm > 1024 ? sm : 1024));
}

// first-fit occupancy grid of a persistent kernel: every sequence its CTA, at most what the GPU runs at once
template <typename K>
cudaError_t occ_grid(K kern, int threads, size_t sm, int B, int sms, int *grid) {
  cudaError_t e = set_smem(kern, sm);
  if (e != cudaSuccess) return e;
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, sm);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  *grid = B < sms * occ ? B : sms * occ;
  return cudaSuccess;
}

}  // namespace

// =====================================================================================================
//                                            host side
// =====================================================================================================
size_t bf_tri_slot(int nmax) { return (tri_size(nmax) + 7) / 8 * 8; }

// ---- configuration: warps per CTA and table placement, from the tuning sweep on B200 (profiles/)
struct FillCfg { int nw, pl; };

// Small batches (a replica-exchange sub-step: B = replicas x targets, often far fewer sequences than the 148 x 2..3 CTA slots):
// what matters is the latency of ONE sequence, so a CTA gets 16 warps instead of 8 when every sequence still gets its own SM.
static bool want_wide(int B, int sms, const BfOpts &o) { return B > 0 && B <= sms && o.wide != 0; }

static bool mfe_fits(int nmax, int nw, int pl) { return mfe_plan(nmax, nw, pl).total <= kSmemBudget; }
static bool pf_fits(int nmax, int nw, int pl) { return pf_plan(nmax, nw, pl).total <= kSmemBudget; }

static bool mfe_blk(int nmax, const FillCfg &c, int blk_min);
// shared partial buffers (atomicMin) where they buy occupancy: CTAs per SM by shared memory, capped by the register limit (4 x 256 threads)
static bool mfe_atom(int nmax, const FillCfg &c, bool blk) {
  auto occ = [&](bool atom) {
    const size_t t = mfe_plan(nmax, c.nw, c.pl, blk, atom).total + 1024;
    const int cap = c.nw == 16 ? 2 : 4;
    const int o = (int)(kSmemBudget / t);
    return t > kSmemBudget ? 0 : (o < cap ? o : cap);
  };
  return occ(true) > occ(false);
}
// blk_min: BF_BLK_MIN (read only when wide)
static FillCfg mfe_cfg(int nmax, bool wide, int blk_min) {
  if (wide)   // same placement rule, 16 warps
    // one CTA per SM: nothing is gained by a small footprint, and with nothing else resident L2 latency is fully exposed --
    // keep on chip whatever fits (fML table + rings, else the rings), shared partial buffers if that is what makes it fit
    for (int pl : {kMfeFmSmem | kMfeRgSmem, kMfeRgSmem, 0}) {
      const FillCfg w{16, pl};
      if (pl != 0 && nmax >= blk_min) continue;   // blocked split: the through-L2 layout measured faster (L=400)
      if (mfe_plan(nmax, 16, pl, mfe_blk(nmax, w, blk_min), true).total <= kSmemBudget) return w;
    }
  // default (tuning sweep, profiles/r01_sweeps.md): rings on chip while >= 3 CTAs still fit on an SM (70 KB), else everything
  // through L2
  const int pl = mfe_plan(nmax, 8, kMfeRgSmem, false, true).total <= 70 * 1024 ? kMfeRgSmem : 0;
  if (mfe_fits(nmax, 8, pl)) return {8, pl};
  return {8, mfe_fits(nmax, 8, 0) ? 0 : -1};
}
static bool pf_blk(int nmax, const FillCfg &c, int blk_min_pf);
static bool pf_half(int nmax, const FillCfg &c);
static FillCfg pf_cfg(int nmax, bool wide, int blk_min_pf) {
  if (wide)   // as for the MFE: one CTA per SM, keep on chip what fits (qm/qm1 + generic ring, else the ring)
    for (int pl : {kPfQmSmem | kPfQgSmem, kPfQgSmem, 0}) {
      const FillCfg w{16, pl};
      if (pl != 0 && nmax >= blk_min_pf) continue;   // blocked split: through-L2 layout only
      if (pf_plan(nmax, 16, pl, pf_half(nmax, w)).total <= kSmemBudget) return w;
    }
  const int pl = pf_plan(nmax, 8, kPfQgSmem).total <= 74 * 1024 ? kPfQgSmem : 0;
  if (pf_fits(nmax, 8, pl)) return {8, pl};
  return {8, pf_fits(nmax, 8, 0) ? 0 : -1};
}

// blocked split (tile-major mirror + block products): for the two default placements.  It pays once the split operands no longer
// fit on chip (measured: L=100 3.86 -> 5.18 ms, L=200 16.1 -> 17.8 ms, L=400 143 -> 117 ms): long sequences only
static bool mfe_blk(int nmax, const FillCfg &c, int blk_min) {
  return (c.pl == 0 || c.pl == kMfeRgSmem) && nmax >= blk_min && mfe_plan(nmax, c.nw, c.pl, true).total <= kSmemBudget;
}
static bool pf_blk(int nmax, const FillCfg &c, int blk_min_pf) { return c.pl == 0 && nmax >= blk_min_pf; }
static bool pf_half(int nmax, const FillCfg &c) {
  // long sequences: with one partial buffer per warp only one CTA fits an SM; sharing buffers between warp pairs fits two
  if (c.nw == 16)   // one CTA per SM: share buffers between warp pairs only when the full set does not fit
    return c.pl == 0 && pf_plan(nmax, 16, 0, false).total > kSmemBudget;
  return c.pl == 0 && pf_plan(nmax, 8, 0, false).total > 113 * 1024 && pf_plan(nmax, 8, 0, true).total <= 113 * 1024;
}

// 0: length not covered by the fill path (the generic kernels take it); else 1 + placement flags.  Decided by the 8-warp
// configuration, which does not depend on the batch.
int bf_fill_mfe_mode(int nmax) {
  if (nmax < 1 || nmax > 2000) return 0;
  return mfe_cfg(nmax, false, 0).pl + 1;
}
int bf_fill_pf_mode(int nmax) {
  if (nmax < 1 || nmax > 2000) return 0;
  return pf_cfg(nmax, false, 0).pl + 1;
}

// ---- the round-1 instantiations, exactly the combinations the rules above return
using MfeFillK = void (*)(const BfParams *, BfBatchDev, int *, int *, size_t, int *, size_t, int *, int *);
struct MfeFillVar { MfeFillK kern; int nw, pl; bool blk, atom; };
#define BF_V(NW_, PL_, BLK_, ATOM_) {bf_k_mfe_fill<NW_, PL_, BLK_, ATOM_>, NW_, PL_, BLK_, ATOM_}
static const MfeFillVar kMfeVars[] = {
    BF_V(8, 0, false, false), BF_V(8, 0, false, true), BF_V(8, 0, true, false), BF_V(8, 0, true, true),
    BF_V(8, kMfeRgSmem, false, false), BF_V(8, kMfeRgSmem, false, true), BF_V(8, kMfeRgSmem, true, false), BF_V(8, kMfeRgSmem, true, true),
    BF_V(16, 0, false, true), BF_V(16, 0, true, false), BF_V(16, 0, true, true),
    BF_V(16, kMfeRgSmem, false, false), BF_V(16, kMfeRgSmem, false, true),
    BF_V(16, kMfeFmSmem | kMfeRgSmem, false, false), BF_V(16, kMfeFmSmem | kMfeRgSmem, false, true)};
#undef BF_V

using PfFillK = void (*)(const BfParams *, BfBatchDev, double *, size_t, double *, size_t, double *, const int *, double *, int *, double *);
struct PfFillVar { PfFillK kern; int nw, pl; bool half, blk; int minb; };
#define BF_V(NW_, PL_, HALF_, BLK_, MINB_) {bf_k_pf_fill<NW_, PL_, HALF_, BLK_, MINB_>, NW_, PL_, HALF_, BLK_, MINB_}
static const PfFillVar kPfVars[] = {
    BF_V(16, kPfQmSmem | kPfQgSmem, false, false, 0), BF_V(16, kPfQgSmem, false, false, 0),
    BF_V(16, 0, true, true, 0), BF_V(16, 0, true, false, 0), BF_V(16, 0, false, true, 0), BF_V(16, 0, false, false, 0),
    BF_V(8, kPfQgSmem, false, false, 0), BF_V(8, 0, true, true, 0), BF_V(8, 0, true, false, 0), BF_V(8, 0, false, true, 0),
    BF_V(8, 0, false, false, 4), BF_V(8, 0, false, false, 3), BF_V(8, 0, false, false, 0)};
#undef BF_V

static cudaError_t round1_mfe_plan(int nmax, int B, bool wide, const BfOpts &o, int sms, BfPlan *p) {
  const FillCfg c = mfe_cfg(nmax, wide, o.blk_min);
  if (c.pl < 0) return cudaErrorInvalidValue;
  const bool blk = mfe_blk(nmax, c, o.blk_min), atom = mfe_atom(nmax, c, blk);
  int key = 0;
  while (key < (int)(sizeof kMfeVars / sizeof kMfeVars[0]) &&
         !(kMfeVars[key].nw == c.nw && kMfeVars[key].pl == c.pl && kMfeVars[key].blk == blk && kMfeVars[key].atom == atom)) key++;
  if (key == (int)(sizeof kMfeVars / sizeof kMfeVars[0])) return cudaErrorInvalidValue;
  p->family = BF_FAM_ROUND1;
  p->key = key;
  p->smem = mfe_plan(nmax, c.nw, c.pl, blk, atom).total;
  // [rings when they are not on chip][tile-major fML mirror when blocked]
  p->ws = 0;
  if (!(c.pl & kMfeRgSmem)) p->ws += ((size_t)3 * kRing * mfe_plan(nmax, c.nw, c.pl).rs + 7) / 8 * 8;
  if (blk) p->ws += (tile_table_entries(nmax) + 7) / 8 * 8;
  return occ_grid(kMfeVars[key].kern, c.nw * 32, p->smem, B, sms, &p->grid);
}

static cudaError_t round1_pf_plan(int nmax, int B, bool wide, const BfOpts &o, int sms, BfPlan *p) {
  const FillCfg c = pf_cfg(nmax, wide, o.blk_min_pf);
  if (c.pl < 0) return cudaErrorInvalidValue;
  const bool half = pf_half(nmax, c), blk = pf_blk(nmax, c, o.blk_min_pf);
  // everything through L2: occupancy is a register question.  Measured (profiles/r01_s4_sweep_pf_minb.log): 4 CTAs per SM pay up
  // to ~135 nt, 3 up to ~185 nt; beyond, the tables of more sequences in flight no longer fit in L2 and the 2-CTA build wins
  const int minb = c.nw == 8 && c.pl == 0 && !half && !blk ? (nmax <= 135 ? 4 : nmax <= 185 ? 3 : 0) : 0;
  int key = 0;
  while (key < (int)(sizeof kPfVars / sizeof kPfVars[0]) &&
         !(kPfVars[key].nw == c.nw && kPfVars[key].pl == c.pl && kPfVars[key].half == half && kPfVars[key].blk == blk && kPfVars[key].minb == minb)) key++;
  if (key == (int)(sizeof kPfVars / sizeof kPfVars[0])) return cudaErrorInvalidValue;
  p->family = BF_FAM_ROUND1;
  p->key = key;
  p->smem = pf_plan(nmax, c.nw, c.pl, half).total;
  // [tables that are not on chip][blocked split: qm/qm1 mirrors, sums]
  size_t ws = pf_ws_doubles(nmax, c.pl);
  if (blk) ws += 2 * ((tile_table_entries(nmax) + 7) / 8 * 8) + (size_t)3 * ((nmax + 3) / 4) * 16;
  p->ws = (ws + 7) / 8 * 8;
  return occ_grid(kPfVars[key].kern, c.nw * 32, p->smem, B, sms, &p->grid);
}

// exterior recursion of a fill that does not run it itself: one CTA per sequence for batches that leave SMs idle (BF_EXT_WIDE=0/1
// overrides), else one warp per sequence
static BfExtRoute ext_route(int stride, int B, int sms, const BfOpts &o) {
  const bool cta = (o.ext_wide >= 0 ? o.ext_wide != 0 : B <= 2 * sms) && bf_ext_wide_ok(stride);
  return cta ? BF_EXT_CTA : BF_EXT_WARP;
}

// The route of a fold pass: the generic kernels for two strands, BF_FORCE_GENERIC and lengths the fill path does not cover; else the
// cluster kernels (rule in bf_cluster.cu; BF_CL=0/1 overrides), then the third-generation kernels (bf_fill3.cu), which take every
// batch they cover -- small batches (want_wide) their 16-warp variants unless BF_FILL3_SMALL=0 --, then the round-1 kernels of this
// file.
cudaError_t bf_plan_mfe(int stride, int B, bool two, bool force_generic, int sms, BfPlan *p) {
  const BfOpts o = bf_opts();
  *p = BfPlan{};
  if (two || force_generic || bf_fill_mfe_mode(stride) == 0) return bf_gen_mfe_plan(stride, B, two, o, sms, p);
  const bool wide = want_wide(B, sms, o), small = wide && o.fill3_small != 0;
  cudaError_t e = cudaSuccess;
  if (!bf_cl_mfe_plan(stride, B, o, p)) {
    if (!wide || small) e = bf_fill3_mfe_plan(stride, B, small, o, sms, p);
    if (e == cudaSuccess && p->family != BF_FAM_TAP) e = round1_mfe_plan(stride, B, wide, o, sms, p);
  }
  const bool in_fill = p->family == BF_FAM_ROUND1 && kMfeVars[p->key].nw == 16;
  p->ext = in_fill ? BF_EXT_IN_FILL : ext_route(stride, B, sms, o);
  return e;
}

cudaError_t bf_plan_pf(int stride, int B, bool two, bool force_generic, int sms, BfPlan *p) {
  const BfOpts o = bf_opts();
  *p = BfPlan{};
  if (two || force_generic || bf_fill_pf_mode(stride) == 0) return bf_gen_pf_plan(stride, B, two, o, sms, p);
  const bool wide = want_wide(B, sms, o), small = wide && o.fill3_small != 0;
  cudaError_t e = cudaSuccess;
  if (!bf_cl_pf_plan(stride, B, o, p)) {
    if (!wide || small) e = bf_fill3_pf_plan(stride, B, small, o, sms, p);
    if (e == cudaSuccess && p->family != BF_FAM_TAP) e = round1_pf_plan(stride, B, wide, o, sms, p);
  }
  const bool in_fill = p->family == BF_FAM_ROUND1 && kPfVars[p->key].nw == 16;
  p->ext = in_fill ? BF_EXT_IN_FILL : ext_route(stride, B, sms, o);
  return e;
}

cudaError_t bf_launch_mfe_fill(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, int *ctri, int *ftri, int *ws, int *work_counter,
                               int *f5_out, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  if (p.family == BF_FAM_CLUSTER) return bf_launch_mfe_cl(p, dP, b, ctri, ftri, ws, work_counter, st);
  if (p.family == BF_FAM_TAP) return bf_launch_mfe_fill3(p, dP, b, ctri, ftri, ws, work_counter, st);
  const MfeFillVar &v = kMfeVars[p.key];
  v.kern<<<p.grid, v.nw * 32, p.smem, st>>>(dP, b, ctri, ftri, bf_tri_slot(b.stride), ws, p.ws, work_counter, f5_out);
  return cudaGetLastError();
}

cudaError_t bf_launch_trace(const BfParams *dP, const BfBatchDev &b, const int *ctri, const int *ftri, int *out_mfe, char *out_ss,
                            int ss_stride, cudaStream_t st, const int *f5_in) {
  auto kern = bf_k_trace<kTraceWPB>;
  const size_t sm = trace_smem(b.stride);
  cudaError_t e = set_smem(kern, sm);
  if (e != cudaSuccess) return e;
  kern<<<(b.B + kTraceWPB - 1) / kTraceWPB, kTraceWPB * 32, sm, st>>>(dP, b, ctri, ftri, bf_tri_slot(b.stride), out_mfe, out_ss, ss_stride, f5_in);
  return cudaGetLastError();
}

cudaError_t bf_launch_pf_fill(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, double *qbtri, double *qmws, double *qmseq,
                              const int *mfe_for_scale, double *lnscale, int *work_counter, double *out5, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  if (p.family == BF_FAM_CLUSTER) return bf_launch_pf_cl(p, dP, b, qbtri, qmws, qmseq, mfe_for_scale, lnscale, work_counter, st);
  if (p.family == BF_FAM_TAP) return bf_launch_pf_fill3(p, dP, b, qbtri, qmws, qmseq, mfe_for_scale, lnscale, work_counter, st);
  const PfFillVar &v = kPfVars[p.key];
  v.kern<<<p.grid, v.nw * 32, p.smem, st>>>(dP, b, qbtri, bf_tri_slot(b.stride), qmws, p.ws, qmseq, mfe_for_scale, lnscale, work_counter, out5);
  return cudaGetLastError();
}

cudaError_t bf_launch_pf_ext(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *lnscale, double *out5,
                             cudaStream_t st) {
  auto kern = bf_k_pf_ext<kTraceWPB>;
  const size_t sm = pfext_smem(b.stride);
  cudaError_t e = set_smem(kern, sm);
  if (e != cudaSuccess) return e;
  kern<<<(b.B + kTraceWPB - 1) / kTraceWPB, kTraceWPB * 32, sm, st>>>(dP, b, qbtri, bf_tri_slot(b.stride), lnscale, out5);
  return cudaGetLastError();
}
