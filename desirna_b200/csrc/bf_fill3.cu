// bf_fill3.cu -- third generation of the single-strand fill kernels (sm_100a): flat tap tables for the interior loops.
//
// Same recurrences, same diagonal-major tables in HBM and the same one-barrier-per-diagonal schedule as bf_fill.cu (the path behind
// fc.mfe() / fc.pf(), utils/energy_scores.py:150-151 in the reference; recurrences SURVEY.md A.4-A.6).  What changed is how a
// diagonal's work is dealt to the lanes, because the round-1 kernels spent 27 thread-instructions per candidate where the candidate
// itself needs two (profiles/r01_s4_ncu_full.txt):
//
//  * Interior loops, the bulk of the work.  The decomposable candidates of a cell (i,j) on diagonal d are
//        ring_kind[(d-2-s) mod 32][i+1+u1] + pen_kind(s,u1)              (u1 + u2 = s <= 30; 375 generic, 54 1xn, 58 bulge)
//    i.e. the SAME 487 (row, column offset, penalty) "taps" for every cell, shifted by i.  One warp takes one pairable cell at a
//    time and its LANES RUN OVER THE TAPS: every lane owns a fixed set of taps (18 "slots": 12 generic, 3 1xn, 3 bulge), keeps their
//    ring offsets and penalties IN REGISTERS for the whole sequence, and a candidate costs exactly one LDS and one add-min
//    (one LDS.64 and one DFMA in the partition function) with no address arithmetic, no penalty load and no idle lane; the warp's
//    minimum / sum is one REDUX / five shuffles per cell.  Advancing to the next diagonal moves every tap one ring row down:
//    two integer instructions per slot (add, wrap by unsigned min).
//    - Taps are assigned to (slot, lane) on the host so that the 32 lanes of a slot hit 32 different banks: the bank of a tap is
//      (u1 - s*c) mod 32 up to a per-cell constant, c = ring row stride mod 32 (mod 16 within each half-warp for the 8-byte
//      partition-function rings).  The row stride is padded to a residue for which the greedy packing succeeds.
//    - Slots are filled in order of loop size, and the short diagonals (d - 6 < 30) run only the leading slots they need.
//    - Nothing is masked: the rings are reset to "no structure" (INF / 0) for every sequence and followed by one neutral row, so a
//      tap that looks at a diagonal which does not exist yet reads a neutral element.
//  * Per-cell constants (outer mismatch terms) are computed once per pairable cell when the diagonal's cell list is compacted
//    (lanes = cells there) and travel in the list entry.
//  * The fML / qm split keeps lanes = cells, all chunks of the diagonal in one thread so that the offset arithmetic (second-order
//    increments of the packed-triangle offsets, no table look-up) is shared by up to four cells; the split points are dealt to
//    the auxiliary warps, partial results meet in the combine step.
//  * Warp specialisation inside a phase: warps [0, NWI) do the tap work; the other warps combine the previous diagonal, evaluate
//    the nine non-decomposable interior candidates and the hairpin (lanes = cells), build the next cell list and do the split.
//    All of it only reads diagonals <= d-2, so a phase still ends with a single barrier.
#include "bf_kernels.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "bf_device.cuh"

#include "bf_taps.cuh"

namespace {


// ---------------------------------------------------------------------------------------------
// per-cell constants: everything that depends on the sequence but not on the DP tables.  A pre-pass (all warps, lanes = cells,
// no barrier between diagonals) writes one entry per PAIRABLE cell, compacted per diagonal, into the CTA's HBM workspace (L2-
// resident); the diagonal loop then contains no energy-table look-up at all.
//   word 0: i      1: mismatchI(outer pair)      2: mismatch1nI(outer pair)     3: hairpin energy
//        4: MLclosing + MLstem(closing pair seen from inside)
//        5: mismatchI(as inner pair)   6: mismatch1nI(as inner pair)   7: terminalAU(pair)   8: MLstem(stem in a multiloop), INF at
//           the sequence ends -- words 5..8 are what lanes 0..3 add to c(i,j) for the three ring rows and the fML candidate
//    9..17: the nine non-decomposable interior candidates (stack, bulge-1, 1x1, 1x2, 2x1, 2x2, 2x3, 3x2): loop energy minus
//           terminalAU(inner pair) -- lanes 0..8 add them to nine more taps on the bulge ring      18, 19: INF (the idle lanes)
// ---------------------------------------------------------------------------------------------
constexpr int kEntWords = 20;
constexpr bool kPrepassInPhases = false;

// ---------------------------------------------------------------------------------------------
// shared-memory plan of the MFE fill
// ---------------------------------------------------------------------------------------------
struct Mfe3Plan {
  size_t o_S, o_SP, o_np, o_ring, o_dml, o_fm, o_stg, o_tmpe, o_stc, o_ps, o_cl, o_pp, total;
};
__host__ __device__ inline Mfe3Plan mfe3_plan(int nmax, int rs, int nw, int nwa) {
  Mfe3Plan p;
  size_t o = 0;
  p.o_ring = o; o += ((size_t)3 * kRing * rs + rs) * sizeof(int);   // three rings + one neutral row
  // split minima: phase d reads row d-2 while the combine writes row d-1, so two rows suffice
  p.o_dml = o; o += (size_t)2 * rs * sizeof(int);
  p.o_fm = o; o += (tri_size(nmax) + 4) * sizeof(int);
  p.o_stg = o; o += (size_t)2 * 3 * rs * sizeof(int);               // newest ring row, staged by the tap warps (double-buffered)
  p.o_tmpe = o; o += (size_t)2 * rs * sizeof(int);                  // c + MLstem of the newest diagonal
  p.o_stc = o; o += (size_t)2 * rs * sizeof(int);                   // c of the newest diagonal (follows TMPE: reset together)
  p.o_ps = o; o += (size_t)2 * nwa * rs * sizeof(int);
  // per-sequence state exists twice: the auxiliary warps prepare the next sequence while the current one is folded
  p.o_np = o; o += (size_t)2 * ((nmax + 4) / 4 * 4) * sizeof(unsigned short);
  p.o_S = o; o += (size_t)2 * ((nmax + 2 + 15) / 16 * 16);
  p.o_SP = o; o += (size_t)2 * ((nmax + 2 + 15) / 16 * 16);
  // per tap warp: the entries of its cells of the current diagonal (copied from L2 one phase ahead)
  o = (o + 15) / 16 * 16;
  p.o_cl = o; o += (size_t)(rs + 2 * nw + 2) * kEntWords * sizeof(int);   // NWI lists of ceil(rs / NWI) + 1 entries each
  p.o_pp = o; o += (size_t)nwa * ((nmax + 7) / 8 * 8) * sizeof(unsigned short);   // pre-pass: pairable cells of one diagonal, per aux warp
  p.total = (o + 15) / 16 * 16;
  return p;
}

__device__ __forceinline__ int lds_s32(unsigned addr) {
  int v;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}

// =====================================================================================================
//                                           MFE fill
// =====================================================================================================
// Phase d of the diagonal loop (one barrier per phase):
//   tap warps [0, NWI):  every pairable cell of diagonal d -- 487 decomposable interior candidates + 9 special ones (taps), hairpin,
//                        multiloop closing (split minima of diagonal d-2) -> c(i,j); staged in STC, in the staging row of the rings
//                        and, with its multiloop-stem term, in TMPE
//   aux warps [NWI, NW): diagonal d-1: staging row -> rings, STC -> c table in HBM (every cell, INF where nothing was staged: one
//                        coalesced row store instead of a scalar store per pairable cell), fML (needs c of d-1, the split minima of
//                        d-1 and fML of d-2); then their share of the split points of diagonal d
// Ring row d must not be written while phase d still reads row d-32 (same slot): hence the staging row.
template <int NW, int NWI>
__global__ void __launch_bounds__(NW * 32, NW <= 8 ? 3 : NW <= 12 ? 2 : 1) bf_k_mfe_fill3(const BfParams *__restrict__ P, BfBatchDev b, int *ctri, int *ftri, size_t tri_slot,
                                                          int *ent_ws, size_t ent_slot, const uint32_t *__restrict__ taps, int RS,
                                                          int *work_counter) {
  constexpr int NWA = NW - NWI;
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq;
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(BF_FULL, tid >> 5, 0);
  const int nmax = b.stride;
  const Mfe3Plan pl = mfe3_plan(nmax, RS, NW, NWA);
  const int seq_pad = (nmax + 2 + 15) / 16 * 16, np_pad = (nmax + 4) / 4 * 4;
  int *RG = reinterpret_cast<int *>(dyn + pl.o_ring);
  int *CG = RG, *C1 = RG + kRing * RS, *CB = RG + 2 * kRing * RS;
  int *DML = reinterpret_cast<int *>(dyn + pl.o_dml);
  int *fms = reinterpret_cast<int *>(dyn + pl.o_fm);
  int *STG = reinterpret_cast<int *>(dyn + pl.o_stg);
  int *TMPE = reinterpret_cast<int *>(dyn + pl.o_tmpe);
  int *STC = reinterpret_cast<int *>(dyn + pl.o_stc);
  int *PS = reinterpret_cast<int *>(dyn + pl.o_ps);
  const BfSmallI &T = P->si;
  const bool tapw = warp < NWI;
  const unsigned char *meta = reinterpret_cast<const unsigned char *>(taps + kNSlot * 32);   // TapMeta: ng[32], n1[32], nb[32]
  int *ent_base = ent_ws + (size_t)blockIdx.x * ent_slot;   // two halves: current and next sequence
  const int tauE = T.TerminalAU;

  // this lane's taps: penalties for the whole launch, ring offsets (bytes) re-based for every sequence
  int pen[kNSlot], xk[kNSlot];
#pragma unroll
  for (int k = 0; k < kNSlot; k++) {
    const uint32_t tp = tapw ? __ldg(taps + k * 32 + lane) : 0u;
    const int s = tp & 255, u1 = (tp >> 8) & 255;
    int v = BF_INF;
    if (tp >> 16) {
      if (k < kNSG) v = T.interior[s] + min(T.ninio_max, abs(s - 2 * u1) * T.ninio_m);
      else if (k < kNSG + kNS1) v = T.interior[s] + min(T.ninio_max, (s - 2) * T.ninio_m);
      else if (k < kNSG + kNS1 + kNSB) v = T.bulge[s];
      else v = 0;   // special slot: the energy travels in the cell's entry
    }
    pen[k] = v;
    xk[k] = 0;
  }
  const unsigned wrap = (unsigned)(kRing * RS);
  const unsigned sCG = (unsigned)__cvta_generic_to_shared(CG);
  const unsigned sFM = (unsigned)__cvta_generic_to_shared(fms);

  // ---- per-sequence state, slot 0 / 1
  auto load_seq = [&](int sq, int slot) -> int {   // all threads; returns the length (warp-uniform for the compiler)
    const int n1 = __shfl_sync(BF_FULL, b.len[sq], 0);
    uint8_t *S1 = dyn + pl.o_S + slot * seq_pad, *SP1 = dyn + pl.o_SP + slot * seq_pad;
    const char *src = b.seq + (size_t)sq * b.stride;
    const uint8_t *np = b.nopair ? b.nopair + (size_t)sq * b.stride : nullptr;
    for (int k = tid; k <= n1 + 1; k += blockDim.x) {
      const int code = (k >= 1 && k <= n1) ? bf_base_code(src[k - 1]) : 0;
      S1[k] = (uint8_t)code;
      SP1[k] = (uint8_t)((np && k >= 1 && k <= n1 && np[k - 1]) ? 0 : code);
    }
    return n1;
  };
  // pre-pass of one diagonal by one warp: per-cell constants (everything that depends on the sequence only) of its pairable cells,
  // compacted, into the slot's half of the workspace.  First the pairable cells are compacted (ballot), then the look-ups run with
  // every lane busy.
  auto prepass_diag = [&](int d, int slot, int n1, unsigned short *cl) {
    const uint8_t *S1 = dyn + pl.o_S + slot * seq_pad, *SP1 = dyn + pl.o_SP + slot * seq_pad;
    unsigned short *NP1 = reinterpret_cast<unsigned short *>(dyn + pl.o_np) + slot * np_pad;
    int *ent1 = ent_base + (size_t)slot * (ent_slot / 2);
    int count = 0;
    const int od = tri_off(n1, d);
    for (int base = 1; base <= n1 - d; base += 32) {
      const int i = base + lane;
      const bool in = i <= n1 - d;
      const int t = in ? bf_ptype_bases(SP1[i], SP1[i + d]) : 0;
      const unsigned mk = __ballot_sync(BF_FULL, t != 0);
      if (t) cl[count + __popc(mk & ((1u << lane) - 1))] = (unsigned short)i;
      count += __popc(mk);
    }
    if (lane == 0) NP1[d] = (unsigned short)count;
    __syncwarp();
    for (int c = lane; c < count; c += 32) {
      const int i = cl[c], j = i + d;
      const int t = bf_ptype_bases(SP1[i], SP1[j]);
      const int si1 = S1[i + 1], sj1 = S1[j - 1], sim = S1[i - 1], sjp = S1[j + 1], tr = bf_rtype(t);
      int4 *dst = reinterpret_cast<int4 *>(ent1 + (size_t)(od + c) * kEntWords);
      dst[0] = make_int4(i, T.mmI[t][si1][sj1], T.mm1nI[t][si1][sj1], bf_e_hairpin(P, T, S1, i, j, t));
      dst[1] = make_int4(T.MLclosing + bf_e_mlstem(T, tr, sj1, si1), T.mmI[tr][sjp][sim], T.mm1nI[tr][sjp][sim], t > 2 ? tauE : 0);
      int w[12];
      w[0] = (i > 1 && j < n1) ? bf_e_mlstem(T, t, sim, sjp) : BF_INF;
#pragma unroll
      for (int k = 0; k < 9; k++) {   // branch-free: the look-ups of a candidate do not wait for the previous candidate
        const int u1 = special_u1(k), u2 = special_u2(k);
        const bool ok = (j - 1 - u2) - (i + 1 + u1) > BF_TURN;
        const int p = ok ? i + 1 + u1 : i + 1, q = ok ? j - 1 - u2 : j - 1;
        const int t2 = ok ? bf_ptype_bases(SP1[p], SP1[q]) : 0;
        const int e = bf_e_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S1[p - 1], S1[q + 1]);
        w[1 + k] = t2 ? e - (t2 > 2 ? tauE : 0) : 0;   // no inner pair: the ring holds INF there
      }
      w[10] = w[11] = BF_INF;
      dst[2] = make_int4(w[0], w[1], w[2], w[3]);
      dst[3] = make_int4(w[4], w[5], w[6], w[7]);
      dst[4] = make_int4(w[8], w[9], w[10], w[11]);
    }
    __syncwarp();
  };

  // ---- first sequence of this CTA: pre-pass by all warps
  if (tid == 0) s_seq = atomicAdd(work_counter, 1);
  __syncthreads();
  int sq = s_seq;
  if (sq >= b.B) return;
  int cur = 0;
  int n = load_seq(sq, 0);
  __syncthreads();
  // (all warps, before any tap list is in use: their scratch lists live in the tap warps' list area)
  unsigned short *cl_all = reinterpret_cast<unsigned short *>(dyn + pl.o_cl) + (size_t)warp * ((nmax + 7) / 8 * 8);
  unsigned short *cl_aux = reinterpret_cast<unsigned short *>(dyn + pl.o_pp) + (size_t)(warp >= NWI ? warp - NWI : 0) * ((nmax + 7) / 8 * 8);
  for (int d = BF_TURN + 1 + warp; d <= n - 1; d += NW) prepass_diag(d, 0, n, cl_all);

  for (;;) {
    __syncthreads();   // the state of sequence sq (slot cur) is complete; nobody reads s_seq or the other slot any more
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    for (int k = tid; k < 3 * kRing * RS + RS; k += blockDim.x) RG[k] = BF_INF;
    for (int k = tid; k < 2 * RS; k += blockDim.x) DML[k] = BF_INF;
    for (int k = tid; k < 6 * RS; k += blockDim.x) STG[k] = BF_INF;
    for (int k = tid; k < 4 * RS; k += blockDim.x) TMPE[k] = BF_INF;   // TMPE and STC
    __syncthreads();
    // the next sequence: its codes now, its pre-pass diagonal by diagonal on the auxiliary warps during the phases below
    const int sqn = s_seq;
    const bool have_next = sqn < b.B;
    const int n1 = have_next ? load_seq(sqn, cur ^ 1) : 0;
    int pd = BF_TURN + 1 + (warp - NWI);   // next pre-pass diagonal of this auxiliary warp
    const unsigned short *NP = reinterpret_cast<const unsigned short *>(dyn + pl.o_np) + cur * np_pad;
    const int *ent = ent_base + (size_t)cur * (ent_slot / 2);
    int *cg_out = ctri + (size_t)sq * tri_slot;
    int *fg_out = ftri + (size_t)sq * tri_slot;
    if (tapw) {
#pragma unroll
      for (int k = 0; k < kNSlot; k++) {
        const uint32_t tp = __ldg(taps + k * 32 + lane);
        const int s = tp & 255, u1 = (tp >> 8) & 255;
        // bytes from the generic ring's origin: ring of the slot's kind, row of diagonal d-2-s for d = TURN+1, column offset 1+u1
        xk[k] = 4 * (((BF_TURN + 1 - 2 - s) & (kRing - 1)) * RS + 1 + u1);   // relative to the origin of the slot's ring variant
      }
    }
    __syncthreads();
    // tap warp: asynchronous copy (LDGSTS) of the entries of its cells (c = warp, warp + NWI, ...) of diagonal dn into its list
    int *wl = reinterpret_cast<int *>(dyn + pl.o_cl) + (size_t)warp * ((RS + NWI - 1) / NWI + 1) * kEntWords;
    auto stage = [&](int dn) {
      const int mine = (NP[dn] - warp + NWI - 1) / NWI;
      const char *src = reinterpret_cast<const char *>(ent + ((size_t)tri_off(n, dn) + warp) * kEntWords);
      const unsigned dst = (unsigned)__cvta_generic_to_shared(wl);
      for (int idx = lane; idx < mine * (kEntWords / 4); idx += 32) {
        const int m = idx / (kEntWords / 4), q = idx - m * (kEntWords / 4);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + (unsigned)(m * kEntWords * 4 + q * 16)),
                     "l"(src + (size_t)m * NWI * kEntWords * 4 + q * 16)
                     : "memory");
      }
    };
    if (tapw && n - 1 >= BF_TURN + 1) stage(BF_TURN + 1);

    for (int d = BF_TURN + 1; d <= n; d++) {
      const int buf = d & 1;
      if (tapw) {
        // ------------------------------------------------------------ tap warps: c(i,j) of every pairable cell of diagonal d
        if (d <= n - 1) {
          const int np = NP[d];
          const unsigned sdml = (unsigned)__cvta_generic_to_shared(DML + ((d - 2) & 1) * RS + 1);
          // lanes 0..2 write the staged ring row (generic, 1xn, bulge variant), lane 3 the fML candidate, lane 4 c itself: lane's
          // target array, and the mask that drops the entry word lane 4 would add
          const unsigned stail = (unsigned)__cvta_generic_to_shared(lane < 3 ? STG + (buf * 3 + lane) * RS : lane == 3 ? TMPE + buf * RS : STC + buf * RS);
          const int tlmask = lane == 4 ? 0 : -1;
          const int smax = min(BF_MAXLOOP, d - 6);
          const int mi = smax + 1 < 0 ? 0 : smax + 1;
          const int ng = __ldg(meta + mi), n1 = __ldg(meta + 32 + mi), nb = __ldg(meta + 64 + mi);
          const int lsp = 9 + min(lane, 9), ltl = 5 + min(lane, 3);
          auto cells = [&](auto cg_, auto c1_, auto cb_) {
            constexpr int G = decltype(cg_)::value, O = decltype(c1_)::value, Bn = decltype(cb_)::value;
            // the warp's entries were copied from L2 into its private list while the previous phase finished
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncwarp();
            const int *p = wl;
            for (int c = warp; c < np; c += NWI, p += kEntWords) {
              const int4 ea = *reinterpret_cast<const int4 *>(p);   // i, mismatchI, mismatch1nI, hairpin
              const int ic = ea.x, mlc = p[4], tau = p[7], esp = p[lsp], etl = p[ltl] & tlmask;
              // the cell index is the same in every lane: taken through REDUX it lands in a uniform register, and a tap load
              // becomes LDS [R + UR] -- the lane's byte offset in a register, the cell's ring address uniform
              const unsigned i4 = 4u * (unsigned)__reduce_min_sync(BF_FULL, ic);
              const unsigned ug = sCG + i4, u1n = ug + 4u * wrap, ubg = ug + 8u * wrap;   // generic, 1xn, bulge ring
              int ag = BF_INF, a1 = BF_INF, ab = BF_INF;
#pragma unroll
              for (int k = 0; k < G; k++) ag = min(ag, lds_s32(ug + xk[k]) + pen[k]);
#pragma unroll
              for (int k = 0; k < O; k++) a1 = min(a1, lds_s32(u1n + xk[kNSG + k]) + pen[kNSG + k]);
#pragma unroll
              for (int k = 0; k < Bn; k++) ab = min(ab, lds_s32(ubg + xk[kNSG + kNS1 + k]) + pen[kNSG + kNS1 + k]);
              const int vs = lds_s32(ubg + xk[kNSlot - 1]) + esp;   // special candidates (lanes 0..8; the others add INF)
              int tot = min(min(ag + ea.y, a1 + ea.z), min(ab + tau, vs));
              tot = __reduce_min_sync(BF_FULL, tot);
              tot = min(tot, ea.w);                                  // hairpin
              const int dm = lds_s32(sdml + i4);                     // split minimum of (i+1, j-1)
              if (dm < kInfThr) tot = min(tot, dm + mlc);            // multiloop closed by (i,j)
              const bool fin = tot < kInfThr;
              const int v = (fin && etl < kInfThr) ? tot + etl : BF_INF;
              if (lane < 5) asm volatile("st.shared.s32 [%0], %1;" ::"r"(stail + i4), "r"(v) : "memory");
            }
          };
          using std::integral_constant;
          if (ng <= 2 && n1 <= 1 && nb <= 1) cells(integral_constant<int, 2>(), integral_constant<int, 1>(), integral_constant<int, 1>());
          else if (ng <= 5 && n1 <= 2 && nb <= 2) cells(integral_constant<int, 5>(), integral_constant<int, 2>(), integral_constant<int, 2>());
          else if (ng <= 8) cells(integral_constant<int, 8>(), integral_constant<int, kNS1>(), integral_constant<int, kNSB>());
          else cells(integral_constant<int, kNSG>(), integral_constant<int, kNS1>(), integral_constant<int, kNSB>());
          __syncwarp();
          if (d + 1 <= n - 1) stage(d + 1);
        }
        // every tap moves one ring row down for the next diagonal
#pragma unroll
        for (int k = 0; k < kNSlot; k++) {   // add, wrap by unsigned min
          const unsigned x = (unsigned)xk[k] + 4u * (unsigned)RS;
          xk[k] = (int)min(x, x - 4u * wrap);
        }
      } else {
        const int a = warp - NWI;   // auxiliary warp index
        // ------------------------------------------------------------ diagonal d-1: staging row -> rings, fML
        if (d > BF_TURN + 1) {
          const int dd = d - 1, ncell = n - dd, pb = dd & 1;
          int *stg = STG + pb * 3 * RS, *tmpe = TMPE + pb * RS, *stc = STC + pb * RS;
          const int *ps = PS + pb * NWA * RS;
          const int row = (dd & (kRing - 1)) * RS;
          const int o0 = tri_off(n, dd), om = dd > BF_TURN + 1 ? tri_off(n, dd - 1) : 0;
          for (int cell = a * 32 + lane; cell < ncell; cell += NWA * 32) {
            const int i = cell + 1;
            int sp = BF_INF;
#pragma unroll
            for (int w = 0; w < NWA; w++) sp = min(sp, ps[w * RS + cell]);
            if (sp >= kInfThr) sp = BF_INF;
            const int eg = stg[i], e1 = stg[RS + i], eb = stg[2 * RS + i], te = tmpe[i], cv = stc[i];
            stg[i] = BF_INF; stg[RS + i] = BF_INF; stg[2 * RS + i] = BF_INF; tmpe[i] = BF_INF; stc[i] = BF_INF;   // only pairable cells are written
            CG[row + i] = eg; C1[row + i] = e1; CB[row + i] = eb;
            cg_out[o0 + i - 1] = cv;
            int m = min(sp, te);
            if (dd > BF_TURN + 1) m = min(m, min(fms[om + i], fms[om + i - 1]) + T.MLbase);
            if (m >= kInfThr) m = BF_INF;
            fg_out[o0 + i - 1] = m;
            fms[o0 + i - 1] = m;
            DML[(dd & 1) * RS + i] = sp;
          }
        }
        if (d <= n - 1) {
          const int ncell = n - d;
          // ------------------------------------------------------------ fML split: this warp's share of the split points, every cell
          int *ps = PS + (buf * NWA + a) * RS;
          constexpr int Q = NWA;
          // operands of split point k: fML(i, i+k-1) at off(k-1) + cell, fML(i+k, j) at off(d-k) + k + cell.  The offsets are
          // warp-uniform and advance by second-order increments (off(x+Q) - off(x) = Q(n-x) - Q(Q-1)/2): they live in uniform
          // registers, a load is LDS [lane's cell offset + uniform].
          for (int c0 = 0; c0 < ncell; c0 += 128) {
            int ii[4], acc[4];
#pragma unroll
            for (int u = 0; u < 4; u++) { ii[u] = 4 * min(c0 + 32 * u + lane, ncell - 1); acc[u] = BF_INF; }   // byte offset of the lane's cell
            const bool many = c0 + 64 < ncell;   // warp-uniform: more than two chunks left
            int k = 5 + a;
            if (k <= d - 4) {
              // running byte addresses of the two operands of every chunk; both advance by the same (uniform) first differences
              const int oL = 4 * tri_off(n, k - 1), oR = 4 * (tri_off(n, d - k) + k);
              int dL = 4 * (Q * (n - k + 1) - Q * (Q - 1) / 2), dR = 4 * (-Q * (n - d + k + Q) + Q * (Q - 1) / 2 + Q);
              unsigned pL[4], pR[4];
#pragma unroll
              for (int u = 0; u < 4; u++) { pL[u] = sFM + (unsigned)(oL + ii[u]); pR[u] = sFM + (unsigned)(oR + ii[u]); }
              if (many) {
#pragma unroll 2
                for (; k <= d - 4; k += Q) {
#pragma unroll
                  for (int u = 0; u < 4; u++) { acc[u] = min(acc[u], lds_s32(pL[u]) + lds_s32(pR[u])); pL[u] += dL; pR[u] += dR; }
                  dL -= 4 * Q * Q; dR -= 4 * Q * Q;
                }
              } else {
#pragma unroll 4
                for (; k <= d - 4; k += Q) {
#pragma unroll
                  for (int u = 0; u < 2; u++) { acc[u] = min(acc[u], lds_s32(pL[u]) + lds_s32(pR[u])); pL[u] += dL; pR[u] += dR; }
                  dL -= 4 * Q * Q; dR -= 4 * Q * Q;
                }
              }
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
              const int cell = c0 + 32 * u + lane;
              if (cell < ncell) ps[cell] = acc[u];
            }
          }
        }
        // ------------------------------------------------------------ one diagonal of the NEXT sequence's pre-pass
        // (measured: two auxiliary warps cannot hide it -- 780 instructions per 32 pairable cells, 3.07 against 2.57 ms per 4096
        // folds at L = 100 -- so by default all warps do it between two sequences, below)
        if (kPrepassInPhases && have_next && pd <= n1 - 1) {
          prepass_diag(pd, cur ^ 1, n1, cl_aux);
          pd += NWA;
        }
      }
      __syncthreads();
    }
    if (!have_next) break;
    // what the auxiliary warps did not reach (a next sequence much longer than this one): all warps
    for (int d = BF_TURN + 1 + (kPrepassInPhases ? NWA * (n - BF_TURN > 0 ? n - BF_TURN : 0) : 0) + warp; d <= n1 - 1; d += NW)
      prepass_diag(d, cur ^ 1, n1, cl_all);
    sq = sqn;
    n = n1;
    cur ^= 1;
  }
}

// =====================================================================================================
//                                   partition function (inside) fill
// =====================================================================================================
// Same organisation as bf_k_mfe_fill3 with sums of Boltzmann weights (fp64) in place of minima:
//   qb(i,j)  = hairpin + sum over the taps (ring value x weight) + qms(i+1,j-1) x closing            -- tap warps, phase d
//   qm1(i,j) = qm1(i,j-1) bu + qb(i,j) xMLstem;  au(i,j) = bu (qm1(i+1,j) + au(i+1,j));  qm = qms + au + qm1   -- aux warps, phase d+1
//   qms(i,j) = sum_k qm(i,i+k-1) qm1(i+k,j)                                                         -- aux warps, phase d
// Tap weights carry the per-sequence scale (pf_scale^-(s+2)), so they are rebuilt for every sequence; a tap costs one LDS.64 and
// one DFMA, the warp's sum five shuffle steps.  Entry of a pairable cell: 20 doubles
//   0: i (int)   1: xmismatchI(outer)   2: xmismatch1nI(outer)   3: hairpin weight x scale   4: xMLclosing x xMLstem(closing)
//   5: xmismatchI(inner role)   6: xmismatch1nI(inner role)   7: xterminalAU(pair)   8: xMLstem(stem), 0 at the sequence ends
//   9..17: weights of the nine non-decomposable interior candidates / xterminalAU(inner pair)     18, 19: 0
constexpr int kEntD = 20;

struct Pf3Plan {
  size_t o_S, o_np, o_ring, o_qms, o_au, o_qm, o_qm1, o_stg, o_tmpq, o_ps, o_scl, o_cl, o_pp, total;
};
__host__ __device__ inline Pf3Plan pf3_plan(int nmax, int rs, int nw, int nwa, bool qms) {
  Pf3Plan p;
  size_t o = 0;
  p.o_ring = o; o += ((size_t)3 * kRing * rs + rs) * sizeof(double);
  p.o_qms = o; o += (size_t)4 * rs * sizeof(double);
  p.o_au = o; o += (size_t)2 * rs * sizeof(double);
  p.o_qm = o; o += qms ? (tri_size(nmax) + 4) * sizeof(double) : 0;
  p.o_qm1 = o; o += qms ? (tri_size(nmax) + 4) * sizeof(double) : 0;
  p.o_stg = o; o += (size_t)2 * 3 * rs * sizeof(double);
  p.o_tmpq = o; o += (size_t)2 * rs * sizeof(double);
  p.o_ps = o; o += (size_t)2 * nwa * rs * sizeof(double);
  p.o_scl = o; o += (size_t)(nmax + 8 > 40 ? nmax + 8 : 40) * sizeof(double);   // the tap weights need scale^k up to k = 32
  o = (o + 15) / 16 * 16;   // LDGSTS copies 16 bytes at a time
  p.o_cl = o; o += (size_t)(rs + 2 * nw + 2) * kEntD * sizeof(double);   // NWI lists of ceil(rs / NWI) + 1 entries each
  p.o_np = o; o += (size_t)((nmax + 4) / 4 * 4) * sizeof(unsigned short);
  p.o_pp = o; o += (size_t)nw * ((nmax + 7) / 8 * 8) * sizeof(unsigned short);
  p.o_S = o; o += (nmax + 2 + 15) / 16 * 16;
  p.total = (o + 15) / 16 * 16;
  return p;
}

__device__ __forceinline__ double lds_f64(unsigned addr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}

// PAIR: a tap warp works on two cells at a time (twice the loads in flight, one shared butterfly: lanes 0..15 end up with the
// first cell's sum, lanes 16..31 with the second's); costs ~40 registers, used by the configurations that can afford them
template <int NW, int NWI, bool QMSM, bool PAIR = false>
__global__ void __launch_bounds__(NW * 32, NW <= 8 ? 2 : 1) bf_k_pf_fill3(const BfParams *__restrict__ P, BfBatchDev b, double *qbtri, size_t tri_slot,
                                                                          double *ws, size_t ws_slot, double *qm_perseq,
                                                                          const int *__restrict__ mfe_for_scale, double *lnscale_out,
                                                                          const uint32_t *__restrict__ taps, int RS, int *work_counter) {
  constexpr int NWA = NW - NWI;
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq;
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(BF_FULL, tid >> 5, 0);
  const int nmax = b.stride;
  const Pf3Plan pl = pf3_plan(nmax, RS, NW, NWA, QMSM);
  uint8_t *S = dyn + pl.o_S;
  unsigned short *NP = reinterpret_cast<unsigned short *>(dyn + pl.o_np);
  double *RG = reinterpret_cast<double *>(dyn + pl.o_ring);
  double *QG = RG, *Q1 = RG + kRing * RS, *QBB = RG + 2 * kRing * RS;
  double *QMS = reinterpret_cast<double *>(dyn + pl.o_qms);
  double *AU = reinterpret_cast<double *>(dyn + pl.o_au);
  double *STG = reinterpret_cast<double *>(dyn + pl.o_stg);
  double *TMPQ = reinterpret_cast<double *>(dyn + pl.o_tmpq);
  double *PS = reinterpret_cast<double *>(dyn + pl.o_ps);
  double *scl = reinterpret_cast<double *>(dyn + pl.o_scl);
  const BfSmallD &T = P->sd;
  const bool tapw = warp < NWI;
  const unsigned char *meta = reinterpret_cast<const unsigned char *>(taps + kNSlot * 32);
  // per-CTA HBM workspace: [entries of every cell][qm, qm1 when they are not on chip]
  double *ent = ws + (size_t)blockIdx.x * ws_slot;
  const size_t tri_pad = (tri_size(nmax) + 7) / 8 * 8;
  double *QM = QMSM ? reinterpret_cast<double *>(dyn + pl.o_qm) : ent + tri_pad * kEntD;
  double *QM1 = QMSM ? reinterpret_cast<double *>(dyn + pl.o_qm1) : QM + tri_pad;
  const double xtau = T.x_TerminalAU, inv_tau = 1.0 / xtau;

  double wk[kNSlot - 1];
  int xk[kNSlot];
  const unsigned wrap = (unsigned)(kRing * RS);
  const unsigned sQG = (unsigned)__cvta_generic_to_shared(QG);
  const unsigned sQM = (unsigned)__cvta_generic_to_shared(QM), sQM1 = (unsigned)__cvta_generic_to_shared(QM1);

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int sq = s_seq;
    if (sq >= b.B) break;
    const int n = __shfl_sync(BF_FULL, b.len[sq], 0);
    {
      const char *src = b.seq + (size_t)sq * b.stride;
      for (int k = tid; k <= n + 1; k += blockDim.x) S[k] = (uint8_t)((k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0);
    }
    // per-nucleotide scale (ViennaRNA exp_params_rescale, sfact 1.07; default estimate -185 cal/mol/nt)
    double lns = 185.0 / T.kT;
    if (mfe_for_scale && n > 0) {
      const double m = (double)mfe_for_scale[sq] * 10.0;
      if (m < 0.0) lns = -1.07 * m / T.kT / (double)n;
      if (lns < 185.0 / T.kT * 0.25) lns = 185.0 / T.kT * 0.25;
    }
    for (int k = tid; k <= (n + 2 > 34 ? n + 2 : 34); k += blockDim.x) scl[k] = exp(-lns * k);
    if (tid == 0 && lnscale_out) lnscale_out[sq] = lns;
    const double bu1 = exp(log(T.x_MLbase) - lns);
    const double xclose = T.x_MLclosing * exp(-2.0 * lns);
    for (int k = tid; k < 3 * kRing * RS + RS; k += blockDim.x) RG[k] = 0.0;
    for (int k = tid; k < 4 * RS; k += blockDim.x) QMS[k] = 0.0;
    for (int k = tid; k < 2 * RS; k += blockDim.x) { AU[k] = 0.0; TMPQ[k] = 0.0; }
    for (int k = tid; k < 6 * RS; k += blockDim.x) STG[k] = 0.0;
    double *qb_out = qbtri + (size_t)sq * tri_slot;
    double *qmg = qm_perseq ? qm_perseq + (size_t)sq * 2 * tri_slot : nullptr;   // the outside pass wants qm / qm1 of every sequence
    __syncthreads();
    if (tapw) {
#pragma unroll
      for (int k = 0; k < kNSlot; k++) {
        const uint32_t tp = __ldg(taps + k * 32 + lane);
        const int s = tp & 255, u1 = (tp >> 8) & 255;
        xk[k] = 8 * (((BF_TURN + 1 - 2 - s) & (kRing - 1)) * RS + 1 + u1);   // relative to the origin of the slot's ring variant
        if (k < kNSlot - 1) {
          double v = 0.0;
          if (tp >> 16) {
            if (k < kNSG) v = T.x_interior[s] * T.x_ninio[abs(s - 2 * u1)] * scl[s + 2];
            else if (k < kNSG + kNS1) v = T.x_interior[s] * T.x_ninio[s - 2] * scl[s + 2];
            else v = T.x_bulge[s] * scl[s + 2];
          }
          wk[k] = v;
        }
      }
    }
    // ------------------------------------------------------------ pre-pass: per-cell constants of every diagonal
    {
      unsigned short *cl = reinterpret_cast<unsigned short *>(dyn + pl.o_pp) + (size_t)warp * ((nmax + 7) / 8 * 8);
      for (int d = BF_TURN + 1 + warp; d <= n - 1; d += NW) {
        int count = 0;
        const int od = tri_off(n, d);
        for (int base = 1; base <= n - d; base += 32) {
          const int i = base + lane;
          const bool in = i <= n - d;
          const int t = in ? bf_ptype_bases(S[i], S[i + d]) : 0;
          const unsigned mk = __ballot_sync(BF_FULL, t != 0);
          if (in && !t) qb_out[od + i - 1] = 0.0;
          if (t) cl[count + __popc(mk & ((1u << lane) - 1))] = (unsigned short)i;
          count += __popc(mk);
        }
        if (lane == 0) NP[d] = (unsigned short)count;
        __syncwarp();
        for (int c = lane; c < count; c += 32) {
          const int i = cl[c], j = i + d;
          const int t = bf_ptype_bases(S[i], S[j]);
          const int si1 = S[i + 1], sj1 = S[j - 1], sim = S[i - 1], sjp = S[j + 1], tr = bf_rtype(t);
          double2 *dst = reinterpret_cast<double2 *>(ent + (size_t)(od + c) * kEntD);
          dst[0] = make_double2(__longlong_as_double((long long)i), T.x_mmI[t][si1][sj1]);
          dst[1] = make_double2(T.x_mm1nI[t][si1][sj1], bf_x_hairpin(P, T, S, i, j, t) * scl[d + 1]);
          dst[2] = make_double2(xclose * bf_x_mlstem(T, tr, sj1, si1), T.x_mmI[tr][sjp][sim]);
          dst[3] = make_double2(T.x_mm1nI[tr][sjp][sim], t > 2 ? xtau : 1.0);
          double w[12];
          w[0] = (i > 1 && j < n) ? bf_x_mlstem(T, t, sim, sjp) : 0.0;
#pragma unroll
          for (int k = 0; k < 9; k++) {
            const int u1 = special_u1(k), u2 = special_u2(k);
            const bool ok = (j - 1 - u2) - (i + 1 + u1) > BF_TURN;
            const int p = ok ? i + 1 + u1 : i + 1, q = ok ? j - 1 - u2 : j - 1;
            const int t2 = ok ? bf_ptype_bases(S[p], S[q]) : 0;
            const double e = bf_x_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1]) * scl[u1 + u2 + 2];
            w[1 + k] = t2 ? (t2 > 2 ? e * inv_tau : e) : 0.0;   // the bulge ring carries xterminalAU of the inner pair
          }
          w[10] = w[11] = 0.0;
#pragma unroll
          for (int q2 = 0; q2 < 6; q2++) dst[4 + q2] = make_double2(w[2 * q2], w[2 * q2 + 1]);
        }
        __syncwarp();
      }
    }
    __syncthreads();
    // tap warp: asynchronous copy (LDGSTS) of the entries of its cells (c = warp, warp + NWI, ...) of diagonal dn into its list
    double *wl = reinterpret_cast<double *>(dyn + pl.o_cl) + (size_t)warp * ((RS + NWI - 1) / NWI + 1) * kEntD;
    auto stage = [&](int dn) {
      const int mine = ((int)NP[dn] - warp + NWI - 1) / NWI;
      const char *src = reinterpret_cast<const char *>(ent + ((size_t)tri_off(n, dn) + warp) * kEntD);
      const unsigned dst = (unsigned)__cvta_generic_to_shared(wl);
      constexpr int CH = kEntD * 8 / 16;
      for (int idx = lane; idx < mine * CH; idx += 32) {
        const int m = idx / CH, q = idx - m * CH;
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + (unsigned)(m * kEntD * 8 + q * 16)),
                     "l"(src + (size_t)m * NWI * kEntD * 8 + q * 16)
                     : "memory");
      }
    };
    if (tapw && n - 1 >= BF_TURN + 1) stage(BF_TURN + 1);

    for (int d = BF_TURN + 1; d <= n; d++) {
      const int buf = d & 1;
      if (tapw) {
        // ------------------------------------------------------------ tap warps: qb(i,j) of every pairable cell of diagonal d
        if (d <= n - 1) {
          const int np = NP[d];
          const int od = tri_off(n, d);
          const unsigned sqms = (unsigned)__cvta_generic_to_shared(QMS + ((d - 2) & 3) * RS + 1);
          // lanes 0..2 write the staged ring row (generic, 1xn, bulge variant), lane 3 qb x xMLstem: lane's target array
          const int ltail = PAIR ? (lane & 15) : lane;
          const unsigned stail = (unsigned)__cvta_generic_to_shared(ltail < 3 ? STG + (buf * 3 + ltail) * RS : TMPQ + buf * RS);
          const int smax = min(BF_MAXLOOP, d - 6);
          const int mi = smax + 1 < 0 ? 0 : smax + 1;
          const int ng = __ldg(meta + mi), n1 = __ldg(meta + 32 + mi), nb = __ldg(meta + 64 + mi);
          const int lsp = 9 + min(lane, 9), ltl = 5 + min(lane & (PAIR ? 15 : 31), 3);
          auto cells = [&](auto cg_, auto c1_, auto cb_) {
            constexpr int G = decltype(cg_)::value, O = decltype(c1_)::value, Bn = decltype(cb_)::value;
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncwarp();
            if (PAIR) {
              const bool hi = lane >= 16;
              const double *p = wl;
              for (int c = warp; c < np; c += 2 * NWI, p += 2 * kEntD) {
                const bool hasB = c + NWI < np;
                const double *pA = p, *pB = hasB ? p + kEntD : p;   // no second cell: the first once more, its stores dropped
                const double2 a01 = *reinterpret_cast<const double2 *>(pA), b01 = *reinterpret_cast<const double2 *>(pB);
                const double x1A = pA[2], xtA = pA[7], espA = pA[lsp], x1B = pB[2], xtB = pB[7], espB = pB[lsp];
                const unsigned iA = 8u * (unsigned)(int)__double_as_longlong(a01.x), iB = 8u * (unsigned)(int)__double_as_longlong(b01.x);
                const unsigned uA = sQG + iA, uB = sQG + iB, u1A = uA + 8u * wrap, u1B = uB + 8u * wrap, ubA = uA + 16u * wrap, ubB = uB + 16u * wrap;
                double gA = 0.0, gB = 0.0, oA = 0.0, oB = 0.0, bA = 0.0, bB = 0.0;
#pragma unroll
                for (int k = 0; k < G; k++) { gA = fma(lds_f64(uA + xk[k]), wk[k], gA); gB = fma(lds_f64(uB + xk[k]), wk[k], gB); }
#pragma unroll
                for (int k = 0; k < O; k++) {
                  oA = fma(lds_f64(u1A + xk[kNSG + k]), wk[kNSG + k], oA);
                  oB = fma(lds_f64(u1B + xk[kNSG + k]), wk[kNSG + k], oB);
                }
#pragma unroll
                for (int k = 0; k < Bn; k++) {
                  bA = fma(lds_f64(ubA + xk[kNSG + kNS1 + k]), wk[kNSG + kNS1 + k], bA);
                  bB = fma(lds_f64(ubB + xk[kNSG + kNS1 + k]), wk[kNSG + kNS1 + k], bB);
                }
                double tA = fma(lds_f64(ubA + xk[kNSlot - 1]), espA, gA * a01.y), tB = fma(lds_f64(ubB + xk[kNSlot - 1]), espB, gB * b01.y);
                tA = fma(oA, x1A, fma(bA, xtA, tA));
                tB = fma(oB, x1B, fma(bB, xtB, tB));
                // one butterfly for both cells
                double keep = hi ? tB : tA;
                keep += __shfl_xor_sync(BF_FULL, hi ? tA : tB, 16);
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) keep += __shfl_xor_sync(BF_FULL, keep, o);
                const double *pm = hi ? pB : pA;
                const unsigned im = hi ? iB : iA;
                const double qb = keep + pm[3] + lds_f64(sqms + im) * pm[4];   // + hairpin + multiloop closed by (i,j)
                if ((lane & 15) < 4 && (!hi || hasB)) asm volatile("st.shared.f64 [%0], %1;" ::"r"(stail + im), "d"(qb * pm[ltl]) : "memory");
                if ((lane & 15) == 0 && (!hi || hasB)) qb_out[od + (int)(im >> 3) - 1] = qb;
              }
              return;
            }
            const double *p = wl;
            double2 e01n = *reinterpret_cast<const double2 *>(p);   // the next cell's index and first field: one cell ahead
            for (int c = warp; c < np; c += NWI, p += kEntD) {
              const double2 e01 = e01n, e23 = *reinterpret_cast<const double2 *>(p + 2);
              const double mlc = p[4], xt = p[7], esp = p[lsp], etl = p[ltl];
              e01n = *reinterpret_cast<const double2 *>(p + kEntD);   // (the list has one spare entry)
              // every lane holds the same cell index; the addresses are formed per lane (no detour through a uniform register:
              // with 8-byte taps the compiler adds per lane anyway)
              const unsigned i8 = 8u * (unsigned)(int)__double_as_longlong(e01.x);
              const unsigned ug = sQG + i8, u1n = ug + 8u * wrap, ubg = ug + 16u * wrap;
              double ag0 = 0.0, ag1 = 0.0, a1 = 0.0, ab = 0.0;
#pragma unroll
              for (int k = 0; k < G; k++) {
                if (k & 1) ag1 = fma(lds_f64(ug + xk[k]), wk[k], ag1);
                else ag0 = fma(lds_f64(ug + xk[k]), wk[k], ag0);
              }
#pragma unroll
              for (int k = 0; k < O; k++) a1 = fma(lds_f64(u1n + xk[kNSG + k]), wk[kNSG + k], a1);
#pragma unroll
              for (int k = 0; k < Bn; k++) ab = fma(lds_f64(ubg + xk[kNSG + kNS1 + k]), wk[kNSG + kNS1 + k], ab);
              double tot = fma(lds_f64(ubg + xk[kNSlot - 1]), esp, (ag0 + ag1) * e01.y);   // special candidates (lanes 0..8)
              tot = fma(a1, e23.x, fma(ab, xt, tot));
              tot = bf_warp_sum(tot);
              const double qb = tot + e23.y + lds_f64(sqms + i8) * mlc;   // + hairpin + multiloop closed by (i,j)
              if (lane < 4) asm volatile("st.shared.f64 [%0], %1;" ::"r"(stail + i8), "d"(qb * etl) : "memory");
              if (lane == 0) qb_out[od + (int)(i8 >> 3) - 1] = qb;
            }
          };
          using std::integral_constant;
          if (ng <= 2 && n1 <= 1 && nb <= 1) cells(integral_constant<int, 2>(), integral_constant<int, 1>(), integral_constant<int, 1>());
          else if (ng <= 5 && n1 <= 2 && nb <= 2) cells(integral_constant<int, 5>(), integral_constant<int, 2>(), integral_constant<int, 2>());
          else if (ng <= 8) cells(integral_constant<int, 8>(), integral_constant<int, kNS1>(), integral_constant<int, kNSB>());
          else cells(integral_constant<int, kNSG>(), integral_constant<int, kNS1>(), integral_constant<int, kNSB>());
          __syncwarp();
          if (d + 1 <= n - 1) stage(d + 1);
        }
        // every tap moves one ring row down for the next diagonal
#pragma unroll
        for (int k = 0; k < kNSlot; k++) {   // add, wrap by unsigned min
          const unsigned x = (unsigned)xk[k] + 8u * (unsigned)RS;
          xk[k] = (int)min(x, x - 8u * wrap);
        }
      } else {
        const int a = warp - NWI;
        // ------------------------------------------------------------ diagonal d-1: staging row -> rings, qm1, au, qm
        if (d > BF_TURN + 1) {
          const int dd = d - 1, ncell = n - dd, pb = dd & 1;
          double *stg = STG + pb * 3 * RS, *tmpq = TMPQ + pb * RS;
          const double *ps = PS + pb * NWA * RS;
          const int row = (dd & (kRing - 1)) * RS;
          const int o0 = tri_off(n, dd), om = dd > BF_TURN + 1 ? tri_off(n, dd - 1) : 0;
          for (int cell = a * 32 + lane; cell < ncell; cell += NWA * 32) {
            const int i = cell + 1;
            double qms = 0.0;
#pragma unroll
            for (int w = 0; w < NWA; w++) qms += ps[w * RS + cell];
            const double g = stg[i], g1 = stg[RS + i], gb = stg[2 * RS + i], tq = tmpq[i];
            stg[i] = 0.0; stg[RS + i] = 0.0; stg[2 * RS + i] = 0.0; tmpq[i] = 0.0;   // only pairable cells are written
            QG[row + i] = g; Q1[row + i] = g1; QBB[row + i] = gb;
            double qm1 = tq, au = 0.0;
            if (dd > BF_TURN + 1) {
              qm1 = fma(QM1[om + i - 1], bu1, tq);                                   // (i, j-1) plus one unpaired base
              au = bu1 * (QM1[om + i] + AU[((dd - 1) & 1) * RS + i + 1]);            // stems starting right of i
            }
            const double qm = qms + au + qm1;
            QM[o0 + i - 1] = qm;
            QM1[o0 + i - 1] = qm1;
            if (qmg) { qmg[o0 + i - 1] = qm; qmg[tri_slot + o0 + i - 1] = qm1; }
            QMS[(dd & 3) * RS + i] = qms;
            AU[(dd & 1) * RS + i] = au;
          }
        }
        if (d <= n - 1) {
          const int ncell = n - d;
          // ------------------------------------------------------------ qm split: this warp's share of the split points, every cell
          double *ps = PS + (buf * NWA + a) * RS;
          constexpr int Q = NWA;
          for (int c0 = 0; c0 < ncell; c0 += 128) {
            int ii[4];
            double acc[4];
#pragma unroll
            for (int u = 0; u < 4; u++) { ii[u] = 8 * min(c0 + 32 * u + lane, ncell - 1); acc[u] = 0.0; }
            const bool many = c0 + 64 < ncell;
            int k = 5 + a;
            if (k <= d - 4) {
              const int oL = 8 * tri_off(n, k - 1), oR = 8 * (tri_off(n, d - k) + k);
              int dL = 8 * (Q * (n - k + 1) - Q * (Q - 1) / 2), dR = 8 * (-Q * (n - d + k + Q) + Q * (Q - 1) / 2 + Q);
              if (QMSM) {
                unsigned pL[4], pR[4];
#pragma unroll
                for (int u = 0; u < 4; u++) { pL[u] = sQM + (unsigned)(oL + ii[u]); pR[u] = sQM1 + (unsigned)(oR + ii[u]); }
                if (many) {
#pragma unroll 2
                  for (; k <= d - 4; k += Q) {
#pragma unroll
                    for (int u = 0; u < 4; u++) { acc[u] = fma(lds_f64(pL[u]), lds_f64(pR[u]), acc[u]); pL[u] += dL; pR[u] += dR; }
                    dL -= 8 * Q * Q; dR -= 8 * Q * Q;
                  }
                } else {
#pragma unroll 4
                  for (; k <= d - 4; k += Q) {
#pragma unroll
                    for (int u = 0; u < 2; u++) { acc[u] = fma(lds_f64(pL[u]), lds_f64(pR[u]), acc[u]); pL[u] += dL; pR[u] += dR; }
                    dL -= 8 * Q * Q; dR -= 8 * Q * Q;
                  }
                }
              } else {
                const char *pL[4], *pR[4];
#pragma unroll
                for (int u = 0; u < 4; u++) { pL[u] = reinterpret_cast<const char *>(QM) + oL + ii[u]; pR[u] = reinterpret_cast<const char *>(QM1) + oR + ii[u]; }
                if (many) {
#pragma unroll 2
                  for (; k <= d - 4; k += Q) {
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                      acc[u] = fma(*reinterpret_cast<const double *>(pL[u]), *reinterpret_cast<const double *>(pR[u]), acc[u]);
                      pL[u] += dL; pR[u] += dR;
                    }
                    dL -= 8 * Q * Q; dR -= 8 * Q * Q;
                  }
                } else {
#pragma unroll 4
                  for (; k <= d - 4; k += Q) {
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                      acc[u] = fma(*reinterpret_cast<const double *>(pL[u]), *reinterpret_cast<const double *>(pR[u]), acc[u]);
                      pL[u] += dL; pR[u] += dR;
                    }
                    dL -= 8 * Q * Q; dR -= 8 * Q * Q;
                  }
                }
              }
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
              const int cell = c0 + 32 * u + lane;
              if (cell < ncell) ps[cell] = acc[u];
            }
          }
        }
      }
      __syncthreads();
    }
  }
}

struct Mfe3Cfg { bool ok; int rs; size_t smem; };
// small: a batch that leaves SMs idle (a replica-exchange sub-step) -- one 16-warp CTA (12 tap + 4 auxiliary warps) per sequence with the
// whole shared memory of its SM; measured against the 16-warp round-1 kernels at B = 64 (profiles/r02_small_batch_fill3.txt): 36 nt 0.089 ->
// 0.076 ms, 100 nt 0.340 -> 0.257, 148 nt 0.678 -> 0.427, 200 nt 1.07 -> 0.66, as long as the fML table fits on chip (~230 nt)
Mfe3Cfg mfe3_cfg(int nmax, bool small, int fill3) {
  Mfe3Cfg c;
  c.ok = false;
  if (nmax < 1 || fill3 == 0) return c;
  c.rs = pick_rs(nmax, 32);
  // 8 warps: 6 tap + 2 auxiliary.  The fML table has to be on chip: with two auxiliary warps per CTA the split cannot hide L2
  // latency (measured: L = 120 7.8 ms per 4096 folds against 5.96 ms of the round-1 kernel, L = 200 33 against 16).  Three CTAs
  // per SM up to ~105 nt, two up to ~150 nt (112 KB); longer sequences stay on the round-1 kernels (bf_fill.cu).
  c.smem = small ? mfe3_plan(nmax, c.rs, 16, 4).total : mfe3_plan(nmax, c.rs, 8, 2).total;
  c.ok = c.smem <= (small ? kSmemBudget : 112 * 1024);
  return c;
}

struct Pf3Cfg { bool ok; int rs; bool qms, pair; size_t smem; int nw, nwi; };
Pf3Cfg pf3_cfg(int nmax, bool small, int fill3) {
  Pf3Cfg c;
  c.ok = false;
  if (nmax < 1 || fill3 == 0) return c;
  c.rs = pick_rs(nmax, 16);
  // One CTA of 16 warps (12 tap + 4 auxiliary) per SM with qm / qm1 on chip while they fit (~105 nt), through L2 beyond.  Measured
  // at L = 100 (4096 folds): 16 warps on chip 5.01 ms, 12 warps with paired cells 5.13, two CTAs of 8 warps (qm / qm1 in L2) 5.14;
  // at L = 120 / 150 the 16-warp CTA is ahead of the 8-warp pair by 20 / 30 % (profiles/r02_sweep_len.txt).
  // 16 warps with cells in pairs from 90 nt (L = 100: 4.90 ms per 4096 folds against 5.14 for two 8-warp CTAs); below, two or three
  // 8-warp CTAs per SM are ahead (L = 30 / 50 / 75: 0.60 / 1.26 / 2.79 ms against 0.88 / 1.71 / 3.13)
  // small batches (see mfe3_cfg): 16 warps at every length (B = 64: 36 nt 0.071 -> 0.058 ms, 100 nt 0.336 -> 0.227, 148 nt 0.776 -> 0.550,
  // 170 nt 1.00 -> 0.69, 176 nt 1.10 -> 0.72; the plan stops fitting the shared memory at ~178 nt, longer sequences stay on the round-1 kernel)
  // (beyond ~110 nt, qm / qm1 off chip, the split wants more auxiliary warps: paired cells with 10 tap + 6 auxiliary warps, B = 64 x 140 nt 0.51 -> 0.46 ms)
  c.nw = small || nmax >= 90 ? 16 : 8;
  c.pair = small ? nmax > 110 : nmax >= 90;
  c.nwi = c.nw == 8 ? 6 : (small && nmax > 110) ? 10 : 12;
  const int nwa = c.nw - c.nwi;
  const size_t with = pf3_plan(nmax, c.rs, c.nw, nwa, true).total;
  c.qms = c.nw == 16 && with <= kSmemBudget;
  c.smem = c.qms ? with : pf3_plan(nmax, c.rs, c.nw, nwa, false).total;
  // measured against the round-1 kernel (profiles/r02_sweep_len.txt): ahead up to 150 nt, level beyond
  c.ok = c.smem <= kSmemBudget && nmax <= (small ? 230 : 150);
  return c;
}

// The instantiations the rules return, each with its occupancy per stride (0 = not asked yet) and whether its shared-memory
// attribute is set: asked once per instance.
template <typename K>
struct Fill3Inst {
  K kern;
  int nw, nwi;
  bool qms, pair;
  int occ_cache[4096];
  bool attr_set;
};
using Mfe3K = void (*)(const BfParams *, BfBatchDev, int *, int *, size_t, int *, size_t, const uint32_t *, int, int *);
using Pf3K = void (*)(const BfParams *, BfBatchDev, double *, size_t, double *, size_t, double *, const int *, double *, const uint32_t *, int, int *);
Fill3Inst<Mfe3K> g_mfe3[] = {{bf_k_mfe_fill3<8, 6>, 8, 6, false, false, {}, false}, {bf_k_mfe_fill3<16, 12>, 16, 12, false, false, {}, false}};
#define BF_I(NW_, NWI_, QMSM_, PAIR_) {bf_k_pf_fill3<NW_, NWI_, QMSM_, PAIR_>, NW_, NWI_, QMSM_, PAIR_, {}, false}
Fill3Inst<Pf3K> g_pf3[] = {BF_I(8, 6, false, false), BF_I(16, 12, true, false), BF_I(16, 12, true, true), BF_I(16, 12, false, true),
                           BF_I(16, 10, false, true)};
#undef BF_I

template <typename K>
cudaError_t fill3_grid(Fill3Inst<K> &k, int stride, size_t smem, int B, int sms, int *grid) {
  cudaError_t e;
  if (!k.attr_set) {
    e = cudaFuncSetAttribute(k.kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget);
    if (e != cudaSuccess) return e;
    k.attr_set = true;
  }
  int occ_tmp = 0;
  int &occ = stride < 4096 ? k.occ_cache[stride] : occ_tmp;
  if (occ == 0) {
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k.kern, k.nw * 32, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) return cudaErrorInvalidConfiguration;
  }
  *grid = B < sms * occ ? B : sms * occ;
  return cudaSuccess;
}

}  // namespace

cudaError_t bf_fill3_mfe_plan(int nmax, int B, bool small, const BfOpts &o, int sms, BfPlan *p) {
  const Mfe3Cfg c = mfe3_cfg(nmax, small, o.fill3);
  if (!c.ok) return cudaSuccess;
  p->family = BF_FAM_TAP;
  p->key = small ? 1 : 0;
  p->smem = c.smem;
  p->ws = 2 * ((tri_size(nmax) * kEntWords + 7) / 8 * 8);   // ints per CTA: entries of every cell, two sequences
  return fill3_grid(g_mfe3[p->key], nmax, c.smem, B, sms, &p->grid);
}

cudaError_t bf_launch_mfe_fill3(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, int *ctri, int *ftri, int *ws, int *work_counter,
                                cudaStream_t st) {
  const int rs = pick_rs(b.stride, 32);
  const uint32_t *taps = nullptr;
  cudaError_t e = taps_device(rs, 32, &taps);
  if (e != cudaSuccess) return e;
  const Fill3Inst<Mfe3K> &k = g_mfe3[p.key];
  k.kern<<<p.grid, k.nw * 32, p.smem, st>>>(dP, b, ctri, ftri, bf_tri_slot(b.stride), ws, p.ws, taps, rs, work_counter);
  return cudaGetLastError();
}

cudaError_t bf_fill3_pf_plan(int nmax, int B, bool small, const BfOpts &o, int sms, BfPlan *p) {
  const Pf3Cfg c = pf3_cfg(nmax, small, o.fill3);
  if (!c.ok) return cudaSuccess;
  const int n = (int)(sizeof g_pf3 / sizeof g_pf3[0]);
  int key = 0;
  while (key < n && !(g_pf3[key].nw == c.nw && g_pf3[key].nwi == c.nwi && g_pf3[key].qms == c.qms && g_pf3[key].pair == c.pair)) key++;
  if (key == n) return cudaErrorInvalidValue;
  p->family = BF_FAM_TAP;
  p->key = key;
  p->smem = c.smem;
  const size_t tri_pad = (tri_size(nmax) + 7) / 8 * 8;
  p->ws = tri_pad * kEntD + 2 * tri_pad;   // doubles per CTA: entries of every cell, qm and qm1
  return fill3_grid(g_pf3[key], nmax, c.smem, B, sms, &p->grid);
}

cudaError_t bf_launch_pf_fill3(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, double *qbtri, double *ws, double *qmseq,
                               const int *mfe_for_scale, double *lnscale, int *work_counter, cudaStream_t st) {
  const int rs = pick_rs(b.stride, 16);
  const uint32_t *taps = nullptr;
  cudaError_t e = taps_device(rs, 16, &taps);
  if (e != cudaSuccess) return e;
  const Fill3Inst<Pf3K> &k = g_pf3[p.key];
  k.kern<<<p.grid, k.nw * 32, p.smem, st>>>(dP, b, qbtri, bf_tri_slot(b.stride), ws, p.ws, qmseq, mfe_for_scale, lnscale, taps, rs, work_counter);
  return cudaGetLastError();
}
