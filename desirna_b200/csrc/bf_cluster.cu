// bf_cluster.cu -- one thread-block CLUSTER per sequence: the fill kernels for long sequences and for small batches (sm_100a).
//
// Same recurrences and the same tables in HBM as bf_fill.cu / bf_fill3.cu (the path behind fc.mfe() / fc.pf(),
// utils/energy_scores.py:150-151 in the reference; recurrences SURVEY.md A.4-A.6), so bf_k_trace / bf_k_pf_ext / bf_k_pf_out2 read the
// result unchanged.  What is new is where the O(N^2) state lives while a sequence is folded.  A single CTA can keep the rings and the
// split operands (fML, or qm / qm1) on chip only up to ~150 nt; beyond that the round-1 kernels stream them through L2, and with
// 300-600 sequences in flight the L2 overflows (52 MB (MFE) / 98 MB (PF) of DRAM traffic per 400-nt fold against 0.6 / 3.5 MB of
// tables).  Here a cluster of C CTAs (2..16 SMs) folds ONE sequence, every table is partitioned over the cluster's shared memories,
// every READ is a local shared-memory read and everything that crosses CTAs is a fire-and-forget DSMEM STORE
// (st.shared::cluster) ordered by the one cluster barrier that ends a diagonal:
//
//  * cells are owned block-cyclically by their row: cell (i, j) belongs to the CTA  ((i-1) / BW) mod C.  The owner does the cell's
//    interior-loop taps (lanes over the 487 taps, bf_taps.cuh), hairpin, multiloop closing and its combine step.
//  * RINGS (the last 34 diagonals of the pair table in its three "inner term folded in" variants) are stored as WINDOWS: for each of
//    its blocks a CTA holds the block's BW columns and the 32 columns to their right -- exactly the columns the taps of its cells read.
//    A finished pair value is stored to every CTA whose windows contain its column (1 + 32 / BW stores per variant).
//  * the fML / qm split  min_u fML(i,u-1) + fML(u,j)  is partitioned by the SPLIT POSITION u: CTA (u mod C) holds column u-1 (left
//    operands) and row u (right operands) and computes, for every cell of the diagonal, the partial result over its own u; the partial
//    goes to the cell's owner.  A finished fML(i,j) is stored twice: to the CTA of column j+1 ... and to the CTA of row i.  Each CTA
//    holds 2/C of the table, the work is balanced exactly, and no operand is ever read remotely.
//  * phase d (one cluster barrier per diagonal): taps of diagonal d (read diagonals <= d-2) | combine of diagonal d-1 | split partials
//    of diagonal d (read diagonals <= d-5).  All warps take tap cells first, then split items.
#include "bf_kernels.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "bf_device.cuh"

#include "bf_taps.cuh"

namespace {

constexpr int kDepth = 35;     // ring rows: row d is cleared in phase d-2 (behind the barrier's arrive), written in phase d, read in phases d+2 .. d+32
constexpr int kEntW = 20;      // words per cell entry (layout of bf_fill3.cu; word 19 = the cell's window column)
constexpr int kPMax = 2;       // a chunk's split positions may be dealt to two warps
constexpr int kNWcl = 16;      // warps per CTA (one CTA per SM)
constexpr int kNoWrite = -2147483647 - 1;   // staging slot without a value
constexpr int kNTcl = 8;       // of them tap warps; the others combine, split and clear

__device__ __forceinline__ unsigned cl_rank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned cl_index() { unsigned r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned cl_map(unsigned saddr, unsigned rank) {
  unsigned r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cl_st_s32(unsigned caddr, int v) { asm volatile("st.shared::cluster.s32 [%0], %1;" ::"r"(caddr), "r"(v) : "memory"); }
__device__ __forceinline__ void cl_st_f64(unsigned caddr, double v) { asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(caddr), "d"(v) : "memory"); }
__device__ __forceinline__ void cl_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cl_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cl_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ int lds_i(unsigned addr) {
  int v;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ double lds_d(unsigned addr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}

// geometry of one launch (host-computed, passed by value)
struct ClGeom {
  int C, logC, BW, logBW, WIN, NLB, K;   // cluster size, block width, window = BW + 32, local blocks per CTA, stores per ring value
  int RS;                                // ring row stride (elements): NLB windows, padded to a residue the tap packing accepts
  int ncl;                               // own cell slots per diagonal = NLB * BW
  int colcap, rowcap;                    // elements of the column / row stores of one CTA
  int lcap;                              // entries of one warp's cell list
};

// split-operand stores of rank r: column of split position m = q C + r starts at  C q(q-1)/2 + q r  (m slots: rows 1 .. m-5 used),
// row m starts at  q (n+1-r) - C q(q-1)/2  (n+1-m slots: columns m+4 .. n used, index j-m-4)
__host__ __device__ __forceinline__ int col_base(int C, int r, int q) { return C * (q * (q - 1) / 2) + q * r; }
__host__ __device__ __forceinline__ int row_base(int C, int r, int q, int n1) { return q * (n1 - r) - C * (q * (q - 1) / 2); }

struct MfeClPlan {
  unsigned o_ring, o_dml, o_fp, o_tmpe, o_cst, o_col, o_row, o_spart, o_np, o_S, o_SP, o_cl, o_pp, total;
};
MfeClPlan mfe_cl_plan(int nmax, const ClGeom &g) {
  MfeClPlan p;
  size_t o = 0;
  p.o_ring = o; o += ((size_t)3 * kDepth * g.RS + g.RS) * 4;
  p.o_dml = o; o += (size_t)4 * g.RS * 4;
  p.o_fp = o; o += (size_t)2 * g.RS * 4;
  p.o_tmpe = o; o += (size_t)2 * g.ncl * 4;
  p.o_cst = o; o += (size_t)2 * g.ncl * 4;   // pair energies on their way to the HBM table (written there one phase later)
  p.o_col = o; o += (size_t)g.colcap * 4;
  p.o_row = o; o += (size_t)g.rowcap * 4;
  p.o_spart = o; o += (size_t)2 * g.C * kPMax * g.ncl * 4;
  p.o_np = o; o += (size_t)((nmax + 4) / 4 * 4) * 2;
  p.o_S = o; o += (size_t)(nmax + 2 + 15) / 16 * 16;
  p.o_SP = o; o += (size_t)(nmax + 2 + 15) / 16 * 16;
  o = (o + 15) / 16 * 16;
  p.o_cl = o; o += (size_t)kNTcl * g.lcap * kEntW * 4;
  p.o_pp = o; o += (size_t)kNWcl * ((g.ncl + 7) / 8 * 8) * 2;
  p.total = (unsigned)((o + 15) / 16 * 16);
  return p;
}

// =====================================================================================================
//                                           MFE fill, cluster per sequence
// =====================================================================================================
template <int NW, int NT>
__global__ void __launch_bounds__(NW * 32, 1) bf_k_mfe_cl(const BfParams *__restrict__ P, BfBatchDev b, int *ctri, int *ftri, size_t tri_slot,
                                                          int *ent_ws, size_t ent_slot, const uint32_t *__restrict__ taps, MfeClPlan pl, ClGeom g,
                                                          int *work_counter) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq;
  __shared__ unsigned char s_meta[96];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(BF_FULL, tid >> 5, 0);
  const int r = (int)cl_rank(), C = g.C, logC = g.logC, BW = g.BW, logBW = g.logBW, WIN = g.WIN, RS = g.RS, ncl = g.ncl;
  int *RG = reinterpret_cast<int *>(dyn + pl.o_ring);
  int *DML = reinterpret_cast<int *>(dyn + pl.o_dml);
  int *FP = reinterpret_cast<int *>(dyn + pl.o_fp);
  int *TMPE = reinterpret_cast<int *>(dyn + pl.o_tmpe);
  int *CST = reinterpret_cast<int *>(dyn + pl.o_cst);
  int *COL = reinterpret_cast<int *>(dyn + pl.o_col);
  int *ROW = reinterpret_cast<int *>(dyn + pl.o_row);
  int *SPART = reinterpret_cast<int *>(dyn + pl.o_spart);
  unsigned short *NP = reinterpret_cast<unsigned short *>(dyn + pl.o_np);
  uint8_t *S = dyn + pl.o_S, *SP = dyn + pl.o_SP;
  const BfSmallI &T = P->si;
  if (tid < 96) s_meta[tid] = reinterpret_cast<const unsigned char *>(taps + kNSlot * 32)[tid];   // TapMeta: slots needed by loop size
  const int MLbase = T.MLbase;
  int *ent = ent_ws + (size_t)cl_index() * ent_slot + (size_t)r * (ent_slot / C);   // this CTA's entries: diagonal d at (d-4) ncl
  const int tauE = T.TerminalAU;
  const unsigned sRG = (unsigned)__cvta_generic_to_shared(RG);
  const unsigned sFP = (unsigned)__cvta_generic_to_shared(FP), sDML = (unsigned)__cvta_generic_to_shared(DML);
  const unsigned sCOL = (unsigned)__cvta_generic_to_shared(COL), sROW = (unsigned)__cvta_generic_to_shared(ROW);
  const unsigned sSPART = (unsigned)__cvta_generic_to_shared(SPART);
  const unsigned wrap = (unsigned)(kDepth * RS);

  // this lane's taps: penalties for the whole launch, ring offsets (bytes) re-based for every sequence
  int pen[kNSlot], xk[kNSlot];
#pragma unroll
  for (int k = 0; k < kNSlot; k++) {
    const uint32_t tp = __ldg(taps + k * 32 + lane);
    const int s = tp & 255, u1 = (tp >> 8) & 255;
    int v = BF_INF;
    if (tp >> 16) {
      if (k < kNSG) v = T.interior[s] + min(T.ninio_max, abs(s - 2 * u1) * T.ninio_m);
      else if (k < kNSG + kNS1) v = T.interior[s] + min(T.ninio_max, (s - 2) * T.ninio_m);
      else if (k < kNSG + kNS1 + kNSB) v = T.bulge[s];
      else v = 0;
    }
    pen[k] = v;
    xk[k] = 0;
  }
  // store lanes of a finished pair value: lane -> (ring variant, destination window); then the fML candidate and the HBM table
  // cells are taken two at a time: lanes 0..15 store for the first cell, lanes 16..31 for the second
  const int nst = 3 * g.K;
  const int l16 = lane & 15, hi = lane >> 4;
  const int st_kind = l16 % 3, st_k = l16 / 3;
  const int ltl = l16 < nst ? 5 + st_kind : 8;
  const int lsp = 9 + min(lane, 9);
  int *wl = reinterpret_cast<int *>(dyn + pl.o_cl) + (size_t)warp * g.lcap * kEntW;
  unsigned short *cl_pp = reinterpret_cast<unsigned short *>(dyn + pl.o_pp) + (size_t)warp * ((ncl + 7) / 8 * 8);

  for (;;) {
    // ---- next sequence of this cluster (rank 0 draws, everybody reads it through DSMEM after the barrier)
    if (r == 0 && tid == 0) s_seq = atomicAdd(work_counter, 1);
    cl_sync();
    int sq;
    {
      const unsigned a0 = cl_map((unsigned)__cvta_generic_to_shared(&s_seq), 0);
      asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(sq) : "r"(a0));
    }
    cl_sync();   // everybody has read it before rank 0 draws again
    if (sq >= b.B) break;
    const int n = __shfl_sync(BF_FULL, b.len[sq], 0);
    {
      const char *src = b.seq + (size_t)sq * b.stride;
      const uint8_t *np = b.nopair ? b.nopair + (size_t)sq * b.stride : nullptr;
      for (int k = tid; k <= n + 1; k += blockDim.x) {
        const int code = (k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0;
        S[k] = (uint8_t)code;
        SP[k] = (uint8_t)((np && k >= 1 && k <= n && np[k - 1]) ? 0 : code);
      }
    }
    for (int k = tid; k < 3 * kDepth * RS + RS; k += blockDim.x) RG[k] = BF_INF;
    for (int k = tid; k < 4 * RS; k += blockDim.x) DML[k] = BF_INF;
    for (int k = tid; k < 2 * RS; k += blockDim.x) FP[k] = BF_INF;
    for (int k = tid; k < 2 * ncl; k += blockDim.x) { TMPE[k] = BF_INF; CST[k] = kNoWrite; }
    int *cg_out = ctri + (size_t)sq * tri_slot;
    int *fg_out = ftri + (size_t)sq * tri_slot;
    __syncthreads();
    // ---- pre-pass: per-cell constants of this CTA's pairable cells, compacted per diagonal (entry layout of bf_fill3.cu)
    for (int d = BF_TURN + 1 + warp; d <= n - 1; d += NW) {
      int count = 0;
      const int od = tri_off(n, d);
      for (int base = 0; base < ncl; base += 32) {
        const int slot = base + lane;
        const int lb = slot >> logBW, o = slot & (BW - 1);
        const int i = (((lb << logC) + r) << logBW) + 1 + o;
        const bool in = slot < ncl && i <= n - d;
        const int t = in ? bf_ptype_bases(SP[i], SP[i + d]) : 0;
        const unsigned mk = __ballot_sync(BF_FULL, t != 0);
        if (in && !t) cg_out[od + i - 1] = BF_INF;
        if (t) cl_pp[count + __popc(mk & ((1u << lane) - 1))] = (unsigned short)i;
        count += __popc(mk);
      }
      if (lane == 0) NP[d] = (unsigned short)count;
      __syncwarp();
      for (int c = lane; c < count; c += 32) {
        const int i = cl_pp[c], j = i + d;
        const int t = bf_ptype_bases(SP[i], SP[j]);
        const int si1 = S[i + 1], sj1 = S[j - 1], sim = S[i - 1], sjp = S[j + 1], tr = bf_rtype(t);
        int4 *dst = reinterpret_cast<int4 *>(ent + ((size_t)(d - 4) * ncl + c) * kEntW);
        dst[0] = make_int4(i, T.mmI[t][si1][sj1], T.mm1nI[t][si1][sj1], bf_e_hairpin(P, T, S, i, j, t));
        dst[1] = make_int4(T.MLclosing + bf_e_mlstem(T, tr, sj1, si1), T.mmI[tr][sjp][sim], T.mm1nI[tr][sjp][sim], t > 2 ? tauE : 0);
        int w[12];
        w[0] = (i > 1 && j < n) ? bf_e_mlstem(T, t, sim, sjp) : BF_INF;
#pragma unroll
        for (int k = 0; k < 9; k++) {
          const int u1 = special_u1(k), u2 = special_u2(k);
          const bool ok = (j - 1 - u2) - (i + 1 + u1) > BF_TURN;
          const int p = ok ? i + 1 + u1 : i + 1, q = ok ? j - 1 - u2 : j - 1;
          const int t2 = ok ? bf_ptype_bases(SP[p], SP[q]) : 0;
          const int e = bf_e_intloop(P, T, u1, u2, t, bf_rtype(t2), si1, sj1, S[p - 1], S[q + 1]);
          w[1 + k] = t2 ? e - (t2 > 2 ? tauE : 0) : 0;
        }
        const int bx = (i - 1) >> logBW;
        w[10] = BF_INF;
        w[11] = (bx >> logC) * WIN + ((i - 1) & (BW - 1));   // window column of the cell
        dst[2] = make_int4(w[0], w[1], w[2], w[3]);
        dst[3] = make_int4(w[4], w[5], w[6], w[7]);
        dst[4] = make_int4(w[8], w[9], w[10], w[11]);
      }
      __syncwarp();
    }
#pragma unroll
    for (int k = 0; k < kNSlot; k++) {
      const uint32_t tp = __ldg(taps + k * 32 + lane);
      const int s = tp & 255, u1 = (tp >> 8) & 255;
      const int row = ((BF_TURN + 1 - 2 - s) % kDepth + kDepth) % kDepth;
      xk[k] = 4 * (row * RS + 1 + u1);   // bytes from the origin of the slot's ring variant
    }
    __threadfence_block();
    cl_sync();   // every CTA of the cluster has reset its tables: remote stores may arrive from here on
    const int st_m5 = lane / 5, st_q5 = lane - 5 * (lane / 5);
    auto stage = [&](int dn) {
      const int mine = ((int)NP[dn] - warp + NT - 1) / NT;
      const char *src = reinterpret_cast<const char *>(ent + ((size_t)(dn - 4) * ncl + warp) * kEntW);
      const unsigned dst = (unsigned)__cvta_generic_to_shared(wl);
      // 16-byte pieces: lane -> (entry lane / 5, piece lane % 5), six entries per pass
      for (int m = st_m5; m < mine && lane < 30; m += 6)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + (unsigned)(m * kEntW * 4 + st_q5 * 16)),
                     "l"(src + (size_t)m * NT * kEntW * 4 + st_q5 * 16)
                     : "memory");
    };
    if (warp < NT && n - 1 >= BF_TURN + 1) stage(BF_TURN + 1);

    auto mfe_flush = [&](int dc, int df) {   // one warp
      for (int slot = lane; slot < ncl; slot += 32) {
        const int lb = slot >> logBW, o = slot & (BW - 1);
        const int i = ((((lb << logC) + r) << logBW)) + 1 + o;
        if (dc >= BF_TURN + 1 && dc <= n - 1) {
          const int v = CST[(dc & 1) * ncl + slot];
          if (v != kNoWrite) { cg_out[tri_off(n, dc) + i - 1] = v; CST[(dc & 1) * ncl + slot] = kNoWrite; }
        }
        if (df >= BF_TURN + 1 && df <= n - 1 && i <= n - df) fg_out[tri_off(n, df) + i - 1] = FP[(df & 1) * RS + lb * WIN + o];
      }
    };
    int rowd = (BF_TURN + 1) % kDepth;   // ring row of diagonal d
    for (int d = BF_TURN + 1; d <= n; d++, rowd = rowd + 1 == kDepth ? 0 : rowd + 1) {
      const int buf = d & 1;
      // ------------------------------------------------------------ taps: c(i,j) of this CTA's pairable cells of diagonal d
      if (warp < NT && d <= n - 1) {
        const int np = NP[d];
        const unsigned sdml = sDML + 4u * (unsigned)(((d - 2) & 3) * RS + 1);
        // lane's store base: ring variant st_kind, row d, window st_k
        const unsigned sbase = sRG + 4u * (unsigned)((st_kind * kDepth + rowd) * RS + st_k * BW);
        const int smax = min(BF_MAXLOOP, d - 6);
        const int mi = smax + 1 < 0 ? 0 : smax + 1;
        const int ng = s_meta[mi], n1 = s_meta[32 + mi], nb = s_meta[64 + mi];
        auto cells = [&](auto cg_, auto c1_, auto cb_) {
          constexpr int G = decltype(cg_)::value, O = decltype(c1_)::value, Bn = decltype(cb_)::value;
          asm volatile("cp.async.wait_all;" ::: "memory");
          __syncwarp();
          const int *p = wl;
          for (int c = warp; c < np; c += 2 * NT, p += 2 * kEntW) {
            const bool hasB = c + NT < np;
            const int *pA = p, *pB = hasB ? p + kEntW : p;   // no second cell: the first once more, its stores dropped
            const int4 ea = *reinterpret_cast<const int4 *>(pA), eb = *reinterpret_cast<const int4 *>(pB);
            const int mlcA = pA[4], tauA = pA[7], espA = pA[lsp], mlcB = pB[4], tauB = pB[7], espB = pB[lsp];
            const unsigned lcA = 4u * (unsigned)__reduce_min_sync(BF_FULL, pA[19]), lcB = 4u * (unsigned)__reduce_min_sync(BF_FULL, pB[19]);
            const unsigned uA = sRG + lcA, uB = sRG + lcB;
            int gA = BF_INF, gB = BF_INF, oA = BF_INF, oB = BF_INF, bA = BF_INF, bB = BF_INF;
#pragma unroll
            for (int k = 0; k < G; k++) { gA = min(gA, lds_i(uA + xk[k]) + pen[k]); gB = min(gB, lds_i(uB + xk[k]) + pen[k]); }
#pragma unroll
            for (int k = 0; k < O; k++) {
              oA = min(oA, lds_i(uA + 4u * wrap + xk[kNSG + k]) + pen[kNSG + k]);
              oB = min(oB, lds_i(uB + 4u * wrap + xk[kNSG + k]) + pen[kNSG + k]);
            }
#pragma unroll
            for (int k = 0; k < Bn; k++) {
              bA = min(bA, lds_i(uA + 8u * wrap + xk[kNSG + kNS1 + k]) + pen[kNSG + kNS1 + k]);
              bB = min(bB, lds_i(uB + 8u * wrap + xk[kNSG + kNS1 + k]) + pen[kNSG + kNS1 + k]);
            }
            const int vsA = lds_i(uA + 8u * wrap + xk[kNSlot - 1]) + espA, vsB = lds_i(uB + 8u * wrap + xk[kNSlot - 1]) + espB;
            int totA = min(min(gA + ea.y, oA + ea.z), min(bA + tauA, vsA)), totB = min(min(gB + eb.y, oB + eb.z), min(bB + tauB, vsB));
            totA = __reduce_min_sync(BF_FULL, totA);
            totB = __reduce_min_sync(BF_FULL, totB);
            // from here on each half-warp finishes its own cell
            const int *pm = hi ? pB : pA;
            int tot = hi ? totB : totA;
            const int4 em = hi ? eb : ea;
            tot = min(tot, em.w);                                             // hairpin
            const int dm = lds_i(sdml + (hi ? lcB : lcA));                    // split minimum of (i+1, j-1)
            if (dm < kInfThr) tot = min(tot, dm + (hi ? mlcB : mlcA));        // multiloop closed by (i,j)
            const bool fin = tot < kInfThr;
            const int etl = pm[ltl];
            const int v = (fin && etl < kInfThr) ? tot + etl : BF_INF;
            const int i = em.x, bx = (i - 1) >> logBW, o = (i - 1) & (BW - 1);
            if (!hi || hasB) {
              if (l16 < nst) {
                const int bxk = bx - st_k;
                if (bxk >= 0) cl_st_s32(cl_map(sbase + 4u * (unsigned)((bxk >> logC) * WIN + o), (unsigned)(bxk & (C - 1))), v);
              } else if (l16 == nst) {
                TMPE[buf * ncl + ((bx >> logC) << logBW) + o] = v;
              } else if (l16 == nst + 1) {
                CST[buf * ncl + ((bx >> logC) << logBW) + o] = fin ? tot : BF_INF;
              }
            }
          }
        };
        using std::integral_constant;
        if (ng <= 2 && n1 <= 1 && nb <= 1) cells(integral_constant<int, 2>(), integral_constant<int, 1>(), integral_constant<int, 1>());
        else if (ng <= 5 && n1 <= 2 && nb <= 2) cells(integral_constant<int, 5>(), integral_constant<int, 2>(), integral_constant<int, 2>());
        else if (ng <= 8) cells(integral_constant<int, 8>(), integral_constant<int, kNS1>(), integral_constant<int, kNSB>());
        else cells(integral_constant<int, kNSG>(), integral_constant<int, kNS1>(), integral_constant<int, kNSB>());
        __syncwarp();
      }
      // ------------------------------------------------------------ combine of diagonal d-1: this CTA's cells (dealt from the last warp down)
      constexpr int NWS = NW - NT;
      const int aw = warp - NT;
      const int ncomb = (ncl + 31) >> 5;
      if (d > BF_TURN + 1 && aw >= 0)
       for (int cp = NWS - 2 - aw; cp >= 0 && cp < ncomb; cp += NWS - 1) {   // from the last-but-one warp down
        const int dd = d - 1, pb = dd & 1;
        const int slot = cp * 32 + lane;
        const int lb = slot >> logBW, o = slot & (BW - 1);
        const int bx = (lb << logC) + r;
        const int i = (bx << logBW) + 1 + o;
        if (slot < ncl && i <= n - dd) {
          const int j = i + dd, lc = lb * WIN + o;
          const int nchp = (n - dd + 31) >> 5;
          const int Pp = (2 * nchp <= NWS) ? kPMax : 1;
          int sp = BF_INF, sp1 = BF_INF;
          {
            const int *sb = SPART + (size_t)pb * C * kPMax * ncl + slot;   // [rank][part] rows of ncl
            if (Pp == 2) {
#pragma unroll 2
              for (int rr = 0; rr < C; rr += 2) {
                const int a = sb[(2 * rr) * ncl], bq = sb[(2 * rr + 1) * ncl], cq = sb[(2 * rr + 2) * ncl], e = sb[(2 * rr + 3) * ncl];
                sp = min(sp, min(a, bq)); sp1 = min(sp1, min(cq, e));
              }
            } else {
#pragma unroll 2
              for (int rr = 0; rr < C; rr += 2) { sp = min(sp, sb[(2 * rr) * ncl]); sp1 = min(sp1, sb[(2 * rr + 2) * ncl]); }
            }
            sp = min(sp, sp1);
          }
          if (sp >= kInfThr) sp = BF_INF;
          const int te = TMPE[pb * ncl + slot];
          TMPE[pb * ncl + slot] = BF_INF;
          int m = min(sp, te);
          if (dd > BF_TURN + 1) m = min(m, min(FP[((dd - 1) & 1) * RS + lc], FP[((dd - 1) & 1) * RS + lc + 1]) + MLbase);
          if (m >= kInfThr) m = BF_INF;
          FP[(dd & 1) * RS + lc] = m;
          DML[(dd & 3) * RS + lc] = sp;
          if (o == 0 && bx >= 1) {   // first cell of a block: also the last column of the previous block's window
            const unsigned rk = (unsigned)((bx - 1) & (C - 1));
            const int lcp = ((bx - 1) >> logC) * WIN + BW;
            cl_st_s32(cl_map(sFP + 4u * (unsigned)((dd & 1) * RS + lcp), rk), m);
            cl_st_s32(cl_map(sDML + 4u * (unsigned)((dd & 3) * RS + lcp), rk), sp);
          }
          // split operands: column j (left operand of split position j+1), row i (right operand of split position i)
          {
            const int mcol = j + 1;
            if (mcol <= n) cl_st_s32(cl_map(sCOL + 4u * (unsigned)(col_base(C, mcol & (C - 1), mcol >> logC) + i - 1), (unsigned)(mcol & (C - 1))), m);
            cl_st_s32(cl_map(sROW + 4u * (unsigned)(row_base(C, i & (C - 1), i >> logC, n + 1) + dd - 4), (unsigned)(i & (C - 1))), m);
          }
        }
      }
      // ------------------------------------------------------------ HBM tables: the last warp writes what the previous phases left in
      // shared memory (c of diagonal d-1, fML of diagonal d-2), so that no thread has a global store in flight when it reaches the
      // cluster barrier's release
      if (aw == NWS - 1) mfe_flush(d - 1, d - 2);
      // ------------------------------------------------------------ split partials of diagonal d over this CTA's split positions
      if (aw >= 0 && d <= n - 1) {
        const int ncell = n - d, nch = (ncell + 31) >> 5;
        const int Pp = (2 * nch <= NWS) ? kPMax : 1;
        const int nitems = nch * Pp;
        for (int it = aw; it < nitems; it += NWS) {   // dealt from the first auxiliary warp up: the last ones combine and write
          const int ch = Pp == 2 ? it >> 1 : it, pp = Pp == 2 ? it & 1 : 0;
          const int i0 = 32 * ch + 1, i = i0 + lane;
          const int ilast = min(i0 + 31, ncell);
          const int lo = i0 + 5, hi = ilast + d - 4;
          const int mfirst = lo + ((r - lo) & (C - 1));
          const int cnt = mfirst > hi ? 0 : ((hi - mfirst) >> logC) + 1;
          const int per = Pp == 2 ? (cnt + 1) >> 1 : cnt;
          const int t0 = pp * per, t1 = min(cnt, t0 + per);
          int acc = BF_INF;
          if (t0 < t1 && d >= 9) {
            int m = mfirst + (t0 << logC);
            int q = m >> logC;
            unsigned aL = sCOL + 4u * (unsigned)(col_base(C, r, q) + i - 1);
            unsigned aR = sROW + 4u * (unsigned)(row_base(C, r, q, n + 1) + i + d - m - 4);
            // lane's cell is a candidate of split position m when  m-d+4 <= i <= m-5  (and the cell exists)
            const int iv = i <= ncell ? i : -100000;
#pragma unroll 4
            for (int t = t0; t < t1; t++) {
              if ((unsigned)(iv - (m - d + 4)) <= (unsigned)(d - 9)) acc = min(acc, lds_i(aL) + lds_i(aR));
              aL += 4u * (unsigned)m;                       // next column of this rank: m slots further
              aR += 4u * (unsigned)(n + 1 - m - C);         // next row: (n+1-m) slots further, and the index j-m-4 drops by C
              m += C;
            }
          }
          if (i <= ncell) {
            const int bx = (i - 1) >> logBW, o = (i - 1) & (BW - 1);
            const int slot = ((bx >> logC) << logBW) + o;
            cl_st_s32(cl_map(sSPART + 4u * (unsigned)(((buf * C + r) * kPMax + pp) * ncl + slot), (unsigned)(bx & (C - 1))), acc);
          }
        }
      }
      cl_arrive();
      // ---- between arrive and wait: work that nobody else sees
      if (warp < NT) {
        if (d + 1 <= n - 1) stage(d + 1);   // entries of this warp's cells of the next diagonal
#pragma unroll
        for (int k = 0; k < kNSlot; k++) {   // every tap one ring row down: add, wrap by unsigned min
          const unsigned x = (unsigned)xk[k] + 4u * (unsigned)RS;
          xk[k] = (int)min(x, x - 4u * wrap);
        }
      } else {   // clear ring row d+2: last read in phase d-1, written from phase d+2 on
        const int row = rowd + 2 >= kDepth ? rowd + 2 - kDepth : rowd + 2;
        for (int x = tid - NT * 32; x < RS; x += (NW - NT) * 32) {
          RG[row * RS + x] = BF_INF; RG[(kDepth + row) * RS + x] = BF_INF; RG[(2 * kDepth + row) * RS + x] = BF_INF;
        }
      }
      cl_wait();
    }
    if (warp == NW - 1) mfe_flush(n, n - 1);   // fML of the last diagonal
  }
  cl_sync();
}

// =====================================================================================================
//                              partition function (inside) fill, cluster per sequence
// =====================================================================================================
// Same organisation with sums of Boltzmann weights (fp64):
//   qb(i,j)  = hairpin + sum over the taps (ring value x weight) + qms(i+1,j-1) x closing                 -- owner, phase d
//   qm1(i,j) = qm1(i,j-1) bu + qb(i,j) xMLstem;  au(i,j) = bu (qm1(i+1,j) + au(i+1,j));  qm = qms + au + qm1   -- owner, phase d+1
//   qms(i,j) = sum_u qm(i,u-1) qm1(u,j): partial sums by split position on CTA (u mod C), added by the owner in a fixed order
// Entry of a pairable cell: the 20 doubles of bf_fill3.cu, word 19 = the cell's window column.
constexpr int kEntDc = 20;

struct PfClPlan {
  unsigned o_ring, o_qms, o_q1p, o_au, o_tmpq, o_qst, o_col, o_row, o_spart, o_scl, o_cl, o_np, o_pp, o_S, total;
};
PfClPlan pf_cl_plan(int nmax, const ClGeom &g) {
  PfClPlan p;
  size_t o = 0;
  p.o_ring = o; o += ((size_t)3 * kDepth * g.RS + g.RS) * 8;
  p.o_qms = o; o += (size_t)4 * g.RS * 8;
  p.o_q1p = o; o += (size_t)2 * g.RS * 8;
  p.o_au = o; o += (size_t)2 * g.RS * 8;
  p.o_tmpq = o; o += (size_t)2 * g.ncl * 8;
  p.o_qst = o; o += (size_t)2 * g.ncl * 8;
  p.o_col = o; o += (size_t)g.colcap * 8;
  p.o_row = o; o += (size_t)g.rowcap * 8;
  p.o_spart = o; o += (size_t)2 * g.C * kPMax * g.ncl * 8;
  p.o_scl = o; o += (size_t)(nmax + 8 > 40 ? nmax + 8 : 40) * 8;
  o = (o + 15) / 16 * 16;
  p.o_cl = o; o += (size_t)kNTcl * g.lcap * kEntDc * 8;
  p.o_np = o; o += (size_t)((nmax + 4) / 4 * 4) * 2;
  p.o_pp = o; o += (size_t)kNWcl * ((g.ncl + 7) / 8 * 8) * 2;
  p.o_S = o; o += (size_t)(nmax + 2 + 15) / 16 * 16;
  p.total = (unsigned)((o + 15) / 16 * 16);
  return p;
}

template <int NW, int NT>
__global__ void __launch_bounds__(NW * 32, 1) bf_k_pf_cl(const BfParams *__restrict__ P, BfBatchDev b, double *qbtri, size_t tri_slot, double *ent_ws,
                                                         size_t ent_slot, double *qm_perseq, const int *__restrict__ mfe_for_scale,
                                                         double *lnscale_out, const uint32_t *__restrict__ taps, PfClPlan pl, ClGeom g,
                                                         int *work_counter) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq;
  __shared__ unsigned char s_meta[96];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(BF_FULL, tid >> 5, 0);
  const int r = (int)cl_rank(), C = g.C, logC = g.logC, BW = g.BW, logBW = g.logBW, WIN = g.WIN, RS = g.RS, ncl = g.ncl;
  double *RG = reinterpret_cast<double *>(dyn + pl.o_ring);
  double *QMS = reinterpret_cast<double *>(dyn + pl.o_qms);
  double *Q1P = reinterpret_cast<double *>(dyn + pl.o_q1p);
  double *AU = reinterpret_cast<double *>(dyn + pl.o_au);
  double *TMPQ = reinterpret_cast<double *>(dyn + pl.o_tmpq);
  double *QST = reinterpret_cast<double *>(dyn + pl.o_qst);
  double *COL = reinterpret_cast<double *>(dyn + pl.o_col);
  double *ROW = reinterpret_cast<double *>(dyn + pl.o_row);
  double *SPART = reinterpret_cast<double *>(dyn + pl.o_spart);
  double *scl = reinterpret_cast<double *>(dyn + pl.o_scl);
  unsigned short *NP = reinterpret_cast<unsigned short *>(dyn + pl.o_np);
  uint8_t *S = dyn + pl.o_S;
  const BfSmallD &T = P->sd;
  if (tid < 96) s_meta[tid] = reinterpret_cast<const unsigned char *>(taps + kNSlot * 32)[tid];
  double *ent = ent_ws + (size_t)cl_index() * ent_slot + (size_t)r * (ent_slot / C);
  const double xtau = T.x_TerminalAU, inv_tau = 1.0 / xtau;
  const unsigned sRG = (unsigned)__cvta_generic_to_shared(RG);
  const unsigned sQMS = (unsigned)__cvta_generic_to_shared(QMS), sQ1P = (unsigned)__cvta_generic_to_shared(Q1P);
  const unsigned sAU = (unsigned)__cvta_generic_to_shared(AU);
  const unsigned sCOL = (unsigned)__cvta_generic_to_shared(COL), sROW = (unsigned)__cvta_generic_to_shared(ROW);
  const unsigned sSPART = (unsigned)__cvta_generic_to_shared(SPART);
  const unsigned wrap = (unsigned)(kDepth * RS);
  double wk[kNSlot - 1];
  int xk[kNSlot];
  const int nst = 3 * g.K;
  const int st_kind = lane % 3, st_k = lane / 3;
  const int ltl = lane < nst ? 5 + st_kind : 8;
  const int lsp = 9 + min(lane, 9);
  double *wl = reinterpret_cast<double *>(dyn + pl.o_cl) + (size_t)warp * g.lcap * kEntDc;
  unsigned short *cl_pp = reinterpret_cast<unsigned short *>(dyn + pl.o_pp) + (size_t)warp * ((ncl + 7) / 8 * 8);

  for (;;) {
    if (r == 0 && tid == 0) s_seq = atomicAdd(work_counter, 1);
    cl_sync();
    int sq;
    {
      const unsigned a0 = cl_map((unsigned)__cvta_generic_to_shared(&s_seq), 0);
      asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(sq) : "r"(a0));
    }
    cl_sync();
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
    if (r == 0 && tid == 0 && lnscale_out) lnscale_out[sq] = lns;
    const double bu1 = exp(log(T.x_MLbase) - lns);
    const double xclose = T.x_MLclosing * exp(-2.0 * lns);
    for (int k = tid; k < 3 * kDepth * RS + RS; k += blockDim.x) RG[k] = 0.0;
    for (int k = tid; k < 4 * RS; k += blockDim.x) QMS[k] = 0.0;
    for (int k = tid; k < 2 * RS; k += blockDim.x) { Q1P[k] = 0.0; AU[k] = 0.0; }
    for (int k = tid; k < 2 * ncl; k += blockDim.x) { TMPQ[k] = 0.0; QST[k] = -1.0; }
    double *qb_out = qbtri + (size_t)sq * tri_slot;
    double *qmg = qm_perseq ? qm_perseq + (size_t)sq * 2 * tri_slot : nullptr;
    __syncthreads();
    if (warp < NT) {
#pragma unroll
      for (int k = 0; k < kNSlot; k++) {
        const uint32_t tp = __ldg(taps + k * 32 + lane);
        const int s = tp & 255, u1 = (tp >> 8) & 255;
        const int row = ((BF_TURN + 1 - 2 - s) % kDepth + kDepth) % kDepth;
        xk[k] = 8 * (row * RS + 1 + u1);
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
    // ---- pre-pass: per-cell constants of this CTA's pairable cells
    for (int d = BF_TURN + 1 + warp; d <= n - 1; d += NW) {
      int count = 0;
      const int od = tri_off(n, d);
      for (int base = 0; base < ncl; base += 32) {
        const int slot = base + lane;
        const int lb = slot >> logBW, o = slot & (BW - 1);
        const int i = (((lb << logC) + r) << logBW) + 1 + o;
        const bool in = slot < ncl && i <= n - d;
        const int t = in ? bf_ptype_bases(S[i], S[i + d]) : 0;
        const unsigned mk = __ballot_sync(BF_FULL, t != 0);
        if (in && !t) qb_out[od + i - 1] = 0.0;
        if (t) cl_pp[count + __popc(mk & ((1u << lane) - 1))] = (unsigned short)i;
        count += __popc(mk);
      }
      if (lane == 0) NP[d] = (unsigned short)count;
      __syncwarp();
      for (int c = lane; c < count; c += 32) {
        const int i = cl_pp[c], j = i + d;
        const int t = bf_ptype_bases(S[i], S[j]);
        const int si1 = S[i + 1], sj1 = S[j - 1], sim = S[i - 1], sjp = S[j + 1], tr = bf_rtype(t);
        double2 *dst = reinterpret_cast<double2 *>(ent + ((size_t)(d - 4) * ncl + c) * kEntDc);
        dst[0] = make_double2((double)i, T.x_mmI[t][si1][sj1]);   // (small integers as values, not as bit patterns)
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
          w[1 + k] = t2 ? (t2 > 2 ? e * inv_tau : e) : 0.0;
        }
        const int bx = (i - 1) >> logBW;
        w[10] = 0.0;
        w[11] = (double)((bx >> logC) * WIN + ((i - 1) & (BW - 1)));
#pragma unroll
        for (int q2 = 0; q2 < 6; q2++) dst[4 + q2] = make_double2(w[2 * q2], w[2 * q2 + 1]);
      }
      __syncwarp();
    }
    __threadfence_block();
    cl_sync();
    const int st_m10 = lane / 10, st_q10 = lane - 10 * (lane / 10);
    auto stage = [&](int dn) {
      const int mine = ((int)NP[dn] - warp + NT - 1) / NT;
      const char *src = reinterpret_cast<const char *>(ent + ((size_t)(dn - 4) * ncl + warp) * kEntDc);
      const unsigned dst = (unsigned)__cvta_generic_to_shared(wl);
      // 16-byte pieces: lane -> (entry lane / 10, piece lane % 10), three entries per pass
      for (int m = st_m10; m < mine && lane < 30; m += 3)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + (unsigned)(m * kEntDc * 8 + st_q10 * 16)),
                     "l"(src + (size_t)m * NT * kEntDc * 8 + st_q10 * 16)
                     : "memory");
    };
    if (warp < NT && n - 1 >= BF_TURN + 1) stage(BF_TURN + 1);

    int rowd = (BF_TURN + 1) % kDepth;
    for (int d = BF_TURN + 1; d <= n; d++, rowd = rowd + 1 == kDepth ? 0 : rowd + 1) {
      const int buf = d & 1;
      // ------------------------------------------------------------ taps: qb(i,j) of this CTA's pairable cells of diagonal d
      if (warp < NT && d <= n - 1) {
        const int np = NP[d];
        const unsigned sqms = sQMS + 8u * (unsigned)(((d - 2) & 3) * RS + 1);
        const unsigned sbase = sRG + 8u * (unsigned)((st_kind * kDepth + rowd) * RS + st_k * BW);
        const int smax = min(BF_MAXLOOP, d - 6);
        const int mi = smax + 1 < 0 ? 0 : smax + 1;
        const int ng = s_meta[mi], n1 = s_meta[32 + mi], nb = s_meta[64 + mi];
        auto cells = [&](auto cg_, auto c1_, auto cb_) {
          constexpr int G = decltype(cg_)::value, O = decltype(c1_)::value, Bn = decltype(cb_)::value;
          asm volatile("cp.async.wait_all;" ::: "memory");
          __syncwarp();
          const double *p = wl;
          for (int c = warp; c < np; c += NT, p += kEntDc) {
            const double2 e01 = *reinterpret_cast<const double2 *>(p), e23 = *reinterpret_cast<const double2 *>(p + 2);
            const double mlc = p[4], xt = p[7], esp = p[lsp], etl = p[ltl];
            const unsigned lc8 = 8u * (unsigned)__double2int_rn(p[19]);
            const unsigned ug = sRG + lc8, u1n = ug + 8u * wrap, ubg = ug + 16u * wrap;
            double ag0 = 0.0, ag1 = 0.0, a1 = 0.0, ab = 0.0;
#pragma unroll
            for (int k = 0; k < G; k++) {
              if (k & 1) ag1 = fma(lds_d(ug + xk[k]), wk[k], ag1);
              else ag0 = fma(lds_d(ug + xk[k]), wk[k], ag0);
            }
#pragma unroll
            for (int k = 0; k < O; k++) a1 = fma(lds_d(u1n + xk[kNSG + k]), wk[kNSG + k], a1);
#pragma unroll
            for (int k = 0; k < Bn; k++) ab = fma(lds_d(ubg + xk[kNSG + kNS1 + k]), wk[kNSG + kNS1 + k], ab);
            double tot = fma(lds_d(ubg + xk[kNSlot - 1]), esp, (ag0 + ag1) * e01.y);
            tot = fma(a1, e23.x, fma(ab, xt, tot));
            tot = bf_warp_sum(tot);
            const double qb = tot + e23.y + lds_d(sqms + lc8) * mlc;   // + hairpin + multiloop closed by (i,j)
            const int i = __double2int_rn(e01.x), bx = (i - 1) >> logBW, o = (i - 1) & (BW - 1);
            const double v = qb * etl;
            if (lane < nst) {
              const int bxk = bx - st_k;
              if (bxk >= 0) cl_st_f64(cl_map(sbase + 8u * (unsigned)((bxk >> logC) * WIN + o), (unsigned)(bxk & (C - 1))), v);
            } else if (lane == nst) {
              TMPQ[buf * ncl + ((bx >> logC) << logBW) + o] = v;
            } else if (lane == nst + 1) {
              QST[buf * ncl + ((bx >> logC) << logBW) + o] = qb;
            }
          }
        };
        using std::integral_constant;
        if (ng <= 2 && n1 <= 1 && nb <= 1) cells(integral_constant<int, 2>(), integral_constant<int, 1>(), integral_constant<int, 1>());
        else if (ng <= 5 && n1 <= 2 && nb <= 2) cells(integral_constant<int, 5>(), integral_constant<int, 2>(), integral_constant<int, 2>());
        else if (ng <= 8) cells(integral_constant<int, 8>(), integral_constant<int, kNS1>(), integral_constant<int, kNSB>());
        else cells(integral_constant<int, kNSG>(), integral_constant<int, kNS1>(), integral_constant<int, kNSB>());
        __syncwarp();
      }
      // ------------------------------------------------------------ combine of diagonal d-1: this CTA's cells
      constexpr int NWS = NW - NT;
      const int aw = warp - NT;
      const int ncomb = (ncl + 31) >> 5;
      if (d > BF_TURN + 1 && aw >= 0)
        for (int cp = NWS - 2 - aw; cp >= 0 && cp < ncomb; cp += NWS - 1) {   // from the last-but-one warp down
          const int dd = d - 1, pb = dd & 1;
          const int slot = cp * 32 + lane;
          const int lb = slot >> logBW, o = slot & (BW - 1);
          const int bx = (lb << logC) + r;
          const int i = (bx << logBW) + 1 + o;
          if (slot < ncl && i <= n - dd) {
            const int j = i + dd, lc = lb * WIN + o;
            const int nchp = (n - dd + 31) >> 5;
            const int Pp = (2 * nchp <= NWS) ? kPMax : 1;
            double qms = 0.0, qms1 = 0.0;   // fixed order: the sum is reproducible
            {
              const double *sb = SPART + (size_t)pb * C * kPMax * ncl + slot;
              if (Pp == 2) {
#pragma unroll 2
                for (int rr = 0; rr < C; rr += 2) {
                  const double a = sb[(2 * rr) * ncl], bq = sb[(2 * rr + 1) * ncl], cq = sb[(2 * rr + 2) * ncl], e = sb[(2 * rr + 3) * ncl];
                  qms += a + bq; qms1 += cq + e;
                }
              } else {
#pragma unroll 2
                for (int rr = 0; rr < C; rr += 2) { qms += sb[(2 * rr) * ncl]; qms1 += sb[(2 * rr + 2) * ncl]; }
              }
              qms += qms1;
            }
            const double tq = TMPQ[pb * ncl + slot];
            TMPQ[pb * ncl + slot] = 0.0;
            double qm1 = tq, au = 0.0;
            if (dd > BF_TURN + 1) {
              const int pr = ((dd - 1) & 1) * RS;
              qm1 = fma(Q1P[pr + lc], bu1, tq);                       // (i, j-1) plus one unpaired base
              au = bu1 * (Q1P[pr + lc + 1] + AU[pr + lc + 1]);        // stems starting right of i
            }
            const double qm = qms + au + qm1;
            const int o0 = tri_off(n, dd);
            if (qmg) { qmg[o0 + i - 1] = qm; qmg[tri_slot + o0 + i - 1] = qm1; }
            Q1P[(dd & 1) * RS + lc] = qm1;
            AU[(dd & 1) * RS + lc] = au;
            QMS[(dd & 3) * RS + lc] = qms;
            if (o == 0 && bx >= 1) {
              const unsigned rk = (unsigned)((bx - 1) & (C - 1));
              const int lcp = ((bx - 1) >> logC) * WIN + BW;
              cl_st_f64(cl_map(sQ1P + 8u * (unsigned)((dd & 1) * RS + lcp), rk), qm1);
              cl_st_f64(cl_map(sAU + 8u * (unsigned)((dd & 1) * RS + lcp), rk), au);
              cl_st_f64(cl_map(sQMS + 8u * (unsigned)((dd & 3) * RS + lcp), rk), qms);
            }
            const int mcol = j + 1;
            if (mcol <= n) cl_st_f64(cl_map(sCOL + 8u * (unsigned)(col_base(C, mcol & (C - 1), mcol >> logC) + i - 1), (unsigned)(mcol & (C - 1))), qm);
            cl_st_f64(cl_map(sROW + 8u * (unsigned)(row_base(C, i & (C - 1), i >> logC, n + 1) + dd - 4), (unsigned)(i & (C - 1))), qm1);
          }
        }
      // ------------------------------------------------------------ HBM table: qb of diagonal d-1, one phase late (see the MFE kernel)
      if (aw == NWS - 1 && d - 1 >= BF_TURN + 1 && d - 1 <= n - 1) {
        const int dc = d - 1;
        for (int slot = lane; slot < ncl; slot += 32) {
          const int lb = slot >> logBW, o = slot & (BW - 1);
          const int i = ((((lb << logC) + r) << logBW)) + 1 + o;
          const double v = QST[(dc & 1) * ncl + slot];
          if (v >= 0.0) { qb_out[tri_off(n, dc) + i - 1] = v; QST[(dc & 1) * ncl + slot] = -1.0; }
        }
      }
      // ------------------------------------------------------------ split partial sums of diagonal d over this CTA's split positions
      if (aw >= 0 && d <= n - 1) {
        const int ncell = n - d, nch = (ncell + 31) >> 5;
        const int Pp = (2 * nch <= NWS) ? kPMax : 1;
        const int nitems = nch * Pp;
        for (int it = aw; it < nitems; it += NWS) {
          const int ch = Pp == 2 ? it >> 1 : it, pp = Pp == 2 ? it & 1 : 0;
          const int i0 = 32 * ch + 1, i = i0 + lane;
          const int ilast = min(i0 + 31, ncell);
          const int lo = i0 + 5, hi = ilast + d - 4;
          const int mfirst = lo + ((r - lo) & (C - 1));
          const int cnt = mfirst > hi ? 0 : ((hi - mfirst) >> logC) + 1;
          const int per = Pp == 2 ? (cnt + 1) >> 1 : cnt;
          const int t0 = pp * per, t1 = min(cnt, t0 + per);
          double acc0 = 0.0, acc1 = 0.0;
          if (t0 < t1 && d >= 9) {
            int m = mfirst + (t0 << logC);
            const int q = m >> logC;
            unsigned aL = sCOL + 8u * (unsigned)(col_base(C, r, q) + i - 1);
            unsigned aR = sROW + 8u * (unsigned)(row_base(C, r, q, n + 1) + i + d - m - 4);
            const int iv = i <= ncell ? i : -100000;
            int t = t0;
            for (; t + 1 < t1; t += 2) {
              if ((unsigned)(iv - (m - d + 4)) <= (unsigned)(d - 9)) acc0 = fma(lds_d(aL), lds_d(aR), acc0);
              aL += 8u * (unsigned)m; aR += 8u * (unsigned)(n + 1 - m - C); m += C;
              if ((unsigned)(iv - (m - d + 4)) <= (unsigned)(d - 9)) acc1 = fma(lds_d(aL), lds_d(aR), acc1);
              aL += 8u * (unsigned)m; aR += 8u * (unsigned)(n + 1 - m - C); m += C;
            }
            if (t < t1 && (unsigned)(iv - (m - d + 4)) <= (unsigned)(d - 9)) acc0 = fma(lds_d(aL), lds_d(aR), acc0);
          }
          if (i <= ncell) {
            const int bx = (i - 1) >> logBW, o = (i - 1) & (BW - 1);
            const int slot = ((bx >> logC) << logBW) + o;
            cl_st_f64(cl_map(sSPART + 8u * (unsigned)(((buf * C + r) * kPMax + pp) * ncl + slot), (unsigned)(bx & (C - 1))), acc0 + acc1);
          }
        }
      }
      cl_arrive();
      // ---- between arrive and wait: work that nobody else sees
      if (warp < NT) {
        if (d + 1 <= n - 1) stage(d + 1);
#pragma unroll
        for (int k = 0; k < kNSlot; k++) {
          const unsigned x = (unsigned)xk[k] + 8u * (unsigned)RS;
          xk[k] = (int)min(x, x - 8u * wrap);
        }
      } else {   // clear ring row d+2: last read in phase d-1, written from phase d+2 on
        const int row = rowd + 2 >= kDepth ? rowd + 2 - kDepth : rowd + 2;
        for (int x = tid - NT * 32; x < RS; x += (NW - NT) * 32) {
          RG[row * RS + x] = 0.0; RG[(kDepth + row) * RS + x] = 0.0; RG[(2 * kDepth + row) * RS + x] = 0.0;
        }
      }
      cl_wait();
    }
  }
  cl_sync();
}

int ilog2(int x) { int l = 0; while ((1 << l) < x) l++; return l; }

bool make_geom(int nmax, int C, int BW, int elem_banks /*32: int, 16: double*/, ClGeom *out) {
  ClGeom g;
  g.C = C; g.logC = ilog2(C); g.BW = BW; g.logBW = ilog2(BW); g.WIN = BW + 32; g.K = 1 + 32 / BW;
  const int nblk = (nmax + BW - 1) / BW;
  g.NLB = (nblk + C - 1) / C;
  g.ncl = g.NLB * BW;
  g.RS = pick_rs(g.NLB * g.WIN - 1, elem_banks);   // >= NLB * WIN + 1
  const int Q = nmax / C + 2;
  int cc = 0, rc = 0;
  for (int r = 0; r < C; r++) {
    cc = std::max(cc, col_base(C, r, Q));
    int best = 0;
    for (int q = 0; q <= Q; q++) best = std::max(best, row_base(C, r, q, nmax + 1));
    rc = std::max(rc, best + nmax + 1);
  }
  g.colcap = cc + 8; g.rowcap = rc + 8;
  g.lcap = (g.ncl + kNTcl - 1) / kNTcl + 2;
  *out = g;
  return true;
}

// ---------------------------------------------------------------------------------------------------- host side
// How many clusters of C CTAs the GPU runs at once (one CTA per SM; clusters do not span GPCs, so this is less than sms / C).
template <class K>
int max_active_clusters(K kern, int C) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3((unsigned)(C * 64), 1, 1);
  cfg.blockDim = dim3(kNWcl * 32, 1, 1);
  cfg.dynamicSmemBytes = kSmemBudget;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
  return n;
}
template <class K>
cudaError_t cl_attrs(K kern) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
}
// slots[log2 C]: clusters in flight, measured once per kernel (0 = that cluster size cannot be launched)
struct ClSlots { bool have = false; int n[5] = {0, 0, 0, 0, 0}; };
ClSlots g_slots_mfe, g_slots_pf;
std::mutex g_slots_mu;
template <class K>
const ClSlots &cl_slots(ClSlots &s, K kern) {
  std::lock_guard<std::mutex> lk(g_slots_mu);
  if (!s.have) {
    if (cl_attrs(kern) == cudaSuccess)
      for (int l = 1; l <= 4; l++) s.n[l] = max_active_clusters(kern, 1 << l);
    else cudaGetLastError();
    s.have = true;
  }
  return s;
}

// Measured on one B200 (scripts/cl_sweep.py, profiles/r02_cluster_sweep.txt; fill + exterior recursion + backtrack per call): a
// cluster folds one sequence in ~2.7 us per diagonal almost independently of its size -- 0.41 / 0.57 / 0.74 / 0.9 / 1.3 ms at
// 150 / 200 / 250 / 300 / 400 nt -- where the single-CTA kernels need 0.59 / 1.03 / 1.87 / 2.6 / 4.3 ms (MFE) and 0.77 / 1.38 / 2.6 /
// 3.7 / 7.2 ms (PF) however few sequences there are.  So the cluster kernels take a batch when it fits in few ROUNDS of the
// clusters in flight: rounds allowed by length.
int mfe_rounds_allowed(int nmax) { return nmax < 130 ? 0 : nmax < 230 ? 1 : nmax < 330 ? 2 : 3; }
int pf_rounds_allowed(int nmax) { return nmax < 130 ? 0 : nmax < 180 ? 1 : nmax < 230 ? 2 : nmax < 350 ? 3 : 5; }

// cforce: BF_CL_C (0: the rule's choice), bw: BF_CL_BW
struct ClCfg { bool ok, dflt; int slots; ClGeom g; MfeClPlan pl; };
ClCfg mfe_cl_cfg(int nmax, int B, int cforce, int bw) {
  ClCfg c;
  c.ok = c.dflt = false; c.slots = 0;
  if (nmax < 1 || nmax > 2000) return c;
  if (bw != 16 && bw != 32) return c;
  const ClSlots &sl = cl_slots(g_slots_mfe, bf_k_mfe_cl<kNWcl, kNTcl>);
  int best_rounds = 1 << 30;
  for (int C : {2, 4, 8, 16}) {
    if (cforce ? C != cforce : C < 4) continue;   // pairs of CTAs measured no faster than one CTA
    ClCfg t = c;
    if (!make_geom(nmax, C, bw, 32, &t.g)) continue;
    t.pl = mfe_cl_plan(nmax, t.g);
    t.slots = sl.n[t.g.logC];
    if (t.pl.total > kSmemBudget || t.slots < 1) continue;
    const int rounds = ((B > 0 ? B : 1) + t.slots - 1) / t.slots;
    if (rounds < best_rounds) { best_rounds = rounds; c = t; c.ok = true; }   // ties: the smaller cluster (leaves SMs to the other stream)
  }
  if (c.ok) c.dflt = best_rounds <= mfe_rounds_allowed(nmax);
  return c;
}

struct PfClCfg { bool ok, dflt; int slots; ClGeom g; PfClPlan pl; };
PfClCfg pf_cl_cfg(int nmax, int B, int cforce, int bw) {
  PfClCfg c;
  c.ok = c.dflt = false; c.slots = 0;
  if (nmax < 1 || nmax > 2000) return c;
  if (bw != 16 && bw != 32) return c;
  const ClSlots &sl = cl_slots(g_slots_pf, bf_k_pf_cl<kNWcl, kNTcl>);
  int best_rounds = 1 << 30;
  for (int C : {2, 4, 8, 16}) {
    if (cforce ? C != cforce : C < 4) continue;
    PfClCfg t = c;
    if (!make_geom(nmax, C, bw, 16, &t.g)) continue;
    t.pl = pf_cl_plan(nmax, t.g);
    t.slots = sl.n[t.g.logC];
    if (t.pl.total > kSmemBudget || t.slots < 1) continue;
    const int rounds = ((B > 0 ? B : 1) + t.slots - 1) / t.slots;
    if (rounds < best_rounds) { best_rounds = rounds; c = t; c.ok = true; }
  }
  if (c.ok) c.dflt = best_rounds <= pf_rounds_allowed(nmax);
  return c;
}

template <class K, class... Args>
cudaError_t cl_launch(K kern, int nclusters, int C, unsigned smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3((unsigned)(nclusters * C), 1, 1);
  cfg.blockDim = dim3(kNWcl * 32, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

}  // namespace

// The cluster kernels take a batch when asked to (BF_CL=1, wherever they cover the length) or, by default, when the batch fits in
// few rounds of the clusters in flight (see *_rounds_allowed); BF_CL=0 switches them off.  A plan is one cluster per sequence, as
// many as run at once; its workspace is one slab of cell entries per CTA.
bool bf_cl_mfe_plan(int nmax, int B, const BfOpts &o, BfPlan *p) {
  if (o.cl == 0 || B <= 0) return false;
  const ClCfg c = mfe_cl_cfg(nmax, B, o.cl_c, o.cl_bw);
  if (!c.ok || !(o.cl == 1 || c.dflt)) return false;
  p->family = BF_FAM_CLUSTER;
  p->key = c.g.C;
  p->bw = c.g.BW;
  p->grid = B < c.slots ? B : c.slots;
  p->smem = c.pl.total;
  p->ws = (size_t)c.g.C * (((size_t)nmax * c.g.ncl * kEntW + 7) / 8 * 8);   // ints
  return true;
}

cudaError_t bf_launch_mfe_cl(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, int *ctri, int *ftri, int *ws, int *work_counter,
                             cudaStream_t st) {
  ClGeom g;
  make_geom(b.stride, p.key, p.bw, 32, &g);
  const uint32_t *taps = nullptr;
  cudaError_t e = taps_device(g.RS, 32, &taps);
  if (e != cudaSuccess) return e;
  return cl_launch(bf_k_mfe_cl<kNWcl, kNTcl>, p.grid, g.C, (unsigned)p.smem, st, dP, b, ctri, ftri, bf_tri_slot(b.stride), ws, p.ws, taps,
                   mfe_cl_plan(b.stride, g), g, work_counter);
}

// ---------------------------------------------------------------------------------------------------- partition function
bool bf_cl_pf_plan(int nmax, int B, const BfOpts &o, BfPlan *p) {
  if (o.cl == 0 || B <= 0) return false;
  const PfClCfg c = pf_cl_cfg(nmax, B, o.cl_c, o.cl_bw);
  if (!c.ok || !(o.cl == 1 || c.dflt)) return false;
  p->family = BF_FAM_CLUSTER;
  p->key = c.g.C;
  p->bw = c.g.BW;
  p->grid = B < c.slots ? B : c.slots;
  p->smem = c.pl.total;
  p->ws = (size_t)c.g.C * (((size_t)nmax * c.g.ncl * kEntDc + 7) / 8 * 8);   // doubles
  return true;
}

cudaError_t bf_launch_pf_cl(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, double *qbtri, double *ws, double *qmseq,
                            const int *mfe_for_scale, double *lnscale, int *work_counter, cudaStream_t st) {
  ClGeom g;
  make_geom(b.stride, p.key, p.bw, 16, &g);
  const uint32_t *taps = nullptr;
  cudaError_t e = taps_device(g.RS, 16, &taps);
  if (e != cudaSuccess) return e;
  return cl_launch(bf_k_pf_cl<kNWcl, kNTcl>, p.grid, g.C, (unsigned)p.smem, st, dP, b, qbtri, bf_tri_slot(b.stride), ws, p.ws, qmseq,
                   mfe_for_scale, lnscale, taps, pf_cl_plan(b.stride, g), g, work_counter);
}
