// bf_outside.cu -- outside passes (sm_100a): of the partition function (base-pair probabilities, ensemble defect) and of the
// minimum free energy (the best structure containing each pair, bf_k_mfe_out below).
//
// Replaces md.compute_bpp=1 + fc.pf() + fc.ensemble_defect(target) (utils/energy_scores.py:362-374 in the reference).
// Formulated as the reverse-mode derivative of the inside recursion of bf_k_pf_fill in GATHER form, so that it runs
// on the same diagonal-major tables with stride-1 accesses, diagonals d = n-1 down to 4 (SURVEY.md A.10):
//
//   bqm(a,b)  = sum_{m>=5} H(a,b+m) qm1(b+1,b+m)                      H(a,j) = bqm(a,j) + G(a-1,j+1)
//   bqm1(a,b) = bqm(a,b) + bu bqm1(a,b+1) + A(a,b) + sum_{m>=5} H(a-m,b) qm(a-m,a-1)
//               A(a,b) = sum_{m>=1} bu^m bqm(a-m,b) = bu (bqm(a-1,b) + A(a-1,b))
//   bqb(a,b)  = q5[a-1] xExt(a,b) q3[b+1] / Z + bqm1(a,b) xMLstem(a,b) + sum_{outer (i,j)} bqb(i,j) B(interior)
//   G(a,b)    = bqb(a,b) B(MLclosing) xMLstem(closing) scale^2,       P(a,b) = bqb(a,b) qb(a,b)
//
// (bq* are d ln Z / d q*; all quantities carry the inside kernel's per-nucleotide scale.)  The outer pair table is kept in
// the same three "outer-term folded in" variants as the inside rings, so a decomposable enclosing loop is one load + fma.
// One persistent CTA per sequence, warps own 32-cell chunks of a diagonal, one barrier per diagonal.
#include "bf_kernels.h"

#include "bf_device.cuh"

namespace {

struct OutPlan {
  int rs;
  size_t o_wg, o_wb, o_w1, o_scl, o_q5, o_q3, o_prow, o_ppair, o_ap, o_bqm, o_bqm1, o_g, o_toff, o_pt, o_stk, o_S, total;
};
__host__ __device__ inline OutPlan out_plan(int nmax) {
  OutPlan p;
  p.rs = (nmax + 8 + 3) / 4 * 4;
  size_t o = 0;
  p.o_wg = o; o += 31 * 32 * sizeof(double);
  p.o_wb = o; o += 32 * sizeof(double);
  p.o_w1 = o; o += 32 * sizeof(double);
  p.o_scl = o; o += (size_t)p.rs * sizeof(double);
  p.o_q5 = o; o += (size_t)p.rs * sizeof(double);
  p.o_q3 = o; o += (size_t)p.rs * sizeof(double);
  p.o_prow = o; o += (size_t)p.rs * sizeof(double);
  p.o_ppair = o; o += (size_t)p.rs * sizeof(double);
  p.o_ap = o; o += (size_t)2 * p.rs * sizeof(double);
  p.o_bqm = o; o += (size_t)2 * p.rs * sizeof(double);
  p.o_bqm1 = o; o += (size_t)2 * p.rs * sizeof(double);
  p.o_g = o; o += (size_t)4 * p.rs * sizeof(double);
  p.o_toff = o; o += (size_t)p.rs * sizeof(int);
  p.o_pt = o; o += (size_t)p.rs * sizeof(short);
  p.o_stk = o; o += (size_t)p.rs * sizeof(short);
  p.o_S = o; o += (nmax + 2 + 15) / 16 * 16;
  p.total = o;
  return p;
}

// KEEP: also write the outside values bf_k_unpaired reads, per sequence three packed triangles at keep + sq * 3 * tri_slot:
// bqb, bqm and bqm1 without its bu * bqm1(a,b+1) self-recursion (qm1(a,b)'s outside value as its parents use it)
template <int NW, bool KEEP = false>
__global__ void __launch_bounds__(NW * 32) bf_k_pf_out(const BfParams *__restrict__ P, BfBatchDev b, const double *qbtri, const double *qmseq,
                                                       size_t tri_slot, double *ws, const double *lnscale, const char *targets,
                                                       int n_targets, int tstride, double *out_defect, double *out_bpp, int *work_counter,
                                                       double *keep) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq, s_bad;
  __shared__ double s_red[NW];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  const OutPlan pl = out_plan(nmax);
  const int RS = pl.rs;
  const BfSmallD &T = P->sd;
  double *wg = reinterpret_cast<double *>(dyn + pl.o_wg);
  double *wb = reinterpret_cast<double *>(dyn + pl.o_wb);
  double *w1 = reinterpret_cast<double *>(dyn + pl.o_w1);
  double *scl = reinterpret_cast<double *>(dyn + pl.o_scl);
  double *q5 = reinterpret_cast<double *>(dyn + pl.o_q5);
  double *q3 = reinterpret_cast<double *>(dyn + pl.o_q3);
  double *prow = reinterpret_cast<double *>(dyn + pl.o_prow);
  double *ppair = reinterpret_cast<double *>(dyn + pl.o_ppair);
  double *AP = reinterpret_cast<double *>(dyn + pl.o_ap);
  double *BQM = reinterpret_cast<double *>(dyn + pl.o_bqm);
  double *BQM1 = reinterpret_cast<double *>(dyn + pl.o_bqm1);
  double *GR = reinterpret_cast<double *>(dyn + pl.o_g);
  int *toff = reinterpret_cast<int *>(dyn + pl.o_toff);
  short *pt = reinterpret_cast<short *>(dyn + pl.o_pt);
  short *stk = reinterpret_cast<short *>(dyn + pl.o_stk);
  uint8_t *S = dyn + pl.o_S;
  // per-CTA workspace: H and the three outer-pair tables, packed triangles
  double *H = ws + (size_t)blockIdx.x * 4 * tri_slot;
  double *OG = H + tri_slot, *O1 = OG + tri_slot, *OB = O1 + tri_slot;

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int sq = s_seq;
    if (sq >= b.B) break;
    const int n = b.len[sq];
    const char *src = b.seq + (size_t)sq * b.stride;
    for (int k = tid; k <= n + 1; k += blockDim.x) S[k] = (uint8_t)((k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0);
    for (int k = tid; k <= n; k += blockDim.x) toff[k] = (k >= 4) ? tri_off(n, k) : 0;
    const double lns = lnscale[sq];
    for (int k = tid; k <= n + 2; k += blockDim.x) { scl[k] = exp(-lns * k); prow[k] = 0.0; ppair[k] = 0.0; pt[k] = 0; }
    for (int k = tid; k < 2 * RS; k += blockDim.x) { AP[k] = 0.0; BQM[k] = 0.0; BQM1[k] = 0.0; }
    for (int k = tid; k < 4 * RS; k += blockDim.x) GR[k] = 0.0;
    if (tid == 0) s_bad = 0;
    __syncthreads();
    for (int k = tid; k < 31 * 32; k += blockDim.x) {
      const int s = k >> 5, u1 = (k & 31) + 2;
      wg[k] = (s >= 6 && u1 <= s - 2) ? T.x_interior[s] * T.x_ninio[abs(s - 2 * u1)] * scl[s + 2] : 0.0;
    }
    if (tid < 32) {
      wb[tid] = (tid >= 2 && tid <= 30) ? T.x_bulge[tid] * scl[tid + 2] : 0.0;
      w1[tid] = (tid >= 4 && tid <= 30) ? T.x_interior[tid] * T.x_ninio[tid - 2] * scl[tid + 2] : 0.0;
    }
    const double *qb = qbtri + (size_t)sq * tri_slot;
    const double *QM = qmseq + (size_t)sq * 2 * tri_slot, *QM1 = QM + tri_slot;
    const double bu1 = exp(log(T.x_MLbase) - lns), sc1 = scl[1];
    const double xtau = T.x_TerminalAU, inv_tau = 1.0 / xtau;
    const double xclose = T.x_MLclosing * scl[2];
    auto xext = [&](int i, int j, int t) -> double { return bf_x_ext(T, t, (i > 1) ? S[i - 1] : -1, (j < n) ? S[j + 1] : -1); };
    // target pair table (thread 0) + exterior chains q5 (warp 0) and q3 (warp 1)
    if (tid == 0 && targets) {
      const char *db = targets + (size_t)sq * n_targets * tstride;
      int sp = 0;
      for (int i = 1; i <= n; i++) {
        const char ch = db[i - 1];
        if (ch == '(') stk[sp++] = (short)i;
        else if (ch == ')') {
          if (!sp) { s_bad = 1; break; }
          const int o = stk[--sp];
          pt[o] = (short)i; pt[i] = (short)o;
        }
      }
      if (sp) s_bad = 1;
    }
    if (warp == 0) {
      if (lane == 0) q5[0] = 1.0;
      __syncwarp();
      for (int j = 1; j <= n; j++) {
        double sum = 0.0;
        for (int i = 1 + lane; i < j - BF_TURN; i += 32) {
          const int t = bf_ptype_bases(S[i], S[j]);
          if (t) sum += q5[i - 1] * qb[toff[j - i] + i - 1] * xext(i, j, t);
        }
        sum = bf_warp_sum(sum);
        if (lane == 0) q5[j] = sum + q5[j - 1] * sc1;
        __syncwarp();
      }
    } else if (warp == 1 || NW == 1) {
      if (lane == 0) q3[n + 1] = 1.0;
      __syncwarp();
      for (int i = n; i >= 1; i--) {
        double sum = 0.0;
        for (int j = i + BF_TURN + 1 + lane; j <= n; j += 32) {
          const int t = bf_ptype_bases(S[i], S[j]);
          if (t) sum += qb[toff[j - i] + i - 1] * xext(i, j, t) * q3[j + 1];
        }
        sum = bf_warp_sum(sum);
        if (lane == 0) q3[i] = sum + q3[i + 1] * sc1;
        __syncwarp();
      }
    }
    __syncthreads();
    const double invZ = 1.0 / q5[n];

    for (int d = n - 1; d >= BF_TURN + 1; d--) {
      const int ncell = n - d;
      const int r0 = (d & 1) * RS, r1 = ((d + 1) & 1) * RS;
      for (int c = warp * 32; c < ncell; c += NW * 32) {
        const int a = c + lane + 1;
        if (a > ncell) continue;
        const int bb = a + d;
        const int t = bf_ptype_bases(S[a], S[bb]);
        // ---- bqm(a,b): (a,b) as the left part of a longer multiloop segment
        double bqm = 0.0;
        for (int m = 5; a + d + m <= n; m++) bqm = fma(H[toff[d + m] + a - 1], QM1[toff[m - 1] + a + d], bqm);
        const double gprev = (a > 1 && bb < n && d + 2 <= n - 1) ? GR[((d + 2) & 3) * RS + a - 1] : 0.0;
        const double hab = bqm + gprev;
        // ---- bqm1(a,b)
        double u2 = 0.0;
        for (int m = 5; m <= a - 1; m++) u2 = fma(H[toff[d + m] + a - m - 1], QM[toff[m - 1] + a - m - 1], u2);
        double ap = 0.0, bqm1 = bqm + u2;
        if (d + 1 <= n - 1) {
          if (a > 1) ap = bu1 * (BQM[r1 + a - 1] + AP[r1 + a - 1]);
          if (bb + 1 <= n) bqm1 += BQM1[r1 + a] * bu1;
        }
        bqm1 += ap;
        // ---- bqb(a,b)
        double bqb = 0.0;
        if (t) {
          bqb = q5[a - 1] * xext(a, bb, t) * q3[bb + 1] * invZ;
          if (a > 1 && bb < n) bqb = fma(bqm1, bf_x_mlstem(T, t, S[a - 1], S[bb + 1]), bqb);
          const int t2 = bf_rtype(t), sq1 = S[bb + 1], sp1 = S[a - 1];
          double accg = 0.0, acc1 = 0.0, accb = 0.0, accs = 0.0;
          const int smax = min(BF_MAXLOOP, n - 1 - d - 2);
          for (int s = 0; s <= smax; s++) {
            const int o = toff[d + 2 + s];
            for (int u1 = 0; u1 <= s; u1++) {
              const int i = a - 1 - u1, j = bb + 1 + s - u1, u2l = s - u1;
              if (i < 1 || j > n) continue;
              const int nl = max(u1, u2l), ns = min(u1, u2l);
              if (ns == 0 && nl >= 2) accb = fma(OB[o + i - 1], wb[s], accb);
              else if (ns == 1 && nl >= 3) acc1 = fma(O1[o + i - 1], w1[s], acc1);
              else if (ns >= 2 && !(ns == 2 && nl <= 3)) accg = fma(OG[o + i - 1], wg[(s << 5) + u1 - 2], accg);
              else {
                const int to = bf_ptype_bases(S[i], S[j]);
                if (!to) continue;
                double ov = OB[o + i - 1];
                if (to > 2) ov *= inv_tau;
                accs = fma(ov, bf_x_intloop(P, T, u1, u2l, to, t2, S[i + 1], S[j - 1], sp1, sq1) * scl[s + 2], accs);
              }
            }
          }
          bqb += accg * T.x_mmI[t2][sq1][sp1] + acc1 * T.x_mm1nI[t2][sq1][sp1] + accb * (t > 2 ? xtau : 1.0) + accs;
        }
        const int o = toff[d] + a - 1;
        if (KEEP) {
          double *K = keep + (size_t)sq * 3 * tri_slot;
          K[o] = bqb; K[tri_slot + o] = bqm; K[2 * tri_slot + o] = bqm + u2 + ap;
        }
        H[o] = hab;
        BQM[r0 + a] = bqm;
        AP[r0 + a] = ap;
        BQM1[r0 + a] = bqm1;
        double g = 0.0, og = 0.0, o1 = 0.0, ob = 0.0;
        if (t) {
          const int si1 = S[a + 1], sj1 = S[bb - 1];
          g = bqb * xclose * bf_x_mlstem(T, bf_rtype(t), sj1, si1);
          og = bqb * T.x_mmI[t][si1][sj1];
          o1 = bqb * T.x_mm1nI[t][si1][sj1];
          ob = (t > 2) ? bqb * xtau : bqb;
          const double p = bqb * qb[o];
          atomicAdd(&prow[a], p);
          atomicAdd(&prow[bb], p);
          if (pt[a] == bb) { ppair[a] = p; ppair[bb] = p; }
          if (out_bpp) out_bpp[((size_t)sq * b.stride + (a - 1)) * b.stride + (bb - 1)] = p;
        }
        GR[(d & 3) * RS + a] = g;
        OG[o] = og; O1[o] = o1; OB[o] = ob;
      }
      __syncthreads();
    }
    // ---- ensemble defect of target 0: (1/n) sum_i (paired ? 1 - P(i, pt i) : sum_j P(i,j))
    if (out_defect) {
      double e = 0.0;
      for (int i = 1 + tid; i <= n; i += blockDim.x) e += pt[i] ? 1.0 - ppair[i] : prow[i];
      e = bf_warp_sum(e);
      if (lane == 0) s_red[warp] = e;
      __syncthreads();
      if (tid == 0) {
        double tot = 0.0;
        for (int w = 0; w < NW; w++) tot += s_red[w];
        out_defect[sq] = (s_bad || n == 0) ? -1.0 : tot / n;
      }
    }
  }
}


// =====================================================================================================
//  v2: same recursion, scheduled like bf_k_pf_fill -- phase d = combine diagonal d+1 || partial sums of diagonal d, one
//  barrier per diagonal; pairable cells compacted; the enclosing-loop sums split over the warps by loop size with the
//  decomposable classes as load + fma against warp-uniform weights; the two multiloop sums split over the warps by m.
//  The outer-pair tables only look ahead 32 diagonals, so they are 32-deep rings (generic one on chip when RGS), stored with
//  32 zeros left of position 1 and zeros right of the diagonal's end: out-of-range enclosing pairs contribute exactly 0
//  and need no predicate.
// =====================================================================================================
constexpr int kORing = 32;

struct Out2Plan {
  int rs, rr;
  size_t o_wg, o_wb, o_w1, o_scl, o_q5, o_q3, o_prow, o_ppair, o_ap, o_bqm, o_bqm1, o_g, o_pi, o_p1, o_p2, o_og, o_h, o_toff, o_pt, o_stk, o_list, o_S, total;
};
// hsm: the H triangle this pass writes and the qm / qm1 triangles of the inside pass on chip too (short sequences, one CTA per SM)
__host__ __device__ inline Out2Plan out2_plan(int nmax, int nw, bool rgs, bool hsm = false) {
  Out2Plan p;
  p.rs = (nmax + 8 + 3) / 4 * 4;
  p.rr = p.rs + 32;
  size_t o = 0;
  p.o_wg = o; o += 31 * 32 * sizeof(double);
  p.o_wb = o; o += 32 * sizeof(double);
  p.o_w1 = o; o += 32 * sizeof(double);
  p.o_scl = o; o += (size_t)p.rs * sizeof(double);
  p.o_q5 = o; o += (size_t)p.rs * sizeof(double);
  p.o_q3 = o; o += (size_t)p.rs * sizeof(double);
  p.o_prow = o; o += (size_t)p.rs * sizeof(double);
  p.o_ppair = o; o += (size_t)p.rs * sizeof(double);
  p.o_ap = o; o += (size_t)2 * p.rs * sizeof(double);
  p.o_bqm = o; o += (size_t)2 * p.rs * sizeof(double);
  p.o_bqm1 = o; o += (size_t)2 * p.rs * sizeof(double);
  p.o_g = o; o += (size_t)4 * p.rs * sizeof(double);
  p.o_pi = o; o += (size_t)2 * nw * p.rs * sizeof(double);
  p.o_p1 = o; o += (size_t)2 * nw * p.rs * sizeof(double);
  p.o_p2 = o; o += (size_t)2 * nw * p.rs * sizeof(double);
  p.o_og = o; o += rgs ? (size_t)kORing * p.rr * sizeof(double) : 0;
  p.o_h = o; o += hsm ? (size_t)3 * ((tri_size(nmax) + 7) / 8 * 8) * sizeof(double) : 0;
  p.o_toff = o; o += (size_t)p.rs * sizeof(int);
  p.o_pt = o; o += (size_t)p.rs * sizeof(short);
  p.o_stk = o; o += (size_t)p.rs * sizeof(short);
  p.o_list = o; o += (size_t)2 * p.rs * sizeof(unsigned short);
  p.o_S = o; o += (nmax + 2 + 15) / 16 * 16;
  p.total = o;
  return p;
}
// doubles of per-CTA HBM workspace: H triangle, then the rings that are not on chip
__host__ __device__ inline size_t out2_ws_doubles(int nmax, bool rgs) {
  const size_t rr = (nmax + 8 + 3) / 4 * 4 + 32;
  return ((tri_size(nmax) + 7) / 8 * 8) + (size_t)(rgs ? 2 : 3) * kORing * rr;
}

#define BF_OUT_FOR_MY_S(NW, warp, smax, s)                                                      \
  for (int idx_ = (warp), flip_ = 0, s = (smax) - idx_; s >= 0;                                  \
       idx_ += flip_ ? 2 * (warp) + 1 : 2 * ((NW) - 1 - (warp)) + 1, flip_ ^= 1, s = (smax) - idx_)

template <int NW, bool RGS, bool HSM, bool KEEP = false>   // KEEP: as for bf_k_pf_out
__global__ void __launch_bounds__(NW * 32) bf_k_pf_out2(const BfParams *__restrict__ P, BfBatchDev b, const double *qbtri, const double *qmseq,
                                                        size_t tri_slot, double *ws, size_t ws_slot, const double *lnscale, const char *targets,
                                                        int n_targets, int tstride, double *out_defect, double *out_bpp, int *work_counter,
                                                        double *keep) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq, s_bad, s_np[2];
  __shared__ double s_red[NW];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  const Out2Plan pl = out2_plan(nmax, NW, RGS, HSM);
  const int RS = pl.rs, RR = pl.rr;
  const BfSmallD &T = P->sd;
  double *wg = reinterpret_cast<double *>(dyn + pl.o_wg);
  double *wb = reinterpret_cast<double *>(dyn + pl.o_wb);
  double *w1 = reinterpret_cast<double *>(dyn + pl.o_w1);
  double *scl = reinterpret_cast<double *>(dyn + pl.o_scl);
  double *q5 = reinterpret_cast<double *>(dyn + pl.o_q5);
  double *q3 = reinterpret_cast<double *>(dyn + pl.o_q3);
  double *prow = reinterpret_cast<double *>(dyn + pl.o_prow);
  double *ppair = reinterpret_cast<double *>(dyn + pl.o_ppair);
  double *AP = reinterpret_cast<double *>(dyn + pl.o_ap);
  double *BQM = reinterpret_cast<double *>(dyn + pl.o_bqm);
  double *BQM1 = reinterpret_cast<double *>(dyn + pl.o_bqm1);
  double *GR = reinterpret_cast<double *>(dyn + pl.o_g);
  double *PI = reinterpret_cast<double *>(dyn + pl.o_pi);
  double *P1 = reinterpret_cast<double *>(dyn + pl.o_p1);
  double *P2 = reinterpret_cast<double *>(dyn + pl.o_p2);
  int *toff = reinterpret_cast<int *>(dyn + pl.o_toff);
  short *pt = reinterpret_cast<short *>(dyn + pl.o_pt);
  short *stk = reinterpret_cast<short *>(dyn + pl.o_stk);
  unsigned short *LST = reinterpret_cast<unsigned short *>(dyn + pl.o_list);
  uint8_t *S = dyn + pl.o_S;
  double *wsp = ws + (size_t)blockIdx.x * ws_slot;
  const size_t tri_pad = (tri_size(nmax) + 7) / 8 * 8;
  double *HQ = reinterpret_cast<double *>(dyn + pl.o_h);   // HSM: H, qm, qm1 of the sequence in work
  double *H = HSM ? HQ : wsp;
  double *rings = wsp + tri_pad;
  double *OG = RGS ? reinterpret_cast<double *>(dyn + pl.o_og) : rings + 2 * kORing * RR;
  double *O1 = rings, *OB = rings + kORing * RR;
  // ring entry of position p (1-based index along the diagonal) of diagonal x: row (x & 31), offset 32 + p
#define BF_OROW(x) (((x) & (kORing - 1)) * RR + 32)

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int sq = s_seq;
    if (sq >= b.B) break;
    const int n = b.len[sq];
    const char *src = b.seq + (size_t)sq * b.stride;
    for (int k = tid; k <= n + 1; k += blockDim.x) S[k] = (uint8_t)((k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0);
    for (int k = tid; k <= n; k += blockDim.x) toff[k] = (k >= 4) ? tri_off(n, k) : 0;
    const double lns = lnscale[sq];
    for (int k = tid; k <= n + 2; k += blockDim.x) { scl[k] = exp(-lns * k); prow[k] = 0.0; ppair[k] = 0.0; pt[k] = 0; }
    for (int k = tid; k < 2 * RS; k += blockDim.x) { AP[k] = 0.0; BQM[k] = 0.0; BQM1[k] = 0.0; }
    for (int k = tid; k < 4 * RS; k += blockDim.x) GR[k] = 0.0;
    for (int k = tid; k < kORing * RR; k += blockDim.x) { OG[k] = 0.0; O1[k] = 0.0; OB[k] = 0.0; }
    if (tid == 0) s_bad = 0;
    __syncthreads();
    for (int k = tid; k < 31 * 32; k += blockDim.x) {
      const int s = k >> 5, u1 = (k & 31) + 2;
      wg[k] = (s >= 6 && u1 <= s - 2) ? T.x_interior[s] * T.x_ninio[abs(s - 2 * u1)] * scl[s + 2] : 0.0;
    }
    if (tid < 32) {
      wb[tid] = (tid >= 2 && tid <= 30) ? T.x_bulge[tid] * scl[tid + 2] : 0.0;
      w1[tid] = (tid >= 4 && tid <= 30) ? T.x_interior[tid] * T.x_ninio[tid - 2] * scl[tid + 2] : 0.0;
    }
    const double *qb = qbtri + (size_t)sq * tri_slot;
    const double *QMg = qmseq + (size_t)sq * 2 * tri_slot;
    const double *QM = HSM ? HQ + tri_pad : QMg, *QM1 = HSM ? HQ + 2 * tri_pad : QMg + tri_slot;
    if (HSM) {   // visible after the barrier that precedes the diagonal loop
      const int nt = (int)tri_size(n);
      for (int k = tid; k < nt; k += blockDim.x) { HQ[tri_pad + k] = QMg[k]; HQ[2 * tri_pad + k] = QMg[tri_slot + k]; }
    }
    const double bu1 = exp(log(T.x_MLbase) - lns), sc1 = scl[1];
    const double xtau = T.x_TerminalAU, inv_tau = 1.0 / xtau;
    const double xclose = T.x_MLclosing * scl[2];
    auto xext = [&](int i, int j, int t) -> double { return bf_x_ext(T, t, (i > 1) ? S[i - 1] : -1, (j < n) ? S[j + 1] : -1); };
    // target pair table (thread 0 of the last warp) + exterior chains q5 (warp 0) and q3 (warp 1) + first pair list (warp 2)
    if (tid == (NW - 1) * 32 && targets) {
      const char *db = targets + (size_t)sq * n_targets * tstride;
      int sp = 0;
      for (int i = 1; i <= n; i++) {
        const char ch = db[i - 1];
        if (ch == '(') stk[sp++] = (short)i;
        else if (ch == ')') {
          if (!sp) { s_bad = 1; break; }
          const int o = stk[--sp];
          pt[o] = (short)i; pt[i] = (short)o;
        }
      }
      if (sp) s_bad = 1;
    }
    if (warp == 0) {
      if (lane == 0) q5[0] = 1.0;
      __syncwarp();
      for (int j = 1; j <= n; j++) {
        double sum = 0.0;
        for (int i = 1 + lane; i < j - BF_TURN; i += 32) {
          const int t = bf_ptype_bases(S[i], S[j]);
          if (t) sum += q5[i - 1] * qb[toff[j - i] + i - 1] * xext(i, j, t);
        }
        sum = bf_warp_sum(sum);
        if (lane == 0) q5[j] = sum + q5[j - 1] * sc1;
        __syncwarp();
      }
    } else if (warp == 1 || NW == 1) {
      if (lane == 0) q3[n + 1] = 1.0;
      __syncwarp();
      for (int i = n; i >= 1; i--) {
        double sum = 0.0;
        for (int j = i + BF_TURN + 1 + lane; j <= n; j += 32) {
          const int t = bf_ptype_bases(S[i], S[j]);
          if (t) sum += qb[toff[j - i] + i - 1] * xext(i, j, t) * q3[j + 1];
        }
        sum = bf_warp_sum(sum);
        if (lane == 0) q3[i] = sum + q3[i + 1] * sc1;
        __syncwarp();
      }
    }
    if (warp == (NW > 2 ? 2 : 0) && n - 1 > BF_TURN) {  // pairable cells of the first (longest-range) diagonal n-1
      int count = 0;
      const int d0 = n - 1;
      for (int base = 1; base <= n - d0; base += 32) {
        const int i = base + lane;
        const bool ok = (i <= n - d0) && bf_ptype_bases(S[i], S[i + d0]) != 0;
        const unsigned mk = __ballot_sync(BF_FULL, ok);
        if (ok) LST[(d0 & 1) * RS + count + __popc(mk & ((1u << lane) - 1))] = (unsigned short)i;
        count += __popc(mk);
      }
      if (lane == 0) s_np[d0 & 1] = count;
    }
    __syncthreads();
    const double invZ = 1.0 / q5[n];

    for (int d = n - 1; d >= BF_TURN; d--) {
      // ------------------------------------------------------------ pairable cells of the next diagonal (d-1)
      if (warp == NW - 1 && d - 1 > BF_TURN) {
        const int dn = d - 1;
        int count = 0;
        for (int base = 1; base <= n - dn; base += 32) {
          const int i = base + lane;
          const bool ok = (i <= n - dn) && bf_ptype_bases(S[i], S[i + dn]) != 0;
          const unsigned mk = __ballot_sync(BF_FULL, ok);
          if (ok) LST[(dn & 1) * RS + count + __popc(mk & ((1u << lane) - 1))] = (unsigned short)i;
          count += __popc(mk);
        }
        if (lane == 0) s_np[dn & 1] = count;
      }
      // ------------------------------------------------------------ combine diagonal d+1
      if (d + 1 <= n - 1) {
        const int dd = d + 1, ncell = n - dd, buf = dd & 1;
        const int r0 = (dd & 1) * RS, r1 = ((dd + 1) & 1) * RS;
        const double *pi = PI + buf * NW * RS, *p1 = P1 + buf * NW * RS, *p2 = P2 + buf * NW * RS;
        for (int cell = tid; cell < ncell; cell += blockDim.x) {
          const int a = cell + 1, bb = a + dd;
          const int t = bf_ptype_bases(S[a], S[bb]);
          double bqm = 0.0, u2 = 0.0;
#pragma unroll
          for (int w = 0; w < NW; w++) { bqm += p1[w * RS + cell]; u2 += p2[w * RS + cell]; }
          const double gprev = (a > 1 && bb < n && dd + 2 <= n - 1) ? GR[((dd + 2) & 3) * RS + a - 1] : 0.0;
          const double hab = bqm + gprev;
          double ap = 0.0, bqm1 = bqm + u2;
          if (dd + 1 <= n - 1) {
            if (a > 1) ap = bu1 * (BQM[r1 + a - 1] + AP[r1 + a - 1]);
            if (bb + 1 <= n) bqm1 += BQM1[r1 + a] * bu1;
          }
          bqm1 += ap;
          double bqb = 0.0;
          if (t) {
            bqb = q5[a - 1] * xext(a, bb, t) * q3[bb + 1] * invZ;
            if (a > 1 && bb < n) bqb = fma(bqm1, bf_x_mlstem(T, t, S[a - 1], S[bb + 1]), bqb);
            double enc = 0.0;
#pragma unroll
            for (int w = 0; w < NW; w++) enc += pi[w * RS + cell];
            bqb += enc;
          }
          const int o = toff[dd] + a - 1;
          if (KEEP) {
            double *K = keep + (size_t)sq * 3 * tri_slot;
            K[o] = bqb; K[tri_slot + o] = bqm; K[2 * tri_slot + o] = bqm + u2 + ap;
          }
          H[o] = hab;
          BQM[r0 + a] = bqm;
          AP[r0 + a] = ap;
          BQM1[r0 + a] = bqm1;
          double g = 0.0, og = 0.0, o1 = 0.0, ob = 0.0;
          if (t) {
            const int si1 = S[a + 1], sj1 = S[bb - 1];
            g = bqb * xclose * bf_x_mlstem(T, bf_rtype(t), sj1, si1);
            og = bqb * T.x_mmI[t][si1][sj1];
            o1 = bqb * T.x_mm1nI[t][si1][sj1];
            ob = (t > 2) ? bqb * xtau : bqb;
            const double p = bqb * qb[o];
            atomicAdd(&prow[a], p);
            atomicAdd(&prow[bb], p);
            if (pt[a] == bb) { ppair[a] = p; ppair[bb] = p; }
            if (out_bpp) out_bpp[((size_t)sq * b.stride + (a - 1)) * b.stride + (bb - 1)] = p;
          }
          GR[(dd & 3) * RS + a] = g;
          const int ro = BF_OROW(dd) + a;
          OG[ro] = og; O1[ro] = o1; OB[ro] = ob;
        }
      }
      // ------------------------------------------------------------ partial sums of diagonal d
      if (d > BF_TURN) {
        const int ncell = n - d, buf = d & 1;
        double *pi = PI + (buf * NW + warp) * RS, *p1 = P1 + (buf * NW + warp) * RS, *p2 = P2 + (buf * NW + warp) * RS;
        // ---- enclosing loops of the pairable cells: outer pair (a-1-u1, b+1+u2) on diagonal d+2+s, s = u1+u2
        const int smax = min(BF_MAXLOOP, n - 1 - d - 2);
        const int np = s_np[buf];
        const unsigned short *list = LST + buf * RS;
        for (int c = 0; c < np; c += 32) {
          const int kk = c + lane;
          const int a = list[min(kk, np - 1)];
          const int bb = a + d;
          const int t = bf_ptype_bases(S[a], S[bb]);
          const int t2 = bf_rtype(t), sq1 = S[bb + 1], sp1 = S[a - 1];
          double accg = 0.0, acc1 = 0.0, accb = 0.0;
          if (smax >= 0) {
            BF_OUT_FOR_MY_S(NW, warp, smax, s) {
              const int row = BF_OROW(d + 2 + s) + a;
              if (s >= 2) accb += (OB[row - 1] + OB[row - 1 - s]) * wb[s];
              if (s >= 4) acc1 += (O1[row - 2] + O1[row - s]) * w1[s];
              if (s >= 6) {
                const double *qp = OG + row - 3;
                const double *w = wg + (s << 5);
                const int kn = s - 3;
                double a0 = 0.0, a1 = 0.0;
                int k = 0;
                for (; k + 1 < kn; k += 2) { a0 = fma(qp[-k], w[k], a0); a1 = fma(qp[-k - 1], w[k + 1], a1); }
                if (k < kn) a0 = fma(qp[-k], w[k], a0);
                accg += a0 + a1;
              }
            }
          }
          double tot = accg * T.x_mmI[t2][sq1][sp1] + acc1 * T.x_mm1nI[t2][sq1][sp1] + accb * (t > 2 ? xtau : 1.0);
          for (int k = (warp + c + d) % NW; k < 9; k += NW) {
            const int u1 = (0x322211100ull >> (4 * k)) & 15, u2l = (0x232121010ull >> (4 * k)) & 15;
            const int i = a - 1 - u1, j = bb + 1 + u2l;
            if (i < 1 || j > n) continue;
            const int to = bf_ptype_bases(S[i], S[j]);
            if (!to) continue;
            double ov = OB[BF_OROW(j - i) + i];
            if (to > 2) ov *= inv_tau;
            tot = fma(ov, bf_x_intloop(P, T, u1, u2l, to, t2, S[i + 1], S[j - 1], sp1, sq1) * scl[u1 + u2l + 2], tot);
          }
          if (kk < np) pi[a - 1] = tot;
        }
        // ---- the two multiloop sums of every cell, split over the warps by m
        for (int c = 0; c < ncell; c += 32) {
          const int cell = c + lane;
          const int a = min(cell, ncell - 1) + 1;
          double s1 = 0.0, s2 = 0.0;
          const int mmax = n - d - 1;  // the largest m any cell of this diagonal can use
#pragma unroll 4
          for (int m = 5 + warp; m <= mmax; m += NW) {
            const int oh = toff[d + m], oq = toff[m - 1];
            const bool v1 = a + d + m <= n, v2 = m <= a - 1;
            const double h1 = v1 ? H[oh + a - 1] : 0.0, x1 = v1 ? QM1[oq + a + d] : 0.0;
            const double h2 = v2 ? H[oh + a - m - 1] : 0.0, x2 = v2 ? QM[oq + a - m - 1] : 0.0;
            s1 = fma(h1, x1, s1);
            s2 = fma(h2, x2, s2);
          }
          if (cell < ncell) { p1[cell] = s1; p2[cell] = s2; }
        }
      }
      __syncthreads();
    }
    // ---- ensemble defect of target 0: (1/n) sum_i (paired ? 1 - P(i, pt i) : sum_j P(i,j))
    if (out_defect) {
      double e = 0.0;
      for (int i = 1 + tid; i <= n; i += blockDim.x) e += pt[i] ? 1.0 - ppair[i] : prow[i];
      e = bf_warp_sum(e);
      if (lane == 0) s_red[warp] = e;
      __syncthreads();
      if (tid == 0) {
        double tot = 0.0;
        for (int w = 0; w < NW; w++) tot += s_red[w];
        out_defect[sq] = (s_bad || n == 0) ? -1.0 : tot / n;
      }
    }
  }
}

// =====================================================================================================
//  Minimum-free-energy outside pass: for every pair (a,b) the lowest energy of the rest of a structure that contains it,
//  Cout(a,b), over the packed c / fML triangles of the MFE fill, so that E_pair(a,b) = C(a,b) + Cout(a,b).
//
//    Cout(a,b) = min { f5[a-1] + ext(a,b) + f3[b+1],                                          exterior loop
//                      Cout(i,j) + E_int(i,j;a,b)                      (a-i-1)+(j-b-1) <= 30,   enclosing interior loop
//                      mlstem(a,b) + min( A(a,b), min_i fML(i+1,a-1) + Hall(i,b) ) }          enclosing multiloop
//    G(i,j)    = Cout(i,j) + MLclosing + mlstem(closing (i,j))
//    Hm(i,b)   = min_j G(i,j) + fML(b+1,j-1)                           right of the stem: a multiloop segment
//    Hu(i,b)   = min(G(i,b+1), Hu(i,b+1) + MLbase)                     right of the stem: unpaired only
//    Hall      = min(Hm, Hu),   A(a,b) = min(Hm(a-1,b), A(a-1,b) + MLbase)   (left of the stem unpaired, right a segment)
//
//  The min-plus twin of the PF pass's row accumulators: every term is O(n) per cell, the pass O(n^3).  Cells are processed a
//  diagonal at a time from n-1 down to 4 (one barrier per diagonal), lanes on consecutive cells; the Cout, G and Hall triangles
//  live in the CTA's HBM workspace, Hm / Hu / A in two-diagonal rings on chip.  f5 / f3 are computed first by warps 0 and 1.
// =====================================================================================================
constexpr int kMoutNW = 8;

struct MoutPlan {
  int rs;
  size_t o_f5, o_f3, o_toff, o_hm, o_hu, o_ap, o_S, o_SP, total;
};
__host__ __device__ inline MoutPlan mout_plan(int nmax) {
  MoutPlan p;
  p.rs = (nmax + 8 + 3) / 4 * 4;
  size_t o = 0;
  p.o_f5 = o; o += (size_t)p.rs * sizeof(int);
  p.o_f3 = o; o += (size_t)p.rs * sizeof(int);
  p.o_toff = o; o += (size_t)p.rs * sizeof(int);
  p.o_hm = o; o += (size_t)2 * p.rs * sizeof(int);
  p.o_hu = o; o += (size_t)2 * p.rs * sizeof(int);
  p.o_ap = o; o += (size_t)2 * p.rs * sizeof(int);
  p.o_S = o; o += (nmax + 2 + 15) / 16 * 16;
  p.o_SP = o; o += (nmax + 2 + 15) / 16 * 16;
  p.total = o;
  return p;
}
// ints of per-CTA HBM workspace: the Cout, G and Hall triangles
__host__ __device__ inline size_t mout_ws_ints(int nmax) { return 3 * ((tri_size(nmax) + 7) / 8 * 8); }

__global__ void __launch_bounds__(kMoutNW * 32) bf_k_mfe_out(const BfParams *__restrict__ P, BfBatchDev b, const int *__restrict__ ctri,
                                                            const int *__restrict__ ftri, size_t tri_slot, int *ws, size_t ws_slot,
                                                            int *e_pair, int *work_counter) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  const MoutPlan pl = mout_plan(nmax);
  const int RS = pl.rs;
  const BfSmallI &T = P->si;
  int *f5 = reinterpret_cast<int *>(dyn + pl.o_f5);
  int *f3 = reinterpret_cast<int *>(dyn + pl.o_f3);
  int *toff = reinterpret_cast<int *>(dyn + pl.o_toff);
  int *HM = reinterpret_cast<int *>(dyn + pl.o_hm);
  int *HU = reinterpret_cast<int *>(dyn + pl.o_hu);
  int *AR = reinterpret_cast<int *>(dyn + pl.o_ap);
  uint8_t *S = dyn + pl.o_S, *SP = dyn + pl.o_SP;
  const size_t tri_pad = (tri_size(nmax) + 7) / 8 * 8;
  int *CO = ws + (size_t)blockIdx.x * ws_slot, *GT = CO + tri_pad, *HA = GT + tri_pad;
  const int mlbase = T.MLbase;

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int sq = s_seq;
    if (sq >= b.B) break;
    const int n = b.len[sq];
    const char *src = b.seq + (size_t)sq * b.stride;
    const uint8_t *np = b.nopair ? b.nopair + (size_t)sq * b.stride : nullptr;
    for (int k = tid; k <= n + 1; k += blockDim.x) {
      const uint8_t s = (uint8_t)((k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0);
      S[k] = s;
      SP[k] = (np && k >= 1 && k <= n && np[k - 1]) ? 0 : s;
    }
    for (int k = tid; k <= n; k += blockDim.x) toff[k] = (k >= 4) ? tri_off(n, k) : 0;
    for (int k = tid; k < 2 * RS; k += blockDim.x) { HM[k] = BF_INF; HU[k] = BF_INF; AR[k] = BF_INF; }
    int *out = e_pair + (size_t)sq * nmax * nmax;
    for (size_t k = tid; k < (size_t)nmax * nmax; k += blockDim.x) out[k] = BF_INF;
    const int *c = ctri + (size_t)sq * tri_slot, *fm = ftri + (size_t)sq * tri_slot;
    __syncthreads();
    auto ext = [&](int i, int j, int t) -> int { return bf_e_ext(T, t, (i > 1) ? S[i - 1] : -1, (j < n) ? S[j + 1] : -1); };
    // exterior prefix f5 (warp 0) and suffix f3 (warp 1)
    if (warp == 0) {
      if (lane == 0) f5[0] = 0;
      __syncwarp();
      for (int j = 1; j <= n; j++) {
        int e = BF_INF;
        for (int i = 1 + lane; i < j - BF_TURN; i += 32) {
          const int t = bf_ptype_bases(SP[i], SP[j]);
          const int cc = t ? c[toff[j - i] + i - 1] : BF_INF;
          if (cc < BF_INF) e = min(e, f5[i - 1] + cc + ext(i, j, t));
        }
        e = bf_warp_min(e);
        if (lane == 0) f5[j] = min(e, f5[j - 1]);
        __syncwarp();
      }
    } else if (warp == 1) {
      if (lane == 0) f3[n + 1] = 0;
      __syncwarp();
      for (int i = n; i >= 1; i--) {
        int e = BF_INF;
        for (int j = i + BF_TURN + 1 + lane; j <= n; j += 32) {
          const int t = bf_ptype_bases(SP[i], SP[j]);
          const int cc = t ? c[toff[j - i] + i - 1] : BF_INF;
          if (cc < BF_INF) e = min(e, cc + ext(i, j, t) + f3[j + 1]);
        }
        e = bf_warp_min(e);
        if (lane == 0) f3[i] = min(e, f3[i + 1]);
        __syncwarp();
      }
    }
    __syncthreads();

    for (int d = n - 1; d >= BF_TURN + 1; d--) {
      const int ncell = n - d;
      const int r0 = (d & 1) * RS, r1 = ((d + 1) & 1) * RS;
      for (int a = tid + 1; a <= ncell; a += blockDim.x) {
        const int bb = a + d;
        // Hm: the stem ends at bb, the closing pair (a, j) of its multiloop, fML(bb+1, j-1) between
        int hm = BF_INF;
        for (int m = 6; bb + m <= n; m++) {
          const int g = GT[toff[d + m] + a - 1], f = fm[toff[m - 2] + bb];
          hm = min(hm, g + f);
        }
        if (hm >= BF_INF) hm = BF_INF;
        int hu = BF_INF;
        if (bb < n) hu = min(GT[toff[d + 1] + a - 1], HU[r1 + a] + mlbase);
        if (hu >= BF_INF) hu = BF_INF;
        int ap = BF_INF;
        if (a > 1) ap = min(HM[r1 + a - 1], AR[r1 + a - 1] + mlbase);
        if (ap >= BF_INF) ap = BF_INF;
        const int o = toff[d] + a - 1;
        const int t = bf_ptype_bases(SP[a], SP[bb]);
        const int cab = t ? c[o] : BF_INF;
        int e = BF_INF;
        if (cab < BF_INF) {
          e = f5[a - 1] + ext(a, bb, t) + f3[bb + 1];
          // enclosing interior loops: outer pair (a-1-u1, bb+1+u2), s = u1 + u2
          const int t2 = bf_rtype(t), sp1 = S[a - 1], sq1 = S[bb + 1];
          const int smax = min(BF_MAXLOOP, n - 1 - d - 2);
          for (int s = 0; s <= smax; s++) {
            const int od = toff[d + 2 + s];
            for (int u1 = max(0, s - (n - bb - 1)); u1 <= min(s, a - 2); u1++) {
              const int i = a - 1 - u1, j = bb + 1 + s - u1;
              const int co = CO[od + i - 1];
              if (co >= BF_INF) continue;
              const int to = bf_ptype_bases(S[i], S[j]);
              e = min(e, co + bf_e_intloop(P, T, u1, s - u1, to, t2, S[i + 1], S[j - 1], sp1, sq1));
            }
          }
          // enclosing multiloops: left of the stem unpaired (A) or a segment fML(i+1, a-1)
          if (a > 1 && bb < n) {
            int ml = ap;
            for (int m = 6; m <= a - 1; m++) {
              const int i = a - m;
              ml = min(ml, fm[toff[m - 2] + i] + HA[toff[d + m] + i - 1]);
            }
            if (ml < BF_INF) e = min(e, ml + bf_e_mlstem(T, t, sp1, sq1));
          }
          if (e >= BF_INF) e = BF_INF;
        }
        CO[o] = e;
        GT[o] = e < BF_INF ? e + T.MLclosing + bf_e_mlstem(T, bf_rtype(t), S[bb - 1], S[a + 1]) : BF_INF;
        HA[o] = min(hm, hu);
        HM[r0 + a] = hm;
        HU[r0 + a] = hu;
        AR[r0 + a] = ap;
        if (e < BF_INF) out[(size_t)(a - 1) * nmax + (bb - 1)] = cab + e;
      }
      __syncthreads();
    }
  }
}

}  // namespace

// ---- host side: v2 whenever its plan fits the CTA's shared memory (generic ring on chip when that still leaves two CTAs per
// SM), else the first version
namespace {
// B = 0: the variant without the on-chip H / qm / qm1 tables (what sizes the workspace)
int out_version(int nmax, bool *rgs, bool *hsm, int B, int sms) {
  *hsm = false;
  // H / qm / qm1 of the sequence on chip as well: measured against reading them through L2 (profiles/r02_outside_hsm.txt) -- ahead
  // while two CTAs still share an SM (<= ~60 nt: 3-5 %) and for batches that leave SMs idle (B = 64: 0.96 -> 0.82 ms at 100 nt);
  // behind for big batches once it costs the second CTA (4096 x 100 nt: 16.2 against 11.3 ms).
  const bool want = B > 0 && (out2_plan(nmax, 8, true, true).total <= 113 * 1024 || B <= sms);
  if (want && out2_plan(nmax, 8, true, true).total <= kSmemBudget) { *rgs = true; *hsm = true; return 2; }
  if (out2_plan(nmax, 8, true).total <= 113 * 1024) { *rgs = true; return 2; }
  if (out2_plan(nmax, 8, false).total <= kSmemBudget) { *rgs = false; return 2; }
  return 1;
}

// bf_k_pf_out2 without and with the generic ring on chip, and with H / qm / qm1 on chip as well; then the same with KEEP
using OutK = void (*)(const BfParams *, BfBatchDev, const double *, const double *, size_t, double *, size_t, const double *, const char *, int,
                      int, double *, double *, int *, double *);
const OutK kOut2[] = {bf_k_pf_out2<8, false, false>, bf_k_pf_out2<8, true, false>, bf_k_pf_out2<8, true, true>,
                      bf_k_pf_out2<8, false, false, true>, bf_k_pf_out2<8, true, false, true>, bf_k_pf_out2<8, true, true, true>};
using Out1K = void (*)(const BfParams *, BfBatchDev, const double *, const double *, size_t, double *, const double *, const char *, int, int,
                       double *, double *, int *, double *);
const Out1K kOut1[] = {bf_k_pf_out<8>, bf_k_pf_out<8, true>};
}  // namespace

// key: 0 = bf_k_pf_out, else kOut2[key - 1]; + 4 with keep (the KEEP instantiation).  The workspace is sized for the variant without
// H on chip, so with it the slab is larger than it needs to be.
cudaError_t bf_plan_out(int stride, int B, int sms, BfPlan *p, bool keep) {
  *p = BfPlan{};
  bool rgs = false, hsm = false;
  p->ws = out_version(stride, &rgs, &hsm, 0, sms) == 2 ? (out2_ws_doubles(stride, rgs) + 7) / 8 * 8 : 4 * ((tri_size(stride) + 7) / 8 * 8);
  const void *kern;
  if (out_version(stride, &rgs, &hsm, B, sms) == 2) {
    p->key = 1 + rgs + hsm;
    p->smem = out2_plan(stride, 8, rgs, hsm).total;
    kern = (const void *)kOut2[p->key - 1 + (keep ? 3 : 0)];
  } else {
    p->key = 0;
    p->smem = out_plan(stride).total;
    kern = (const void *)kOut1[keep];
  }
  if (keep) p->key += 4;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(p->smem > 1024 ? p->smem : 1024));
  if (e != cudaSuccess) return e;
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, p->smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  p->grid = B < sms * occ ? B : sms * occ;
  return cudaSuccess;
}

cudaError_t bf_launch_pf_out(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *qmseq, double *ws,
                             const double *lnscale, const char *targets, int n_targets, int tstride, double *out_defect, double *out_bpp,
                             int *work_counter, cudaStream_t st, double *keep) {
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  const size_t tslot = (tri_size(b.stride) + 7) / 8 * 8;
  const int k = p.key & 3, kp = p.key >> 2;
  if (k == 0)
    kOut1[kp]<<<p.grid, 256, p.smem, st>>>(dP, b, qbtri, qmseq, tslot, ws, lnscale, targets, n_targets, tstride, out_defect, out_bpp,
                                           work_counter, keep);
  else
    kOut2[k - 1 + 3 * kp]<<<p.grid, 256, p.smem, st>>>(dP, b, qbtri, qmseq, tslot, ws, p.ws, lnscale, targets, n_targets, tstride, out_defect,
                                                      out_bpp, work_counter, keep);
  return cudaGetLastError();
}

cudaError_t bf_plan_mfe_out(int stride, int B, int sms, BfPlan *p) {
  *p = BfPlan{};
  p->ws = mout_ws_ints(stride);
  p->smem = mout_plan(stride).total;
  cudaError_t e = cudaFuncSetAttribute(bf_k_mfe_out, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(p->smem > 1024 ? p->smem : 1024));
  if (e != cudaSuccess) return e;
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bf_k_mfe_out, kMoutNW * 32, p->smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  p->grid = B < sms * occ ? B : sms * occ;
  return cudaSuccess;
}

cudaError_t bf_launch_mfe_out(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, const int *ctri, const int *ftri, int *ws, int *e_pair,
                              int *work_counter, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  bf_k_mfe_out<<<p.grid, kMoutNW * 32, p.smem, st>>>(dP, b, ctri, ftri, bf_tri_slot(b.stride), ws, p.ws, e_pair, work_counter);
  return cudaGetLastError();
}
