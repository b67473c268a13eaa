// bf_unpaired.cu -- accessibility (sm_100a): probabilities that stretches of a strand are entirely unpaired (RNAplfold -u), and
// RNAplfold's window averages of them and of the pair probabilities.
//
// bf_k_unpaired reads finished tables only: qb, qm1 of the PF fill, the outside triangles the outside pass keeps (bqb, bqm and
// out1 = qm1's outside value without its bu * bqm1(a,b+1) self-recursion, bf_outside.cu) and lnscale.  With dangles = 2 an
// unpaired nucleotide's weight does not depend on its neighbours, so the probability of stretch [i,j] splits by the loop that holds
// it.  Every loop other than the exterior one holds its unpaired nucleotides in maximal runs [a,b] bounded by paired bases, and in
// the grammar of bf_k_pf_fill (header of bf_sample.cu) each run is produced exactly once:
//
//   hairpin (a-1, b+1)                 bqb(a-1,b+1) xHairpin s^(b-a+3)
//   interior loop, left gap            sum  bqb(a-1,q) xInt qb(b+1,l) s^(g+h+2)        q = l+1+h, g + h <= 30
//   interior loop, right gap           sum  bqb(p,b+1) xInt qb(k,a-1) s^(g+h+2)        p = k-1-h
//   multiloop, after a stem (u, a-1)   sum_u out1(u,b) qb(u,a-1) xMLstem(u,a-1) bu^g  qm1(u,b): the stem, then the run
//   multiloop, first run (a-1 closes)  sum_j bqm(a,j) qm1(b+1,j) bu^g                   qm(a,j) starting with the run
//
// (g = b-a+1, bu = xMLbase s, s = exp(-lnscale).)  Their sum R(a,b) is the probability that [a,b] is such a run, and
//
//   P_u(i, j-i+1) = q5[i-1] s^(j-i+1) q3[j+1] / Z  +  sum_{a <= i, b >= j} R(a,b)
//
// the dominance sum taken by a suffix scan along b and a prefix scan along a.  Work per sequence: O(n^3) for the multiloop sums
// and ~2 x 496 n^2 interior-loop candidates, the interior term of the outside pass.  Mapping: one persistent 8-warp CTA per
// sequence; R is a dense n x n table in the CTA's HBM workspace; threads take runs for the O(n) sums, a warp takes a run of at
// most 30 nt for its interior-loop candidates, threads take rows / columns for the scans.
#include <algorithm>

#include "bf_kernels.h"

#include "bf_device.cuh"

namespace {

constexpr int kUpNW = 8;

struct UpPlan {
  size_t o_scl, o_q5, o_q3, o_toff, o_S, total;
};
__host__ __device__ inline UpPlan up_plan(int nmax) {
  UpPlan p;
  const size_t rs = (nmax + 8 + 3) / 4 * 4;
  size_t o = 0;
  p.o_scl = o; o += rs * sizeof(double);
  p.o_q5 = o; o += rs * sizeof(double);
  p.o_q3 = o; o += rs * sizeof(double);
  p.o_toff = o; o += rs * sizeof(int);
  p.o_S = o; o += (nmax + 2 + 15) / 16 * 16;
  p.total = o;
  return p;
}

__global__ void __launch_bounds__(kUpNW * 32) bf_k_unpaired(const BfParams *__restrict__ P, BfBatchDev b, const double *__restrict__ qbtri,
                                                           const double *__restrict__ qmseq, const double *__restrict__ keep, size_t tri_slot,
                                                           const double *__restrict__ lnscale, double *ws, size_t ws_slot, int max_u,
                                                           double *pu_out, int *work_counter) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ int s_seq;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  const UpPlan pl = up_plan(nmax);
  const BfSmallD &T = P->sd;
  double *scl = reinterpret_cast<double *>(dyn + pl.o_scl);
  double *q5 = reinterpret_cast<double *>(dyn + pl.o_q5);
  double *q3 = reinterpret_cast<double *>(dyn + pl.o_q3);
  int *toff = reinterpret_cast<int *>(dyn + pl.o_toff);
  uint8_t *S = dyn + pl.o_S;
  double *R = ws + (size_t)blockIdx.x * ws_slot;

  for (;;) {
    __syncthreads();
    if (tid == 0) s_seq = atomicAdd(work_counter, 1);
    __syncthreads();
    const int sq = s_seq;
    if (sq >= b.B) break;
    const int n = b.len[sq];
    const char *src = b.seq + (size_t)sq * b.stride;
    const double lns = lnscale[sq];
    for (int k = tid; k <= n + 1; k += blockDim.x) S[k] = (uint8_t)((k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0);
    for (int k = tid; k <= n; k += blockDim.x) toff[k] = (k >= 4) ? tri_off(n, k) : 0;
    for (int k = tid; k <= n + 2; k += blockDim.x) scl[k] = exp(-lns * k);
    __syncthreads();
    const double *qb = qbtri + (size_t)sq * tri_slot;
    const double *QM1 = qmseq + (size_t)sq * 2 * tri_slot + tri_slot;
    const double *KB = keep + (size_t)sq * 3 * tri_slot, *KM = KB + tri_slot, *K1 = KM + tri_slot;
    const double lbu = log(T.x_MLbase) - lns, sc1 = scl[1];
    auto at = [&](int i, int j) { return toff[j - i] + i - 1; };
    auto xext = [&](int i, int j, int t) -> double { return bf_x_ext(T, t, (i > 1) ? S[i - 1] : -1, (j < n) ? S[j + 1] : -1); };
    // exterior chains q5 (warp 0) and q3 (warp 1), as in the outside pass
    if (warp == 0) {
      if (lane == 0) q5[0] = 1.0;
      __syncwarp();
      for (int j = 1; j <= n; j++) {
        double sum = 0.0;
        for (int i = 1 + lane; i < j - BF_TURN; i += 32) {
          const int t = bf_ptype_bases(S[i], S[j]);
          if (t) sum += q5[i - 1] * qb[at(i, j)] * xext(i, j, t);
        }
        sum = bf_warp_sum(sum);
        if (lane == 0) q5[j] = sum + q5[j - 1] * sc1;
        __syncwarp();
      }
    } else if (warp == 1) {
      if (lane == 0) q3[n + 1] = 1.0;
      __syncwarp();
      for (int i = n; i >= 1; i--) {
        double sum = 0.0;
        for (int j = i + BF_TURN + 1 + lane; j <= n; j += 32) {
          const int t = bf_ptype_bases(S[i], S[j]);
          if (t) sum += qb[at(i, j)] * xext(i, j, t) * q3[j + 1];
        }
        sum = bf_warp_sum(sum);
        if (lane == 0) q3[i] = sum + q3[i + 1] * sc1;
        __syncwarp();
      }
    }
    // ---- R(a,b), a <= b: hairpins and multiloop runs, one run per thread
    for (int idx = tid; idx < n * n; idx += blockDim.x) {
      const int a = idx / n + 1, bb = idx % n + 1;
      if (bb < a) continue;
      const int p = a - 1, q = bb + 1;
      double r = 0.0;
      if (p >= 1) {
        if (q <= n && q - p > BF_TURN) {
          const int t = bf_ptype_bases(S[p], S[q]);
          if (t) r = KB[at(p, q)] * bf_x_hairpin(P, T, S, p, q, t) * scl[q - p + 1];
        }
        double ml = 0.0;
        for (int u = 1; u + BF_TURN < p; u++) {   // after the stem (u, p) of segment qm1(u, bb)
          const int t = bf_ptype_bases(S[u], S[p]);
          if (t) ml += K1[at(u, bb)] * qb[at(u, p)] * bf_x_mlstem(T, t, S[u - 1], S[p + 1]);
        }
        for (int j = q + BF_TURN + 1; j <= n; j++) ml += KM[at(a, j)] * QM1[at(q, j)];   // first run of qm(a, j)
        r += ml * exp(lbu * (bb - a + 1));
      }
      R[idx] = r;
    }
    __syncthreads();
    // ---- interior-loop gaps: a warp per run [a, a+g-1] of g <= 30 nt, lanes over the other side's candidates
    for (int it = warp; it < n * BF_MAXLOOP; it += kUpNW) {
      const int a = it / BF_MAXLOOP + 1, g = it % BF_MAXLOOP + 1, bb = a + g - 1;
      if (bb > n) continue;
      double acc = 0.0;
      const int p = a - 1, k = bb + 1;   // left gap: outer (p, q), inner (k, l), h = q-l-1
      if (p >= 1 && k <= n) {
        for (int h = 0; g + h <= BF_MAXLOOP; h++)
          for (int l = k + BF_TURN + 1 + lane; l + 1 + h <= n; l += 32) {
            const int q = l + 1 + h;
            const int to = bf_ptype_bases(S[p], S[q]), ti = bf_ptype_bases(S[k], S[l]);
            if (to && ti)
              acc += KB[at(p, q)] * qb[at(k, l)] * bf_x_intloop(P, T, g, h, to, bf_rtype(ti), S[p + 1], S[q - 1], S[k - 1], S[l + 1]) *
                     scl[g + h + 2];
          }
      }
      const int l0 = a - 1, q0 = bb + 1;   // right gap: inner (kk, l0), outer (pp, q0), h = kk-pp-1
      if (l0 >= 1 && q0 <= n) {
        for (int h = 0; g + h <= BF_MAXLOOP; h++)
          for (int kk = h + 2 + lane; kk + BF_TURN < l0; kk += 32) {
            const int pp = kk - 1 - h;
            const int to = bf_ptype_bases(S[pp], S[q0]), ti = bf_ptype_bases(S[kk], S[l0]);
            if (to && ti)
              acc += KB[at(pp, q0)] * qb[at(kk, l0)] * bf_x_intloop(P, T, h, g, to, bf_rtype(ti), S[pp + 1], S[q0 - 1], S[kk - 1], S[l0 + 1]) *
                     scl[g + h + 2];
          }
      }
      acc = bf_warp_sum(acc);
      if (lane == 0) R[(size_t)(a - 1) * n + bb - 1] += acc;
    }
    __syncthreads();
    // ---- dominance sums: suffix along b (a row per thread), then prefix along a (a column per thread)
    for (int a = tid + 1; a <= n; a += blockDim.x) {
      double *row = R + (size_t)(a - 1) * n;
      double acc = 0.0;
      for (int bb = n; bb >= a; bb--) { acc += row[bb - 1]; row[bb - 1] = acc; }
    }
    __syncthreads();
    for (int j = tid + 1; j <= n; j += blockDim.x) {
      double acc = 0.0;
      for (int a = 1; a <= j; a++) { acc += R[(size_t)(a - 1) * n + j - 1]; R[(size_t)(a - 1) * n + j - 1] = acc; }
    }
    __syncthreads();
    const double invZ = 1.0 / q5[n];
    double *out = pu_out + (size_t)sq * nmax * max_u;
    for (int idx = tid; idx < n * max_u; idx += blockDim.x) {
      const int i = idx / max_u + 1, u = idx % max_u + 1, j = i + u - 1;
      double v = 0.0;
      if (j <= n) v = fmin(1.0, fmax(0.0, q5[i - 1] * scl[u] * q3[j + 1] * invZ + R[(size_t)(i - 1) * n + j - 1]));
      out[idx] = v;
    }
  }
}

// RNAplfold averages (bf_kernels.h, BfPlfoldDev): blockIdx.y over the strands of the chunk, threads over a strand's output elements
__global__ void __launch_bounds__(256) bf_k_plfold_avg(BfPlfoldDev d, const double *__restrict__ qbtri, const double *__restrict__ keep,
                                                       size_t tri_slot, const double *__restrict__ pu, double *bpp_acc, double *pu_acc) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  for (int r = d.r0 + blockIdx.y; r < d.r1; r += gridDim.y) {
    const int n = d.len[r], W = d.wlen[r], nwin = n > 0 ? n - W + 1 : 0;
    const long long g0 = d.win0[r];   // global index of window s = 1
    const int c_lo = (int)max(1LL, d.w0 - g0 + 1), c_hi = (int)min((long long)nwin, d.w0 + d.nw - g0);
    if (c_lo > c_hi) continue;
    // stretch or pair [i, j]: windows s = max(1, j-W+1) .. min(i, nwin) hold it; this chunk adds those in c_lo .. c_hi
    auto span = [&](int i, int j, int *lo, int *hi, int *s_lo, int *s_hi) {
      *s_lo = max(1, j - W + 1); *s_hi = min(i, nwin);
      *lo = max(*s_lo, c_lo); *hi = min(*s_hi, c_hi);
    };
    if (bpp_acc && x < n * d.winsize) {
      const int i = x / d.winsize + 1, dd = x % d.winsize, j = i + dd;
      int lo, hi, s_lo, s_hi;
      span(i, j, &lo, &hi, &s_lo, &s_hi);
      if (dd > BF_TURN && j <= n && dd < W && lo <= hi) {
        double *e = bpp_acc + ((size_t)r * d.stride + i - 1) * d.winsize + dd;
        double acc = *e;
        const int o = tri_off(W, dd) + i - 1;
        for (int s = lo; s <= hi; s++) {
          const size_t row = (size_t)(g0 + s - 1 - d.w0);
          acc += keep[row * 3 * tri_slot + o - (s - 1)] * qbtri[row * tri_slot + o - (s - 1)];
        }
        if (hi == s_hi) acc /= (double)(s_hi - s_lo + 1);
        *e = acc;
      }
    }
    if (pu_acc && x < n * d.max_u) {
      const int i = x / d.max_u + 1, u = x % d.max_u + 1, j = i + u - 1;
      int lo, hi, s_lo, s_hi;
      span(i, j, &lo, &hi, &s_lo, &s_hi);
      if (j <= n && lo <= hi) {
        double *e = pu_acc + ((size_t)r * d.stride + i - 1) * d.max_u + u - 1;
        double acc = *e;
        for (int s = lo; s <= hi; s++) {
          const size_t row = (size_t)(g0 + s - 1 - d.w0);
          acc += pu[(row * d.wstride + (i - s)) * d.max_u + u - 1];
        }
        if (hi == s_hi) acc /= (double)(s_hi - s_lo + 1);
        *e = acc;
      }
    }
  }
}

}  // namespace

size_t bf_unpaired_ws_bytes(int stride) { return (size_t)stride * stride * sizeof(double); }

cudaError_t bf_launch_unpaired(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *qmseq, const double *keep,
                               const double *lnscale, double *ws, size_t ws_bytes, int max_u, double *pu_out, int *work_counter, int sms,
                               cudaStream_t st) {
  const size_t sm = up_plan(b.stride).total, slot = bf_unpaired_ws_bytes(b.stride) / sizeof(double);
  cudaError_t e = cudaFuncSetAttribute(bf_k_unpaired, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sm > 1024 ? sm : 1024));
  if (e != cudaSuccess) return e;
  int occ = 0;
  if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bf_k_unpaired, kUpNW * 32, sm)) != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  const long long grid = std::min<long long>({(long long)b.B, (long long)occ * sms, (long long)(ws_bytes / (slot * sizeof(double)))});
  if (grid < 1) return cudaErrorInvalidValue;
  if ((e = cudaMemsetAsync(work_counter, 0, sizeof(int), st)) != cudaSuccess) return e;
  bf_k_unpaired<<<(int)grid, kUpNW * 32, sm, st>>>(dP, b, qbtri, qmseq, keep, bf_tri_slot(b.stride), lnscale, ws, slot, max_u, pu_out,
                                                   work_counter);
  return cudaGetLastError();
}

cudaError_t bf_launch_plfold_avg(const BfPlfoldDev &d, const double *qbtri, const double *keep, const double *pu, double *bpp_acc,
                                 double *pu_acc, cudaStream_t st) {
  const int per = d.stride * std::max(bpp_acc ? d.winsize : 0, pu_acc ? d.max_u : 0);
  const dim3 grid((per + 255) / 256, std::min(d.r1 - d.r0, 65535));
  if (grid.x == 0 || grid.y == 0) return cudaSuccess;
  bf_k_plfold_avg<<<grid, 256, 0, st>>>(d, qbtri, keep, bf_tri_slot(d.wstride), pu, bpp_acc, pu_acc);
  return cudaGetLastError();
}
