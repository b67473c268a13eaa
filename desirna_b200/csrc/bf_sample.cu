// bf_sample.cu -- stochastic backtracking: secondary structures drawn from the Boltzmann ensemble (sm_100a).
//
// ViennaRNA fc.pbacktrack() on the tables the partition-function fill leaves behind: the packed qb triangle, the per-sequence
// qm / qm1 triangles and the per-nucleotide scale lnscale.  The walk follows the unambiguous grammar the inside fill sums over
// (bf_k_pf_fill, bf_fill.cu), with the same loop weights and scale factors:
//
//   q5[j]    = q5[j-1] s + sum_i q5[i-1] qb(i,j) xExt(i,j)                              exterior loop, j unpaired or paired with i
//   qb(i,j)  = xHairpin s^(u+2) + sum_(p,q) qb(p,q) xInt s^(u1+u2+2)                  u1 + u2 <= 30
//              + xMLclosing s^2 xMLstem(closing) sum_u qm(i+1,u-1) qm1(u,j-1)
//   qm1(i,j) = sum_l qb(i,l) xMLstem(i,l) bu^(j-l)                                     bu = xMLbase s
//   qm(i,j)  = sum_u (bu^(u-i) + qm(i,u-1)) qm1(u,j)                                   left part empty or a multiloop segment
//
// (s = exp(-lnscale): every table carries the scale of the nucleotides it spans.)  Each decision draws r = U * (table value) and
// walks its candidates in chunks of 32 across the lanes of a warp: a warp prefix sum and a ballot find the first candidate whose
// running sum passes r.  If rounding leaves r past the last candidate, the last candidate with nonzero weight is taken.
//
// Work unit: one (sequence, sample) pair per warp, units in row-major order over a persistent grid, so one sequence with 10^4
// samples fills the GPU as well as 4096 sequences with one sample each.  Random numbers: one splitmix64 stream per
// (seed, row, sample index), seeded from those three alone -- the output does not depend on the grid, and the first k samples of a
// call with n > k samples are those of a call with k.
#include <algorithm>

#include "bf_kernels.h"

#include "bf_device.cuh"

namespace {

constexpr int kSampleWPB = 8;  // warps (samples in flight) per CTA; three CTAs per SM keep the walk within 85 registers, unspilled
constexpr int kQ5WPB = 4;      // warps (sequences) per CTA of the exterior prefix kernel

// pending segments of a walk: kind in bits 28..29, i in bits 14..27, j in bits 0..13 (stride <= 2000)
enum { kExt = 0, kPair = 1, kQm = 2, kQm1 = 3 };
__device__ __forceinline__ int seg(int kind, int i, int j) { return (kind << 28) | (i << 14) | j; }

__host__ __device__ inline size_t al16(size_t x) { return (x + 15) / 16 * 16; }
// Pending segments are disjoint intervals of >= 5 nucleotides each, also disjoint from the one being expanded: n/5 + 1 entries.
__host__ __device__ inline int stack_cap(int nmax) { return nmax / 5 + 2; }
// per warp: scale powers s^0..s^32, base codes S[0..n+1], the structure being drawn (stride + 1 chars), the segment stack
__host__ __device__ inline size_t sample_warp_bytes(int nmax) {
  return al16(33 * sizeof(double)) + al16(nmax + 2) + al16(nmax + 1) + al16((size_t)stack_cap(nmax) * sizeof(int));
}
__host__ __device__ inline size_t q5_warp_bytes(int nmax) { return al16((nmax + 1) * sizeof(double) + al16(nmax + 2)); }

// Index of the chosen candidate among ncand, weight(c) giving candidate c's weight; -1 only when every weight is zero.
template <typename F>
__device__ __forceinline__ int draw(int ncand, double r, F weight) {
  const int lane = threadIdx.x & 31;
  double run = 0.0;
  int last = -1;
  for (int base = 0; base < ncand; base += 32) {
    const int c = base + lane;
    const double w = c < ncand ? weight(c) : 0.0;
    double incl = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double v = __shfl_up_sync(BF_FULL, incl, o);
      if (lane >= o) incl += v;
    }
    const unsigned hit = __ballot_sync(BF_FULL, w > 0.0 && run + incl > r);
    if (hit) return base + __ffs(hit) - 1;
    const unsigned nz = __ballot_sync(BF_FULL, w > 0.0);
    if (nz) last = base + 31 - __clz(nz);
    run += __shfl_sync(BF_FULL, incl, 31);
  }
  return last;
}

// exterior prefix q5[0..n] of every sequence, one warp per sequence (the sum of bf_k_pf_ext, kept for the walk)
__global__ void __launch_bounds__(kQ5WPB * 32) bf_k_sample_q5(const BfParams *__restrict__ P, BfBatchDev b, const double *__restrict__ qbtri,
                                                             size_t tri_slot, const double *__restrict__ lnscale, double *q5_out) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallD T;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  bf_stage(&T, &P->sd);
  __syncthreads();
  const int sq = blockIdx.x * kQ5WPB + warp;
  if (sq >= b.B) return;
  double *q5 = reinterpret_cast<double *>(dyn + q5_warp_bytes(nmax) * warp);
  uint8_t *S = reinterpret_cast<uint8_t *>(q5 + (nmax + 1));
  const int n = b.len[sq];
  const char *src = b.seq + (size_t)sq * b.stride;
  for (int k = lane; k <= n + 1; k += 32) S[k] = (uint8_t)((k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0);
  const double sc1 = exp(-lnscale[sq]);
  const double *qb = qbtri + (size_t)sq * tri_slot;
  if (lane == 0) q5[0] = 1.0;
  __syncwarp();
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
  double *dst = q5_out + (size_t)sq * (nmax + 1);
  for (int k = lane; k <= n; k += 32) dst[k] = q5[k];
}

__global__ void __launch_bounds__(kSampleWPB * 32, 3) bf_k_sample(const BfParams *__restrict__ P, BfBatchDev b, const double *__restrict__ qbtri,
                                                              const double *__restrict__ qmseq, size_t tri_slot,
                                                              const double *__restrict__ lnscale, const double *__restrict__ q5all,
                                                              int n_samples, unsigned long long seed, char *ss_out) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallD T;
  __shared__ unsigned char s_loop[BF_NCAND][2];  // interior-loop candidate x: its size s = u1 + u2 and u1 (x = s(s+1)/2 + u1)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride;
  bf_stage(&T, &P->sd);
  for (int x = tid; x < BF_NCAND; x += blockDim.x) {
    int s = 0;
    while ((s + 1) * (s + 2) / 2 <= x) s++;
    s_loop[x][0] = (unsigned char)s;
    s_loop[x][1] = (unsigned char)(x - s * (s + 1) / 2);
  }
  __syncthreads();
  unsigned char *base = dyn + sample_warp_bytes(nmax) * warp;
  double *scl = reinterpret_cast<double *>(base);
  uint8_t *S = base + al16(33 * sizeof(double));
  char *ss = reinterpret_cast<char *>(S + al16(nmax + 2));
  int *stk = reinterpret_cast<int *>(ss + al16(nmax + 1));
  // units (row, k) in row-major order, warp w of the grid takes units w, w + step, ...; advanced without 64-bit division
  const int start = blockIdx.x * kSampleWPB + warp, step = gridDim.x * kSampleWPB;
  const int step_rows = step / n_samples, step_k = step % n_samples;
  int row_loaded = -1;
  for (int row = start / n_samples, k = start % n_samples; row < b.B;
       row += step_rows + ((unsigned)k + step_k >= (unsigned)n_samples),
           k = ((unsigned)k + step_k >= (unsigned)n_samples) ? (int)((unsigned)k + step_k - n_samples) : k + step_k) {
    const size_t unit = (size_t)row * n_samples + k;
    const int n = b.len[row];
    const double lns = lnscale[row];
    if (row != row_loaded) {
      const char *src = b.seq + (size_t)row * b.stride;
      for (int x = lane; x <= n + 1; x += 32) S[x] = (uint8_t)((x >= 1 && x <= n) ? bf_base_code(src[x - 1]) : 0);
      for (int x = lane; x <= 32; x += 32) scl[x] = exp(-lns * x);
      row_loaded = row;
    }
    for (int x = lane; x <= nmax; x += 32) ss[x] = x < n ? '.' : '\0';
    __syncwarp();
    const double *qb = qbtri + (size_t)row * tri_slot;
    const double *QM = qmseq + (size_t)row * 2 * tri_slot, *QM1 = QM + tri_slot;
    const double *q5 = q5all + (size_t)row * (nmax + 1);
    auto QB = [=](int i, int j) { return __ldg(qb + tri_off(n, j - i) + i - 1); };
    auto QMv = [=](int i, int j) { return __ldg(QM + tri_off(n, j - i) + i - 1); };
    auto QM1v = [=](int i, int j) { return __ldg(QM1 + tri_off(n, j - i) + i - 1); };
    const double lbu = log(T.x_MLbase) - lns;
    // the stream of (seed, row, sample): every lane holds the same state and draws the same numbers
    unsigned long long s0 = seed;
    unsigned long long s1 = sm64(s0) ^ (((unsigned long long)(unsigned)row << 32) | (unsigned)k);
    unsigned long long rs = sm64(s1);
    int top = 0;
    int cur = n > BF_TURN + 1 ? seg(kExt, 0, n) : -1;
    while (cur >= 0) {
      const int kind = cur >> 28, i = (cur >> 14) & 0x3fff, j = cur & 0x3fff;
      int next = -1;
      if (kind == kExt) {
        // candidate 0: j unpaired; candidate c >= 1: (j-3-c, j) paired
        const double r = u01(rs) * __ldg(q5 + j);
        const int bb = (j < n) ? S[j + 1] : -1;
        const int c = draw(j - BF_TURN, r, [=](int c) -> double {
          if (c == 0) return __ldg(q5 + j - 1) * scl[1];
          const int p = j - BF_TURN - c, t = bf_ptype_bases(S[p], S[j]);
          return t ? __ldg(q5 + p - 1) * QB(p, j) * bf_x_ext(T, t, (p > 1) ? S[p - 1] : -1, bb) : 0.0;
        });
        if (c > 0) {
          const int p = j - BF_TURN - c;
          if (p - 1 > BF_TURN + 1) { if (lane == 0) stk[top] = seg(kExt, 0, p - 1); top++; }
          next = seg(kPair, p, j);
        } else if (c == 0 && j - 1 > BF_TURN + 1) {
          next = seg(kExt, 0, j - 1);
        }
      } else if (kind == kPair) {
        if (lane == 0) { ss[i - 1] = '('; ss[j - 1] = ')'; }
        // candidate 0: hairpin; 1..BF_NCAND: interior loop (u1, u2) with s = u1 + u2, index s(s+1)/2 + u1; then multiloop splits u
        const int t = bf_ptype_bases(S[i], S[j]);
        const double r = u01(rs) * QB(i, j);
        const int nml = max(0, j - i - 10);   // u = i+6 .. j-5
        const double xml = T.x_MLclosing * scl[2] * bf_x_mlstem(T, bf_rtype(t), S[j - 1], S[i + 1]);
        const int c = draw(1 + BF_NCAND + nml, r, [=](int c) -> double {
          if (c == 0) return bf_x_hairpin(P, T, S, i, j, t) * (j - i + 1 <= 32 ? scl[j - i + 1] : exp(-lns * (j - i + 1)));
          if (c <= BF_NCAND) {
            const int s = s_loop[c - 1][0], u1 = s_loop[c - 1][1], u2 = s - u1;
            const int p = i + 1 + u1, q = j - 1 - u2;
            if (q - p <= BF_TURN) return 0.0;
            const int tpq = bf_ptype_bases(S[p], S[q]);
            if (!tpq) return 0.0;
            return QB(p, q) * bf_x_intloop(P, T, u1, u2, t, bf_rtype(tpq), S[i + 1], S[j - 1], S[p - 1], S[q + 1]) * scl[s + 2];
          }
          const int u = i + 6 + (c - 1 - BF_NCAND);
          return QMv(i + 1, u - 1) * QM1v(u, j - 1) * xml;
        });
        if (c > BF_NCAND) {
          const int u = i + 6 + (c - 1 - BF_NCAND);
          if (lane == 0) stk[top] = seg(kQm, i + 1, u - 1);
          top++;
          next = seg(kQm1, u, j - 1);
        } else if (c > 0) {
          const int s = s_loop[c - 1][0], u1 = s_loop[c - 1][1];
          next = seg(kPair, i + 1 + u1, j - 1 - (s - u1));
        }
      } else if (kind == kQm1) {
        // candidate c: stem (i, j-c), c unpaired bases right of it
        const double r = u01(rs) * QM1v(i, j);
        const int c = draw(j - i - BF_TURN, r, [=](int c) -> double {
          const int l = j - c, t = bf_ptype_bases(S[i], S[l]);
          return t ? QB(i, l) * bf_x_mlstem(T, t, S[i - 1], S[l + 1]) * exp(lbu * c) : 0.0;
        });
        if (c >= 0) next = seg(kPair, i, j - c);
      } else {
        // candidate 2m: stem segment qm1(i+m, j) with the m bases left of it unpaired; 2m+1: with a multiloop segment qm(i, i+m-1)
        const double r = u01(rs) * QMv(i, j);
        const int c = draw(2 * (j - i - BF_TURN), r, [=](int c) -> double {
          const int u = i + (c >> 1);
          if (c & 1) return (u - 1 - i > BF_TURN) ? QMv(i, u - 1) * QM1v(u, j) : 0.0;
          return exp(lbu * (u - i)) * QM1v(u, j);
        });
        if (c >= 0) {
          const int u = i + (c >> 1);
          if (c & 1) { if (lane == 0) stk[top] = seg(kQm, i, u - 1); top++; }
          next = seg(kQm1, u, j);
        }
      }
      __syncwarp();
      if (next < 0 && top > 0) next = stk[--top];
      cur = next;
    }
    __syncwarp();
    char *dst = ss_out + (size_t)unit * (nmax + 1);
    for (int x = lane; x <= nmax; x += 32) dst[x] = ss[x];
    __syncwarp();
  }
}

template <typename K>
cudaError_t smem_attr(K kern, size_t sm) {
  return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sm > 1024 ? sm : 1024));
}

}  // namespace

cudaError_t bf_launch_sample(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *qmseq, const double *lnscale, double *q5,
                             int n_samples, unsigned long long seed, char *ss_out, int sms, cudaStream_t st) {
  const size_t slot = bf_tri_slot(b.stride);
  const size_t smq = q5_warp_bytes(b.stride) * kQ5WPB;
  cudaError_t e = smem_attr(bf_k_sample_q5, smq);
  if (e != cudaSuccess) return e;
  bf_k_sample_q5<<<(b.B + kQ5WPB - 1) / kQ5WPB, kQ5WPB * 32, smq, st>>>(dP, b, qbtri, slot, lnscale, q5);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  const size_t sm = sample_warp_bytes(b.stride) * kSampleWPB;
  if ((e = smem_attr(bf_k_sample, sm)) != cudaSuccess) return e;
  int occ = 0;
  if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bf_k_sample, kSampleWPB * 32, sm)) != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  const long long units = (long long)b.B * n_samples, need = (units + kSampleWPB - 1) / kSampleWPB;
  const int grid = (int)std::min<long long>(need, (long long)occ * sms);
  bf_k_sample<<<grid, kSampleWPB * 32, sm, st>>>(dP, b, qbtri, qmseq, slot, lnscale, q5, n_samples, seed, ss_out);
  return cudaGetLastError();
}
