// bf_ext.cu -- exterior-loop recursions for SMALL batches: one CTA per sequence (sm_100a).
//
//   f5[j] = min(f5[j-1], min_i f5[i-1] + c(i,j) + Ext(i,j))            (the tail of fc.mfe(), utils/energy_scores.py:150 in the reference)
//   q5[j] = q5[j-1] scale + sum_i q5[i-1] qb(i,j) xExt(i,j)            (the tail of fc.pf(),  utils/energy_scores.py:151; SURVEY.md A.4 / A.6)
//
// bf_k_trace / bf_k_pf_ext (bf_fill.cu) give a sequence ONE WARP, which is the right shape for thousands of sequences; with a
// replica-exchange sub-step's handful of long sequences the warp walks n^2/2 table entries of a diagonal-major table column by
// column (every load its own cache line, every column an L2 round trip): 1.2 ms at 400 nt, more than the cluster fill kernels
// (bf_cluster.cu) need for the whole table.  Here a CTA takes one sequence: all warps TRANSPOSE 32 (MFE) / 16 (PF) columns at a
// time into shared memory -- for a fixed diagonal the cells of 32 neighbouring columns are 32 neighbouring table entries, so the
// reads are coalesced -- with the exterior-stem term already added (multiplied) in, and warp 0 runs the serial recursion on the
// previous tile meanwhile.  Results: f5 for bf_k_trace (which then only backtracks), the ensemble energies for the caller.
#include "bf_kernels.h"

#include <cstdlib>

#include "bf_device.cuh"

namespace {

constexpr int kExtNW = 8;

// tile row stride: even (so that consecutive lanes, which sit one row and one column apart, hit different banks)
__host__ __device__ __forceinline__ int ext_ts(int nmax) { return (nmax + 4) / 2 * 2 + 2; }

template <int NW, int JB>
__global__ void __launch_bounds__(NW * 32) bf_k_f5_wide(const BfParams *__restrict__ P, BfBatchDev b, const int *__restrict__ ctri, size_t tri_slot,
                                                        int *f5_out) {
  extern __shared__ __align__(16) unsigned char dyn[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride, TS = ext_ts(nmax);
  int *tile = reinterpret_cast<int *>(dyn);                       // [2][JB][TS]
  int *f5 = tile + 2 * JB * TS;                                   // [nmax + 4]
  uint8_t *S = reinterpret_cast<uint8_t *>(f5 + nmax + 4);
  uint8_t *SP = S + (nmax + 2 + 15) / 16 * 16;
  const BfSmallI &T = P->si;
  const int sq = blockIdx.x;
  const int n = b.len[sq];
  {
    const char *src = b.seq + (size_t)sq * b.stride;
    const uint8_t *np = b.nopair ? b.nopair + (size_t)sq * b.stride : nullptr;
    for (int k = tid; k <= n + 1; k += blockDim.x) {
      const int code = (k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0;
      S[k] = (uint8_t)code;
      SP[k] = (uint8_t)((np && k >= 1 && k <= n && np[k - 1]) ? 0 : code);
    }
    if (tid == 0) f5[0] = 0;
  }
  __syncthreads();
  const int *c = ctri + (size_t)sq * tri_slot;
  // columns j0 .. j0+JB-1 into tile buffer bf: nw warps starting at w0 share the diagonals, lane = column; the table reads of
  // eight diagonals are issued before any of them is used (the kernel is L2-latency-bound otherwise)
  auto fill = [&](int j0, int bf, int w0, int nw) {
    int *tl = tile + bf * JB * TS;
    const int j = j0 + lane;
    const bool jin = lane < JB && j <= n;
    const int sj = jin ? SP[j] : 0, bb = (jin && j < n) ? S[j + 1] : -1;
    const int dmax = min(n - 1, j0 + JB - 2);
    for (int d0 = BF_TURN + 1 + (warp - w0); d0 <= dmax; d0 += 8 * nw) {
      int cc[8], tt[8];
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int d = d0 + k * nw, i = j - d;
        tt[k] = (jin && d <= dmax && i >= 1) ? bf_ptype_bases(SP[i], sj) : 0;
        cc[k] = tt[k] ? __ldg(c + tri_off(n, d) + i - 1) : BF_INF;
      }
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int d = d0 + k * nw, i = j - d;
        if (jin && d <= dmax && i >= 1) {
          int v = BF_INF;
          if (tt[k] && cc[k] < BF_INF) v = cc[k] + bf_e_ext(T, tt[k], (i > 1) ? S[i - 1] : -1, bb);
          tl[lane * TS + i] = v;
        }
      }
    }
  };
  fill(1, 0, 0, NW);
  __syncthreads();
  int bf = 0;
  for (int j0 = 1; j0 <= n; j0 += JB, bf ^= 1) {
    if (warp == 0) {
      const int *tl = tile + bf * JB * TS;
      for (int jj = 0; jj < JB && j0 + jj <= n; jj++) {
        const int j = j0 + jj;
        int e0 = BF_INF, e1 = BF_INF;
        const int *row = tl + jj * TS;
        int i = 1 + lane;
        for (; i + 32 < j - BF_TURN; i += 64) { e0 = min(e0, f5[i - 1] + row[i]); e1 = min(e1, f5[i + 31] + row[i + 32]); }
        if (i < j - BF_TURN) e0 = min(e0, f5[i - 1] + row[i]);
        const int e = bf_warp_min(min(e0, e1));
        if (lane == 0) f5[j] = min(e, f5[j - 1]);
        __syncwarp();
      }
    } else if (j0 + JB <= n) {
      fill(j0 + JB, bf ^ 1, 1, NW - 1);   // the other warps transpose the next columns meanwhile
    }
    __syncthreads();
  }
  for (int k = tid; k <= n; k += blockDim.x) f5_out[(size_t)sq * (nmax + 4) + k] = f5[k];
}

template <int NW, int JB>
__global__ void __launch_bounds__(NW * 32) bf_k_q5_wide(const BfParams *__restrict__ P, BfBatchDev b, const double *__restrict__ qbtri, size_t tri_slot,
                                                        const double *__restrict__ lnscale, double *out5) {
  extern __shared__ __align__(16) unsigned char dyn[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = b.stride, TS = ext_ts(nmax);
  double *tile = reinterpret_cast<double *>(dyn);                 // [2][JB][TS]
  double *q5 = tile + 2 * JB * TS;                                // [nmax + 4]
  uint8_t *S = reinterpret_cast<uint8_t *>(q5 + nmax + 4);
  const BfSmallD &T = P->sd;
  const int sq = blockIdx.x;
  const int n = b.len[sq];
  {
    const char *src = b.seq + (size_t)sq * b.stride;
    for (int k = tid; k <= n + 1; k += blockDim.x) S[k] = (uint8_t)((k >= 1 && k <= n) ? bf_base_code(src[k - 1]) : 0);
    if (tid == 0) q5[0] = 1.0;
  }
  __syncthreads();
  const double lns = lnscale[sq], sc1 = exp(-lns);
  const double *qb = qbtri + (size_t)sq * tri_slot;
  // two diagonals per pass (JB = 16 columns per tile: lanes 0..15 one diagonal, 16..31 the next); the table reads of eight passes
  // are issued before any of them is used
  auto fill2 = [&](int j0, int bf, int w0, int nw) {
    double *tl = tile + bf * JB * TS;
    const int col = lane & (JB - 1), half = lane / JB;
    const int j = j0 + col;
    const bool jin = j <= n;
    const int sj = jin ? S[j] : 0, bb = (jin && j < n) ? S[j + 1] : -1;
    const int dmax = min(n - 1, j0 + JB - 2);
    for (int d0 = BF_TURN + 1 + 2 * (warp - w0) + half; d0 <= dmax; d0 += 16 * nw) {
      double q[8];
      int tt[8];
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int d = d0 + 2 * k * nw, i = j - d;
        tt[k] = (jin && d <= dmax && i >= 1) ? bf_ptype_bases(S[i], sj) : 0;
        q[k] = tt[k] ? __ldg(qb + tri_off(n, d) + i - 1) : 0.0;
      }
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int d = d0 + 2 * k * nw, i = j - d;
        if (jin && d <= dmax && i >= 1) tl[col * TS + i] = tt[k] ? q[k] * bf_x_ext(T, tt[k], (i > 1) ? S[i - 1] : -1, bb) : 0.0;
      }
    }
  };
  fill2(1, 0, 0, NW);
  __syncthreads();
  int bf = 0;
  for (int j0 = 1; j0 <= n; j0 += JB, bf ^= 1) {
    if (warp == 0) {
      const double *tl = tile + bf * JB * TS;
      for (int jj = 0; jj < JB && j0 + jj <= n; jj++) {
        const int j = j0 + jj;
        double s0 = 0.0, s1 = 0.0;
        const double *row = tl + jj * TS;
        int i = 1 + lane;
        for (; i + 32 < j - BF_TURN; i += 64) { s0 = fma(q5[i - 1], row[i], s0); s1 = fma(q5[i + 31], row[i + 32], s1); }
        if (i < j - BF_TURN) s0 = fma(q5[i - 1], row[i], s0);
        const double sum = bf_warp_sum(s0 + s1);
        if (lane == 0) q5[j] = sum + q5[j - 1] * sc1;
        __syncwarp();
      }
    } else if (j0 + JB <= n) {
      fill2(j0 + JB, bf ^ 1, 1, NW - 1);
    }
    __syncthreads();
  }
  if (tid == 0 && out5) {
    double *o = out5 + (size_t)sq * 5;
    o[0] = o[1] = o[2] = o[3] = 0.0;
    o[4] = (n > 0) ? -T.kT * (log(q5[n]) + n * lns) / 1000.0 : 0.0;
  }
}

size_t f5_smem(int nmax, int jb) { return ((size_t)2 * jb * ext_ts(nmax) + nmax + 4) * sizeof(int) + 2 * ((nmax + 2 + 15) / 16 * 16); }
size_t q5_smem(int nmax, int jb) { return ((size_t)2 * jb * ext_ts(nmax) + nmax + 4) * sizeof(double) + (nmax + 2 + 15) / 16 * 16; }
constexpr size_t kExtSmemMax = 200 * 1024;

}  // namespace

// lengths the wide exterior kernels cover (tile in shared memory)
bool bf_ext_wide_ok(int nmax) { return nmax >= 1 && f5_smem(nmax, 32) <= kExtSmemMax && q5_smem(nmax, 16) <= kExtSmemMax; }

cudaError_t bf_launch_f5_wide(const BfParams *dP, const BfBatchDev &b, const int *ctri, int *f5_out, cudaStream_t st) {
  auto kern = bf_k_f5_wide<kExtNW, 32>;
  const size_t sm = f5_smem(b.stride, 32);
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kExtSmemMax);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  kern<<<b.B, kExtNW * 32, sm, st>>>(dP, b, ctri, bf_tri_slot(b.stride), f5_out);
  return cudaGetLastError();
}

cudaError_t bf_launch_q5_wide(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *lnscale, double *out5, cudaStream_t st) {
  auto kern = bf_k_q5_wide<kExtNW, 16>;
  const size_t sm = q5_smem(b.stride, 16);
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kExtSmemMax);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  kern<<<b.B, kExtNW * 32, sm, st>>>(dP, b, qbtri, bf_tri_slot(b.stride), lnscale, out5);
  return cudaGetLastError();
}
