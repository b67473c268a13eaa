// bf_interact.cu -- accessibility-aware RNA-RNA interaction (RNAup / RNAplex -a / IntaRNA's site model) on the device (sm_100a).
//
// A site of strands a and b is a duplex chain as in bf_duplex.cu, pairs (k1,l1), ..., (km,lm), k increasing, l decreasing, at most
// 30 unpaired nucleotides between consecutive pairs, whose spans km - k1 + 1 and l1 - lm + 1 are both at most max_span (<= 64).
// Its score is
//
//   E = (double)H / 100.0 + ED_a + ED_b          H: bf_duplex's energy of the chain (dcal/mol), ED = -(kT/1000) ln P_u (kcal/mol)
//
// with ED_a the opening energy of a[k1 .. km] and ED_b that of b[lm .. l1] (tables from bf_k_interact_ed; null: no accessibility).
// Since the opening cost depends on both ends of the site, the DP runs from a fixed start pair (k1,l1) over its max_span x max_span
// window, cells (i,j) = (k1 + di, l1 - dj):
//
//   h(k1,l1) = DuplexInit + Ext(type(k1,l1), a[k1-1], b[l1+1])
//   h(i,j)   = min over k1 <= k < i, j < l <= l1, (i-k-1) + (l-j-1) <= 30:  h(k,l) + IntLoop(...)      (no other start)
//   site (k1, i, j, l1):  H = h(i,j) + Ext(rtype(type(i,j)), b[j-1], a[i+1])
//
// Each pair's result is the site of least E; ties go to the first site in the order k1 ascending, l1 descending, km ascending, lm
// descending (the packed rank below).  The structure is walked back with bf_duplex's rule inside the fixed-start table.
// tests/interact_ref.c holds the same rules in plain C.
//
// Mapping: a unit of work is (pair, start row k1), dealt through a work counter to a persistent grid of 4-warp CTAs.  A warp takes
// one start (k1,l1) that pairs and fills its window in a warp-private shared-memory table (max_span^2 ints) by anti-diagonal, one
// __syncwarp per diagonal; its lanes split a cell's (u1,u2) candidates (bf_duplex's s-major order, bounded by the window) and reduce
// with __reduce_min_sync.  The k1 row of ED_a is staged in shared memory, ED_b is read through L1.  The CTA writes its unit's best
// (E, rank, H) to a slot; bf_k_interact_reduce takes each pair's slots, and bf_k_interact_trace (structures only) re-runs the
// winner's window in one warp and walks it back.  No n1 x n2 table goes to HBM.
#include <math.h>

#include <algorithm>

#include "bf_kernels.h"

#include "bf_device.cuh"

namespace {

constexpr int kIxWarps = 4;

__host__ __device__ inline size_t al16(size_t x) { return (x + 15) / 16 * 16; }

struct IxPair { int ia, ib; };
// pair q of the launch; the grid's from (ia0, ib0) = pair p0 in 32-bit arithmetic (ib0 + q < 2^32)
__device__ __forceinline__ IxPair ix_pair(const BfInteractDev &d, int q) {
  IxPair r;
  if (d.pairs) { r.ia = d.pairs[2 * (d.p0 + q)]; r.ib = d.pairs[2 * (d.p0 + q) + 1]; }
  else { const unsigned t = (unsigned)d.ib0 + (unsigned)q; r.ia = d.ia0 + (int)(t / (unsigned)d.nb); r.ib = (int)(t % (unsigned)d.nb); }
  return r;
}

// k1 ascending, l1 descending, km ascending, lm descending; di = km - k1, dj = l1 - lm < 64
__device__ __forceinline__ long long ix_rank(int n2, int k1, int l1, int di, int dj) {
  return ((long long)((k1 - 1) * n2 + (n2 - l1)) * 64 + di) * 64 + dj;
}
__device__ __forceinline__ bool ix_less(double e, long long r, double be, long long br) { return e < be || (e == be && r < br); }

// (double)v / 100.0 without the division's slow-path call (whose call frame spills): a product and one fma correction step.  Equal
// to the correctly rounded quotient for every integer |v| <= 200000 (the CPU interaction tests check every one); a site's
// H lies far inside that range (at most 64 pairs, |loop energy| < 1000 dcal/mol).
__device__ __forceinline__ double ix_div100(int v) {
  const double x = (double)v, q = x * 0.01;
  return __fma_rn(__fma_rn(-q, 100.0, x), 0.01, q);
}

__device__ __forceinline__ double ix_ed(const double *ed, int strand, int rows, int span, int k, int u) {
  return ed ? ed[((size_t)strand * rows + k - 1) * span + u - 1] : 0.0;
}

// One warp fills the window of start (k1,l1), wa rows along a and wb columns along b: tab[di * span + dj] = h(k1 + di, l1 - dj), or
// BF_INF.  visit(di, dj, h) runs in every lane for each finite cell once it is set.
template <class F>
__device__ __forceinline__ void ix_window(const BfParams *__restrict__ P, const BfSmallI &T, const unsigned char (*cand)[2],
                                          const uint8_t *A, const uint8_t *Bs, int n1, int n2, int k1, int l1, int span, int wa, int wb,
                                          int *tab, F &visit) {
  const int lane = threadIdx.x & 31;
  for (int dg = 0; dg <= wa + wb - 2; dg++) {
    for (int di = max(0, dg - wb + 1); di <= min(wa - 1, dg); di++) {
      const int dj = dg - di, i = k1 + di, j = l1 - dj;
      const int t = bf_ptype_bases(A[i], Bs[j]);
      int h = BF_INF;
      if (t) {
        const int ai = i > 1 ? A[i - 1] : -1, bj = j < n2 ? Bs[j + 1] : -1;
        if (dg == 0) {
          h = T.DuplexInit + bf_e_ext(T, t, ai, bj);
        } else {
          const int um1 = di - 1, um2 = dj - 1;   // u1 <= di - 1 keeps k >= k1, u2 <= dj - 1 keeps l <= l1
          if (um1 >= 0 && um2 >= 0) {
            const int smax = min(BF_MAXLOOP, um1 + um2), ncand = (smax + 1) * (smax + 2) / 2, rt = bf_rtype(t);
            int m = BF_INF;
            for (int x = lane; x < ncand; x += 32) {
              const int s = cand[x][0], u1 = cand[x][1], u2 = s - u1;
              if (u1 > um1 || u2 > um2) continue;
              const int ck = tab[(di - 1 - u1) * span + (dj - 1 - u2)];
              if (ck >= BF_INF) continue;
              const int k = i - 1 - u1, l = j + 1 + u2;
              m = min(m, ck + bf_e_intloop(P, T, u1, u2, bf_ptype_bases(A[k], Bs[l]), rt, A[k + 1], Bs[l - 1], ai, bj));
            }
            h = bf_warp_min(m);
          }
        }
      }
      if (lane == 0) tab[di * span + dj] = h;
      if (h < BF_INF) visit(di, dj, h, t);
    }
    __syncwarp();
  }
}

__device__ void ix_cand_tables(unsigned char (*fill)[2], unsigned char (*bt)[2]) {
  for (int x = threadIdx.x; x < BF_NCAND; x += blockDim.x) {
    int s = 0;
    while ((s + 1) * (s + 2) / 2 <= x) s++;
    fill[x][0] = (unsigned char)s;
    fill[x][1] = (unsigned char)(x - s * (s + 1) / 2);
    if (bt) {
      int u1 = 0, r = x;
      while (r >= 31 - u1) { r -= 31 - u1; u1++; }
      bt[x][0] = (unsigned char)u1;
      bt[x][1] = (unsigned char)r;
    }
  }
}

__device__ void ix_load_strands(const BfInteractDev &d, IxPair pr, int n1, int n2, uint8_t *A, uint8_t *Bs) {
  const char *sa = d.seq_a + (size_t)pr.ia * d.stride_a, *sb = d.seq_b + (size_t)pr.ib * d.stride_b;
  for (int k = threadIdx.x; k <= n1 + 1; k += blockDim.x) A[k] = (uint8_t)((k >= 1 && k <= n1) ? bf_base_code(sa[k - 1]) : 0);
  for (int k = threadIdx.x; k <= n2 + 1; k += blockDim.x) Bs[k] = (uint8_t)((k >= 1 && k <= n2) ? bf_base_code(sb[k - 1]) : 0);
}

size_t ix_smem(const BfInteractDev &d, int warps) {
  return al16((size_t)warps * d.span * d.span * sizeof(int)) + al16((size_t)d.span * sizeof(double)) + al16(d.amax + 2) + al16(d.bmax + 2);
}

// units u = (pair - p0) * amax + k1 - 1 of the launch; slot u holds the unit's best site
__global__ void __launch_bounds__(kIxWarps * 32) bf_k_interact(const BfParams *__restrict__ P, BfInteractDev d, BfInteractSlot *slots,
                                                               int *work_counter) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallI T;
  __shared__ unsigned char s_fill[BF_NCAND][2];
  __shared__ int s_unit;
  __shared__ double s_e[kIxWarps];
  __shared__ long long s_r[kIxWarps];
  __shared__ int s_h[kIxWarps];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, span = d.span;
  int *tab = reinterpret_cast<int *>(dyn) + warp * span * span;
  double *eda = reinterpret_cast<double *>(dyn + al16((size_t)kIxWarps * span * span * sizeof(int)));
  uint8_t *A = reinterpret_cast<uint8_t *>(eda) + al16((size_t)span * sizeof(double));
  uint8_t *Bs = A + al16(d.amax + 2);
  bf_stage(&T, &P->si);
  ix_cand_tables(s_fill, nullptr);
  const long long units = (long long)d.np * d.amax;
  for (;;) {
    __syncthreads();
    if (tid == 0) s_unit = atomicAdd(work_counter, 1);
    __syncthreads();
    const int u = s_unit;
    if (u >= units) break;
    const int q = u / d.amax, k1 = u % d.amax + 1;
    const IxPair pr = ix_pair(d, q);
    const int n1 = d.len_a[pr.ia], n2 = d.len_b[pr.ib];
    if (k1 > n1) {
      if (tid == 0) slots[u] = BfInteractSlot{INFINITY, -1, BF_INF, 0};
      continue;
    }
    ix_load_strands(d, pr, n1, n2, A, Bs);
    for (int x = tid; x < span; x += blockDim.x) eda[x] = k1 + x <= n1 ? ix_ed(d.ed_a, pr.ia, d.rows_a, span, k1, x + 1) : INFINITY;
    __syncthreads();
    double be = INFINITY;
    long long br = -1;
    int bh = BF_INF;
    const int wa = min(span, n1 - k1 + 1);
    for (int l1 = n2 - warp; l1 >= 1; l1 -= kIxWarps) {
      if (!bf_ptype_bases(A[k1], Bs[l1])) continue;
      auto close = [&](int di, int dj, int h, int t) {
        const int i = k1 + di, j = l1 - dj;
        const int v = h + bf_e_ext(T, bf_rtype(t), j > 1 ? Bs[j - 1] : -1, i < n1 ? A[i + 1] : -1);
        const double e = ix_div100(v) + eda[di] + ix_ed(d.ed_b, pr.ib, d.rows_b, span, j, dj + 1);
        const long long r = ix_rank(n2, k1, l1, di, dj);
        if (e < INFINITY && ix_less(e, r, be, br)) { be = e; br = r; bh = v; }
      };
      ix_window(P, T, s_fill, A, Bs, n1, n2, k1, l1, span, wa, min(span, l1), tab, close);
    }
    if (lane == 0) { s_e[warp] = be; s_r[warp] = br; s_h[warp] = bh; }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < kIxWarps; w++)
        if (s_r[w] >= 0 && (br < 0 || ix_less(s_e[w], s_r[w], be, br))) { be = s_e[w]; br = s_r[w]; bh = s_h[w]; }
      slots[s_unit] = BfInteractSlot{be, br, bh, 0};
    }
  }
}

// one warp per pair of the launch: the least (E, rank) of its units
__global__ void __launch_bounds__(256) bf_k_interact_reduce(BfInteractDev d, const BfInteractSlot *__restrict__ slots, BfInteractOut out) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= d.np) return;
  const IxPair pr = ix_pair(d, q);
  const int n1 = d.len_a[pr.ia], n2 = d.len_b[pr.ib];
  double be = INFINITY;
  long long br = -1;
  int bh = BF_INF;
  for (int k = lane; k < n1; k += 32) {
    const BfInteractSlot s = slots[(size_t)q * d.amax + k];
    if (s.rank >= 0 && (br < 0 || ix_less(s.e, s.rank, be, br))) { be = s.e; br = s.rank; bh = s.h; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double oe = __shfl_xor_sync(BF_FULL, be, o);
    const long long orr = __shfl_xor_sync(BF_FULL, br, o);
    const int oh = __shfl_xor_sync(BF_FULL, bh, o);
    if (orr >= 0 && (br < 0 || ix_less(oe, orr, be, br))) { be = oe; br = orr; bh = oh; }
  }
  if (lane != 0) return;
  out.rank[q] = br;
  out.e[q] = be;
  out.h[q] = bh;
  int k1 = 0, km = 0, lm = 0, l1 = 0;
  double ea = 0.0, eb = 0.0;
  if (br >= 0) {
    const long long st = br >> 12;
    const int di = (int)((br >> 6) & 63), dj = (int)(br & 63);
    k1 = (int)(st / n2) + 1; l1 = n2 - (int)(st % n2); km = k1 + di; lm = l1 - dj;
    ea = ix_ed(d.ed_a, pr.ia, d.rows_a, d.span, k1, di + 1);
    eb = ix_ed(d.ed_b, pr.ib, d.rows_b, d.span, lm, dj + 1);
  }
  if (out.ed) { out.ed[2 * q] = ea; out.ed[2 * q + 1] = eb; }
  if (out.site) { int *s = out.site + 4 * q; s[0] = k1; s[1] = km; s[2] = lm; s[3] = l1; }
}

// one warp per pair of the launch: re-run the winner's window and walk it back with bf_duplex's rule
__global__ void __launch_bounds__(32) bf_k_interact_trace(const BfParams *__restrict__ P, BfInteractDev d, const long long *__restrict__ rank,
                                                          char *ss_out, int ss_stride) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallI T;
  __shared__ unsigned char s_fill[BF_NCAND][2], s_bt[BF_NCAND][2];
  const int lane = threadIdx.x, q = blockIdx.x, span = d.span;
  int *tab = reinterpret_cast<int *>(dyn);
  uint8_t *A = dyn + al16((size_t)span * span * sizeof(int));
  uint8_t *Bs = A + al16(d.amax + 2);
  const IxPair pr = ix_pair(d, q);
  const int n1 = d.len_a[pr.ia], n2 = d.len_b[pr.ib];
  char *ss = ss_out + (size_t)q * ss_stride;
  for (int k = lane; k < ss_stride; k += 32) ss[k] = k < n1 || (k > n1 && k <= n1 + n2) ? '.' : k == n1 ? '&' : '\0';
  const long long br = rank[q];
  if (br < 0) return;
  bf_stage(&T, &P->si);
  ix_cand_tables(s_fill, s_bt);
  ix_load_strands(d, pr, n1, n2, A, Bs);
  __syncwarp();
  const long long st = br >> 12;
  const int k1 = (int)(st / n2) + 1, l1 = n2 - (int)(st % n2);
  int di = (int)((br >> 6) & 63), dj = (int)(br & 63);
  auto none = [](int, int, int, int) {};
  ix_window(P, T, s_fill, A, Bs, n1, n2, k1, l1, span, di + 1, dj + 1, tab, none);
  while (true) {
    const int i = k1 + di, j = l1 - dj;
    if (lane == 0) { ss[i - 1] = '('; ss[n1 + j] = ')'; }
    if (di == 0 && dj == 0) break;
    const int hij = tab[di * span + dj], rt = bf_rtype(bf_ptype_bases(A[i], Bs[j]));
    int found = -1;
    for (int base = 0; base < BF_NCAND && found < 0; base += 32) {
      const int x = base + lane;
      bool hit = false;
      if (x < BF_NCAND) {
        const int u1 = s_bt[x][0], u2 = s_bt[x][1];
        if (u1 <= di - 1 && u2 <= dj - 1) {
          const int k = i - 1 - u1, l = j + 1 + u2, ck = tab[(di - 1 - u1) * span + (dj - 1 - u2)];
          hit = ck < BF_INF && hij == ck + bf_e_intloop(P, T, u1, u2, bf_ptype_bases(A[k], Bs[l]), rt, A[k + 1], Bs[l - 1], A[i - 1], Bs[j + 1]);
        }
      }
      const unsigned hm = __ballot_sync(BF_FULL, hit);
      if (hm) found = base + __ffs(hm) - 1;
    }
    if (found < 0) break;
    di -= 1 + s_bt[found][0];
    dj -= 1 + s_bt[found][1];
  }
}

__global__ void __launch_bounds__(256) bf_k_interact_ed(const double *__restrict__ pu, double *ed, size_t n, double kT) {
  for (size_t x = blockIdx.x * (size_t)blockDim.x + threadIdx.x; x < n; x += (size_t)gridDim.x * blockDim.x) {
    const double p = pu[x];
    ed[x] = p > 0.0 ? -(kT / 1000.0) * log(p) : INFINITY;
  }
}

}  // namespace

cudaError_t bf_launch_interact_ed(const double *pu, double *ed, size_t n, double kT, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, 65535);
  bf_k_interact_ed<<<grid, 256, 0, st>>>(pu, ed, n, kT);
  return cudaGetLastError();
}

cudaError_t bf_launch_interact(const BfParams *dP, const BfInteractDev &d, BfInteractSlot *slots, const BfInteractOut &out, char *ss_out,
                               int ss_stride, int *work_counter, int sms, cudaStream_t st) {
  if (d.np <= 0) return cudaSuccess;
  const size_t sm = ix_smem(d, kIxWarps);
  cudaError_t e = cudaFuncSetAttribute(bf_k_interact, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(sm, 1024));
  if (e != cudaSuccess) return e;
  int occ = 0;
  if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bf_k_interact, kIxWarps * 32, sm)) != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  const long long units = (long long)d.np * d.amax;
  const int grid = (int)std::min<long long>(units, (long long)occ * sms);
  if ((e = cudaMemsetAsync(work_counter, 0, sizeof(int), st)) != cudaSuccess) return e;
  bf_k_interact<<<grid, kIxWarps * 32, sm, st>>>(dP, d, slots, work_counter);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  bf_k_interact_reduce<<<(d.np + 7) / 8, 256, 0, st>>>(d, slots, out);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if (!ss_out) return cudaSuccess;
  const size_t smt = al16((size_t)d.span * d.span * sizeof(int)) + al16(d.amax + 2) + al16(d.bmax + 2);
  if ((e = cudaFuncSetAttribute(bf_k_interact_trace, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smt, 1024))) != cudaSuccess)
    return e;
  bf_k_interact_trace<<<d.np, 32, smt, st>>>(dP, d, out.rank, ss_out, ss_stride);
  return cudaGetLastError();
}
