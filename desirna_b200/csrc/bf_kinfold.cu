// bf_kinfold.cu -- folding kinetics on the device (sm_100a): Kinfold-style stochastic trajectories and steepest-descent walks over
// single-pair moves.  include/b200fold.h (bf_kinfold) holds the definition; tests/kinfold_ref.c restates it in plain C.
//
// Mapping: a unit of work is one trajectory (instance r, trajectory k), dealt through a work counter to a persistent grid of 8-warp
// CTAs, one warp per unit.  A warp keeps its trajectory's bases, pair table and loop table (for every position, the 5' end of the
// closing pair of the loop it lies in, or of the loop its pair stands in; 0: the exterior loop) in shared memory.  Per step:
//   1. the warp walks the candidate pairs in (i, j) order, 32 j at a time: a pair of the structure is a deletion; an unpaired i
//      pairs with the unpaired j of its own loop (same loop-table entry, j before the loop's closing pair), canonical, j - i >= 4.
//      Each valid move's dE comes from per-loop summaries (KfLoops) in O(1), except where a deletion leaves a hairpin or an
//      interior loop, which is re-scored (bf_loops.cuh); ballot / popc compact the valid moves in order into
//      a shared buffer, and every full group of 32 is scanned (5-step inclusive warp scan of the rates) and added to the running
//      total.  The running total after each group and the group's first move go to the warp's HBM workspace.
//   2. u1 gives dt; u2 K picks the first group whose running total exceeds it (ballot over the stored totals), and a walk from
//      that group's first move collects its 32 moves again and scans them to pick the move.  No third pass over all moves.
//   3. the move updates the pair table, the loop table (the positions of the loop it splits or merges), E and the running count
//      of differences against the stop structure; one lane rebuilds the loop summaries in one O(n) pass.
// Steepest descent walks once per step and keeps the least (dE, move) per lane, reduced over the warp.
// This is the first mapping and is not tuned.
#include <algorithm>
#include <cassert>
#include <climits>

#include "bf_kernels.h"

#include "bf_device.cuh"
#include "bf_loops.cuh"

namespace {

constexpr int kKfWarps = 8;
constexpr int kKfThreads = kKfWarps * 32;

__host__ __device__ inline size_t kf_al(size_t x) { return (x + 15) / 16 * 16; }
// shared memory of one warp: bases, pair table, loop table, then the move buffer (64 moves and 64 dE)
__host__ __device__ inline size_t kf_warp_smem(int nmax) { return kf_al(nmax + 2) + 2 * kf_al((size_t)(nmax + 2) * 2) + 2 * 64 * 4; }

// HBM workspace of one warp: the running totals and first moves of up to gmax groups, then the loop summaries (KfLoops)
__host__ __device__ inline size_t kf_warp_ws(int gmax, int nmax) {
  return kf_al((size_t)gmax * 8) + kf_al((size_t)gmax * 4) + 3 * kf_al((size_t)(nmax + 2) * 2) + 3 * kf_al((size_t)(nmax + 2) * 4);
}

struct KfWarp {
  uint8_t *S;
  short *pt, *lid;
  int *pm, *pde;   // buffered valid moves (i << 16 | j) and their dE
};

// Per-loop summaries of the current structure, in the warp's HBM workspace, indexed by position.  For a loop closed by (p, q) (p = 0:
// the exterior loop) at index p: its stem count C, unpaired count U, first stem F, sums of its stems' multiloop-stem energies M and
// exterior-stem energies X, and its energy EL.  At an unpaired position x of a loop: C, U, M, X of that loop counted up to and
// including x.  So an insertion (i, j) into loop L finds the stems and unpaired bases strictly inside (i, j) as differences of
// the values at j and i, and its dE in O(1).
struct KfLoops {
  short *C, *U, *F;
  int *M, *X, *EL;
};

// energy of the loop closed by (i, j) with ns stems (first stem (p1, q1)), multiloop-stem sum ml and unp unpaired bases, as fp_loop
__device__ __forceinline__ int kf_close(const BfParams *__restrict__ P, const BfSmallI &T, const uint8_t *S, int i, int j, int ns, int p1,
                                        int q1, int ml, int unp) {
  const int t = fp_type(S, i, j);
  if (ns == 0) return bf_e_hairpin(P, T, S, i, j, t);
  if (ns == 1) return bf_e_intloop(P, T, p1 - i - 1, j - q1 - 1, t, fp_type(S, q1, p1), S[i + 1], S[j - 1], S[p1 - 1], S[q1 + 1]);
  return T.MLclosing + bf_e_mlstem(T, bf_rtype(t), S[j - 1], S[i + 1]) + ml + unp * T.MLbase;
}

// the summaries of the warp's structure (lane 0)
__device__ void kf_summarise(const BfParams *__restrict__ P, const BfSmallI &T, const KfWarp &w, int n, const KfLoops &q) {
  q.C[0] = q.U[0] = q.F[0] = 0;
  q.M[0] = q.X[0] = 0;
  for (int x = 1; x <= n; x++) {
    const int p = w.pt[x], L = w.lid[x];
    if (p == 0) {
      q.U[L]++;
      q.C[x] = q.C[L]; q.U[x] = q.U[L]; q.M[x] = q.M[L]; q.X[x] = q.X[L];
    } else if (p > x) {
      const int t = fp_type(w.S, x, p);
      if (q.C[L] == 0) q.F[L] = (short)x;
      q.C[L]++;
      q.M[L] += bf_e_mlstem(T, t, w.S[x - 1], w.S[p + 1]);
      q.X[L] += bf_e_ext(T, t, x > 1 ? w.S[x - 1] : -1, p < n ? w.S[p + 1] : -1);
      q.C[x] = q.U[x] = q.F[x] = 0;
      q.M[x] = q.X[x] = 0;
    }
  }
  q.EL[0] = q.X[0];
  for (int x = 1; x <= n; x++) {
    const int p = w.pt[x];
    if (p > x) q.EL[x] = kf_close(P, T, w.S, x, p, q.C[x], q.F[x], w.pt[q.F[x]], q.M[x], q.U[x]);
  }
}

// dE of deleting pair (i, j) of the structure (the two loops re-scored), or of inserting (i, j) into the loop of i (from the summaries)
__device__ int kf_de(const BfParams *__restrict__ P, const BfSmallI &T, const KfWarp &w, const KfLoops &q, int n, int i, int j, bool del) {
  const int L = w.lid[i];
  const int t = fp_type(w.S, i, j);
  if (del) {
    // the merged loop: the stems and unpaired bases of both, less the stem (i, j), plus i and j unpaired
    int el;
    if (L == 0) {
      el = q.X[0] - bf_e_ext(T, t, i > 1 ? w.S[i - 1] : -1, j < n ? w.S[j + 1] : -1) + q.X[i];
    } else if (q.C[L] - 1 + q.C[i] >= 2) {
      el = kf_close(P, T, w.S, L, w.pt[L], q.C[L] - 1 + q.C[i], 0, 0, q.M[L] - bf_e_mlstem(T, t, w.S[i - 1], w.S[j + 1]) + q.M[i],
                    q.U[L] + q.U[i] + 2);
    } else {
      const FpView v1{w.pt, -1, -1, i, j};   // a hairpin or an interior loop: re-scored
      el = fp_loop(P, T, w.S, n, v1, L);
    }
    return el - q.EL[L] - q.EL[i];
  }
  const int ns = q.C[j] - q.C[i], ml = q.M[j] - q.M[i], unp = q.U[j] - q.U[i] - 1;
  int p1 = 0, q1 = 0;
  if (ns == 1) {
    for (p1 = i + 1; w.pt[p1] == 0; p1++) {}
    q1 = w.pt[p1];
  }
  const int em = kf_close(P, T, w.S, i, j, ns, p1, q1, ml, unp);
  if (L == 0) return em + bf_e_ext(T, t, i > 1 ? w.S[i - 1] : -1, j < n ? w.S[j + 1] : -1) - (q.X[j] - q.X[i]);
  const int ql = w.pt[L], ns2 = q.C[L] - ns + 1;
  const int el = ns2 == 1 ? kf_close(P, T, w.S, L, ql, 1, i, j, 0, 0)
                          : kf_close(P, T, w.S, L, ql, ns2, 0, 0, q.M[L] - ml + bf_e_mlstem(T, t, w.S[i - 1], w.S[j + 1]), q.U[L] - unp - 2);
  return em + el - q.EL[L];
}

// the valid moves in canonical order from candidate (i0, j0): f(valid, i, j, dE) once per chunk of 32 lanes (warp-uniform);
// f returns true to stop the walk
template <class F>
__device__ void kf_walk(const BfParams *__restrict__ P, const BfSmallI &T, const KfWarp &w, const KfLoops &q, int n, int i0, int j0,
                        F &f) {
  const int lane = threadIdx.x & 31;
  for (int i = i0; i <= n; i++) {
    const int p = w.pt[i];
    if (p > i) {
      const bool valid = lane == 0;
      const int de = valid ? kf_de(P, T, w, q, n, i, p, true) : 0;
      if (f(valid, i, p, de)) return;
    } else if (p == 0) {
      const int L = w.lid[i], hi = L ? w.pt[L] - 1 : n;
      for (int jb = max(i + 4, i == i0 ? j0 : 0); jb <= hi; jb += 32) {
        const int j = jb + lane;
        const bool valid = j <= hi && w.pt[j] == 0 && w.lid[j] == L && bf_ptype_bases(w.S[i], w.S[j]) != 0;
        const int de = valid ? kf_de(P, T, w, q, n, i, j, false) : 0;
        if (f(valid, i, j, de)) return;
      }
    }
  }
}

__device__ __forceinline__ double kf_scan(double v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double y = __shfl_up_sync(BF_FULL, v, o);
    if (lane >= o) v += y;
  }
  return v;
}

__device__ __forceinline__ double kf_rate(const double *__restrict__ rate, int de) {
  assert(de >= -32768 && de <= 32767);
  return __ldg(rate + de + 32768);
}

// appends the valid moves of a chunk to the buffer, in order
struct KfBuffer {
  const KfWarp &w;
  int np = 0;
  __device__ explicit KfBuffer(const KfWarp &w_) : w(w_) {}
  __device__ void append(bool valid, int i, int j, int de) {
    const int lane = threadIdx.x & 31;
    const unsigned bal = __ballot_sync(BF_FULL, valid);
    const int pos = np + __popc(bal & ((1u << lane) - 1));
    if (valid) { w.pm[pos] = i << 16 | j; w.pde[pos] = de; }
    np += __popc(bal);
    __syncwarp();
  }
};

// step 1: K as the running total of the scanned groups; per group, the total so far and its first move
struct KfSum : KfBuffer {
  const double *rate;
  double *gR;
  int *gS;
  int G = 0;
  double R = 0.0;
  __device__ KfSum(const KfWarp &w_, const double *rate_, double *gR_, int *gS_) : KfBuffer(w_), rate(rate_), gR(gR_), gS(gS_) {}
  __device__ void flush(int cnt) {
    const int lane = threadIdx.x & 31;
    const double v = kf_scan(lane < cnt ? kf_rate(rate, w.pde[lane]) : 0.0);
    R += __shfl_sync(BF_FULL, v, 31);
    if (lane == 0) { gR[G] = R; gS[G] = w.pm[0]; }
    G++;
  }
  __device__ bool operator()(bool valid, int i, int j, int de) {
    append(valid, i, j, de);
    if (np >= 32) {
      flush(32);
      const int lane = threadIdx.x & 31;
      const bool mv = lane < np - 32;
      int m = 0, d = 0;
      if (mv) { m = w.pm[32 + lane]; d = w.pde[32 + lane]; }
      __syncwarp();
      if (mv) { w.pm[lane] = m; w.pde[lane] = d; }
      __syncwarp();
      np -= 32;
    }
    return false;
  }
};

// step 2: the first 32 valid moves from a group's first move
struct KfCollect : KfBuffer {
  __device__ explicit KfCollect(const KfWarp &w_) : KfBuffer(w_) {}
  __device__ bool operator()(bool valid, int i, int j, int de) {
    append(valid, i, j, de);
    return np >= 32;
  }
};

// steepest descent: the least (dE, move) of the lane's valid moves
struct KfMin {
  long long best = LLONG_MAX;
  __device__ bool operator()(bool valid, int i, int j, int de) {
    if (valid) best = min(best, (long long)de * 4294967296ll + (long long)(unsigned)(i << 16 | j));
    return false;
  }
};

__device__ void kf_write_ss(const KfWarp &w, int n, int stride, char *out) {
  for (int c = threadIdx.x & 31; c <= stride; c += 32) {
    const int x = c + 1;
    out[c] = c < n ? (w.pt[x] == 0 ? '.' : w.pt[x] > x ? '(' : ')') : '\0';
  }
}

__global__ void __launch_bounds__(kKfThreads) bf_k_kinfold(const BfParams *__restrict__ P, BfKinfoldDev d, unsigned char *ws,
                                                          int *work_counter) {
  __shared__ BfSmallI T;
  extern __shared__ __align__(16) unsigned char kf_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  bf_stage(&T, &P->si);
  __syncthreads();
  const size_t a1 = kf_al(d.nmax + 2), a2 = kf_al((size_t)(d.nmax + 2) * 2);
  unsigned char *base = kf_smem + warp * kf_warp_smem(d.nmax);
  KfWarp w;
  w.S = base;
  w.pt = reinterpret_cast<short *>(base + a1);
  w.lid = reinterpret_cast<short *>(base + a1 + a2);
  w.pm = reinterpret_cast<int *>(base + a1 + 2 * a2);
  w.pde = w.pm + 64;
  unsigned char *wb = ws + ((size_t)blockIdx.x * kKfWarps + warp) * kf_warp_ws(d.gmax, d.nmax);
  const size_t b2 = kf_al((size_t)(d.nmax + 2) * 2), b4 = kf_al((size_t)(d.nmax + 2) * 4);
  double *gR = reinterpret_cast<double *>(wb);
  int *gS = reinterpret_cast<int *>(wb + kf_al((size_t)d.gmax * 8));
  unsigned char *lb = wb + kf_al((size_t)d.gmax * 8) + kf_al((size_t)d.gmax * 4);
  KfLoops lp;
  lp.C = reinterpret_cast<short *>(lb);
  lp.U = reinterpret_cast<short *>(lb + b2);
  lp.F = reinterpret_cast<short *>(lb + 2 * b2);
  lp.M = reinterpret_cast<int *>(lb + 3 * b2);
  lp.X = reinterpret_cast<int *>(lb + 3 * b2 + b4);
  lp.EL = reinterpret_cast<int *>(lb + 3 * b2 + 2 * b4);
  const int S1 = d.stride + 1;
  for (;;) {
    int u = 0;
    if (lane == 0) u = atomicAdd(work_counter, 1);
    u = __shfl_sync(BF_FULL, u, 0);
    if (u >= d.nu) break;
    const long long ug = d.u0 + u;
    const int r = (int)(ug / d.T), k = (int)(ug % d.T);
    const int n = d.len[r];
    const char *seq = d.seq + (size_t)r * d.stride;
    const short *pt0 = d.start + (size_t)r * (d.stride + 2);
    const short *pst = d.stop ? d.stop + (size_t)r * (d.stride + 2) : nullptr;
    for (int x = lane; x <= n + 1; x += 32) {
      w.S[x] = (uint8_t)((x >= 1 && x <= n) ? bf_base_code(seq[x - 1]) : 0);
      w.pt[x] = pt0[x];
    }
    __syncwarp();
    int e = 0;
    if (lane == 0) {
      int cur = 0;
      w.lid[0] = 0;
      for (int x = 1; x <= n; x++) {
        const int q = w.pt[x];
        if (q == 0) w.lid[x] = (short)cur;
        else if (q > x) { w.lid[x] = (short)cur; w.lid[q] = (short)cur; cur = x; }
        else cur = w.lid[x];
      }
      e = fp_eval(P, T, w.S, n, w.pt);
      kf_summarise(P, T, w, n, lp);
    }
    e = __shfl_sync(BF_FULL, e, 0);
    int diff = 0;
    if (pst)
      for (int x = 1 + lane; x <= n; x += 32) diff += (w.pt[x] > x && pst[x] != w.pt[x]) + (pst[x] > x && w.pt[x] != pst[x]);
    diff = __reduce_add_sync(BF_FULL, diff);
    __syncwarp();
    // the stream of (seed, instance, trajectory), as bf_sample seeds (seed, row, sample)
    unsigned long long s0 = d.seed;
    unsigned long long s1 = sm64(s0) ^ (((unsigned long long)(unsigned)r << 32) | (unsigned)k);
    unsigned long long rs = sm64(s1);
    double t = 0.0;
    long long steps = 0;
    int status = 0, s = 0;
    const long long ou = u;
    int *e_snap = d.e_snap + ou * d.n_snap;
    char *ss_snap = d.ss_snap + ou * d.n_snap * S1;
    bool done = pst && diff == 0;
    if (done) status = 1;
    while (!done) {
      int m, de;
      if (d.rule == 2) {
        KfMin f;
        kf_walk(P, T, w, lp, n, 1, 0, f);
        long long b = f.best;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) b = min(b, (long long)__shfl_xor_sync(BF_FULL, b, o));
        if (b == LLONG_MAX || (b >> 32) >= 0) break;
        de = (int)(b >> 32);
        m = (int)(unsigned)(b & 0xffffffffll);
      } else {
        KfSum f(w, d.rate, gR, gS);
        kf_walk(P, T, w, lp, n, 1, 0, f);
        if (f.np) f.flush(f.np);
        __syncwarp();
        if (f.G == 0) { t = d.t_max; break; }   // no move: absorbing until t_max
        const double K = f.R;
        const double u1 = u01(rs), u2 = u01(rs);
        const double tn = t + -log(1.0 - u1) / K;
        if (tn > d.t_max) { t = d.t_max; break; }
        while (s < d.n_snap && d.t_snap[s] < tn) {
          if (lane == 0) e_snap[s] = e;
          kf_write_ss(w, n, d.stride, ss_snap + (size_t)s * S1);
          s++;
        }
        t = tn;
        const double target = u2 * K;
        int g = -1;
        for (int g0 = 0; g0 < f.G; g0 += 32) {
          const bool over = g0 + lane < f.G && gR[g0 + lane] > target;
          const unsigned b = __ballot_sync(BF_FULL, over);
          if (b) { g = g0 + __ffs(b) - 1; break; }
        }
        const bool last = g < 0;   // u2 K rounded up to K: the last valid move
        if (last) g = f.G - 1;
        KfCollect c(w);
        kf_walk(P, T, w, lp, n, gS[g] >> 16, gS[g] & 0xffff, c);
        const int cnt = min(c.np, 32);
        const double v = kf_scan(lane < cnt ? kf_rate(d.rate, w.pde[lane]) : 0.0);
        const double rp = g > 0 ? gR[g - 1] : 0.0;
        const unsigned b = __ballot_sync(BF_FULL, lane < cnt && rp + v > target);
        const int pick = (last || !b) ? cnt - 1 : __ffs(b) - 1;
        m = w.pm[pick];
        de = w.pde[pick];
        __syncwarp();
      }
      // apply move m
      const int i = m >> 16, j = m & 0xffff;
      const bool del = w.pt[i] == j;
      const int L = w.lid[i];
      __syncwarp();
      for (int x = i + 1 + lane; x < j; x += 32) {
        if (del) { if (w.lid[x] == i) w.lid[x] = (short)L; }
        else if (w.lid[x] == L) w.lid[x] = (short)i;
      }
      if (lane == 0) {
        w.pt[i] = del ? 0 : (short)j;
        w.pt[j] = del ? 0 : (short)i;
      }
      __syncwarp();
      if (lane == 0) kf_summarise(P, T, w, n, lp);
      __syncwarp();
      e += de;
      if (pst) diff += ((pst[i] == j) == del) ? 1 : -1;
      steps++;
      if (pst && diff == 0) { status = 1; break; }
      if (steps >= d.max_steps) { status = 2; break; }
    }
    // the snapshots after the end: the final state (t_max or hit), none after a cap or in a descent
    const bool blank = status == 2 || d.rule == 2;
    for (; s < d.n_snap; s++) {
      if (lane == 0) e_snap[s] = blank ? BF_INF : e;
      if (blank) {
        for (int c = lane; c <= d.stride; c += 32) ss_snap[(size_t)s * S1 + c] = '\0';
      } else {
        kf_write_ss(w, n, d.stride, ss_snap + (size_t)s * S1);
      }
    }
    if (lane == 0) {
      d.status[ou] = status;
      d.t_end[ou] = t;
      d.steps[ou] = steps;
      d.e_end[ou] = e;
    }
    kf_write_ss(w, n, d.stride, d.ss_end + ou * S1);
    __syncwarp();
  }
}

}  // namespace

size_t bf_kinfold_smem(int nmax) { return kKfWarps * kf_warp_smem(nmax); }
size_t bf_kinfold_ws_bytes(int gmax, int nmax) { return kKfWarps * kf_warp_ws(gmax, nmax); }

int bf_kinfold_occupancy(int nmax) {
  const size_t sm = bf_kinfold_smem(nmax);
  if (cudaFuncSetAttribute(bf_k_kinfold, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return 1;
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bf_k_kinfold, kKfThreads, sm) != cudaSuccess) return 1;
  return std::max(occ, 1);
}

cudaError_t bf_launch_kinfold(const BfParams *dP, const BfKinfoldDev &d, unsigned char *ws, int grid, int *work_counter, cudaStream_t st) {
  if (d.nu <= 0) return cudaSuccess;
  const size_t sm = bf_kinfold_smem(d.nmax);
  cudaError_t e = cudaFuncSetAttribute(bf_k_kinfold, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  if (e != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(work_counter, 0, sizeof(int), st)) != cudaSuccess) return e;
  bf_k_kinfold<<<grid, kKfThreads, sm, st>>>(dP, d, ws, work_counter);
  return cudaGetLastError();
}
