// bf_findpath.cu -- direct refolding paths between two secondary structures (ViennaRNA's findpath) on the device (sm_100a).
//
// One run (a -> b, width w) is a breadth-limited search over direct paths.  Its moves are the deletions D (pairs of a not in b,
// ascending i), then the insertions I (pairs of b not in a, ascending i); a state is the set of moves done.  Level 0 is {a} with
// saddle E(a); level t+1 holds every valid one-move successor of the states kept at level t, saddle = max(parent saddle, E(child));
// successors with the same move set are one state that keeps the least (saddle, parent rank, move); the states are ordered by
// (saddle, E, parent rank, move) and the first w are kept.  E is bf_k_eval's energy (dangles = 2, non-standard pairs as type 7).
// A call runs w = 1, 2, 4, ... (the powers of two below W), then W, each forward (s1 -> s2) and reverse (s2 -> s1); the result is
// the run of least saddle, ties to the first run in that order.  tests/findpath_ref.c holds the same rules in plain C.
//
// Mapping: a unit of work is one run (instance, w, direction), dealt through a work counter to a persistent grid of 8-warp CTAs,
// widest runs first.  Each CTA owns an HBM workspace: the kept states of two levels (pair table, move bitset, E, saddle, 64-bit
// Zobrist hash of the move set) and the candidate keys of one level.  Per level:
//   1. every thread takes (parent, move) candidates, checks the move against the parent's pair table and forms E(child) as
//      E(parent) + dE, dE re-scoring only the loop closed by the moved pair and its enclosing loop (with dangles = 2 every loop
//      energy is local, so this is exact integer arithmetic); valid candidates append a 128-bit key (saddle, E | parent, move);
//   2. the CTA sorts the keys (bitonic network in the workspace);
//   3. it walks the sorted keys in chunks of 256 and keeps a candidate unless an earlier one -- kept, or earlier in its chunk --
//      has the same move set (hash equal, then an exact bitset compare: a hash match alone never merges), until w are kept;
//   4. it builds the kept states' pair tables and bitsets, and writes a back-pointer (parent rank, move, E) per kept state.
// bf_k_findpath_trace (a thread per instance) takes the run of least (saddle, run index) -- no atomics touch results -- and walks
// its back-pointers from the final state.
#include <algorithm>

#include "bf_kernels.h"

#include "bf_device.cuh"
#include "bf_loops.cuh"

namespace {

constexpr int kFpThreads = 256;
constexpr int kFpChunk = kFpThreads;

__host__ __device__ inline size_t al256(size_t x) { return (x + 255) / 256 * 256; }

struct FpLayout {
  size_t pt, bits, hash, e, sad, state, keys, total;
};
// one CTA's workspace: two levels of W states (pair tables of nmax + 2 shorts, bitsets of kw words, hash, E, saddle), then the keys
__host__ __device__ inline FpLayout fp_layout(int W, int nmax, int kw, long long cap) {
  FpLayout L;
  L.pt = 0;
  L.bits = al256((size_t)W * (nmax + 2) * sizeof(short));
  L.hash = L.bits + al256((size_t)W * kw * 8);
  L.e = L.hash + al256((size_t)W * 8);
  L.sad = L.e + al256((size_t)W * 4);
  L.state = L.sad + al256((size_t)W * 4);
  L.keys = 2 * L.state;
  L.total = L.keys + al256((size_t)cap * 16);
  return L;
}

__host__ __device__ inline long long fp_pow2(long long x) {
  long long p = 1;
  while (p < x) p <<= 1;
  return p;
}

// widths of the schedule: wi < nw - 1 -> 2^wi, wi = nw - 1 -> W
__host__ __device__ inline int fp_nw(int W) {
  int nw = 1;
  while ((1 << (nw - 1)) < W) nw++;
  return nw;
}
__host__ __device__ inline int fp_width(int W, int nw, int wi) { return wi == nw - 1 ? W : 1 << wi; }

__device__ __forceinline__ unsigned long long fp_zobrist(int m) {
  unsigned long long s = 0x243F6A8885A308D3ull * (unsigned long long)(m + 1);
  return sm64(s);
}

__device__ __forceinline__ bool fp_key_less(ulonglong2 a, ulonglong2 b) { return a.x < b.x || (a.x == b.x && a.y < b.y); }
__device__ __forceinline__ unsigned long long fp_hi(int sad, int e) {
  return ((unsigned long long)((unsigned)sad ^ 0x80000000u) << 32) | (unsigned)e ^ 0x80000000u;
}

// the move sets of candidates (p1, m1) and (p2, m2) are equal
__device__ bool fp_same_set(const unsigned long long *bits, int kw, int p1, int m1, int p2, int m2) {
  if (p1 == p2) return m1 == m2;
  const unsigned long long *b1 = bits + (size_t)p1 * kw, *b2 = bits + (size_t)p2 * kw;
  for (int w = 0; w < kw; w++) {
    const unsigned long long x = b1[w] | ((m1 >> 6) == w ? 1ull << (m1 & 63) : 0ull);
    const unsigned long long y = b2[w] | ((m2 >> 6) == w ? 1ull << (m2 & 63) : 0ull);
    if (x != y) return false;
  }
  return true;
}

struct FpState {
  short *pt;
  unsigned long long *bits, *hash;
  int *e, *sad;
};
__device__ FpState fp_state(unsigned char *base, const FpLayout &L) {
  FpState s;
  s.pt = reinterpret_cast<short *>(base + L.pt);
  s.bits = reinterpret_cast<unsigned long long *>(base + L.bits);
  s.hash = reinterpret_cast<unsigned long long *>(base + L.hash);
  s.e = reinterpret_cast<int *>(base + L.e);
  s.sad = reinterpret_cast<int *>(base + L.sad);
  return s;
}

__global__ void __launch_bounds__(kFpThreads) bf_k_findpath(const BfParams *__restrict__ P, BfFindpathDev d, unsigned char *ws,
                                                           int *work_counter) {
  __shared__ BfSmallI T;
  __shared__ uint8_t S[BF_FINDPATH_MAX_LEN + 2];
  __shared__ unsigned long long s_selhash[BF_FINDPATH_MAX_WIDTH], s_selkey[BF_FINDPATH_MAX_WIDTH];
  __shared__ unsigned s_selpm[BF_FINDPATH_MAX_WIDTH];
  __shared__ unsigned long long s_chash[kFpChunk];
  __shared__ unsigned s_cpm[kFpChunk];
  __shared__ int s_wcnt[kFpThreads / 32];
  __shared__ int s_unit, s_ncand, s_nsel;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nmax = d.nmax, kw = d.kw, W = d.width, nw = fp_nw(W);
  const FpLayout L = fp_layout(W, nmax, kw, d.cap);
  unsigned char *base = ws + (size_t)blockIdx.x * L.total;
  ulonglong2 *keys = reinterpret_cast<ulonglong2 *>(base + L.keys);
  bf_stage(&T, &P->si);
  const int units = d.n * 2 * nw;
  for (;;) {
    __syncthreads();
    if (tid == 0) s_unit = atomicAdd(work_counter, 1);
    __syncthreads();
    const int u = s_unit;
    if (u >= units) break;
    // widest runs first
    const int xo = u / d.n, r = u % d.n, wi = nw - 1 - (xo >> 1), dir = xo & 1, x = 2 * wi + dir;
    const int w = fp_width(W, nw, wi), n = d.len[r], d1 = d.nd[2 * r], d2 = d.nd[2 * r + 1], k = d1 + d2;
    const int *mv = d.mv + (size_t)r * d.stride;
    const int nd = dir ? d2 : d1;                  // deletions of this run come first
    auto move_pair = [&](int m) { return dir ? mv[m < d2 ? d1 + m : m - d2] : mv[m]; };
    // back-pointers of this run: level t (1 .. k), rank s at bp[(t - 1) * w + s]
    int sumw = 0;
    for (int y = 0; y < x; y++) sumw += fp_width(W, nw, y >> 1);
    int2 *bp = d.bp + d.bp_off[r] + (long long)k * sumw;
    const char *seq = d.seq + (size_t)r * d.stride;
    for (int y = tid; y <= n + 1; y += blockDim.x) S[y] = (uint8_t)((y >= 1 && y <= n) ? bf_base_code(seq[y - 1]) : 0);
    FpState cur = fp_state(base, L), nxt = fp_state(base + L.state, L);
    const short *pt0 = (dir ? d.pt2 : d.pt1) + (size_t)r * (d.stride + 2);
    for (int y = tid; y <= n + 1; y += blockDim.x) cur.pt[y] = pt0[y];
    for (int y = tid; y < kw; y += blockDim.x) cur.bits[y] = 0ull;
    __syncthreads();
    if (tid == 0) {
      const int e0 = fp_eval(P, T, S, n, cur.pt);
      cur.e[0] = e0; cur.sad[0] = e0; cur.hash[0] = 0ull;
      d.run_e0[(size_t)r * 2 * nw + x] = e0;
    }
    int npar = 1;
    const int ps = nmax + 2;   // pair-table stride of the workspace
    for (int t = 0; t < k; t++) {
      if (tid == 0) { s_ncand = 0; s_nsel = 0; }
      __syncthreads();
      // 1. candidates (parent, move) of this level
      const int ncand_all = npar * k;
      for (int c = tid; c < ncand_all; c += blockDim.x) {
        const int p = c / k, m = c % k;
        if ((cur.bits[(size_t)p * kw + (m >> 6)] >> (m & 63)) & 1ull) continue;
        const short *pt = cur.pt + (size_t)p * ps;
        const int ij = move_pair(m), i = ij >> 16, j = ij & 0xffff;
        int de;
        const int enc = fp_enclosing(pt, i);
        const FpView v0{pt, -1, -1, -1, -1};
        if (m < nd) {
          const FpView v1{pt, -1, -1, i, j};
          de = fp_loop(P, T, S, n, v1, enc) - fp_loop(P, T, S, n, v0, enc) - fp_loop(P, T, S, n, v0, i);
        } else {
          if (pt[i] || pt[j]) continue;
          bool ok = true;
          for (int y = i + 1; y < j;) {
            const int q = pt[y];
            if (q == 0) y++;
            else if (q > y && q < j) y = q + 1;
            else { ok = false; break; }
          }
          if (!ok) continue;
          const FpView v1{pt, i, j, -1, -1};
          de = fp_loop(P, T, S, n, v1, enc) + fp_loop(P, T, S, n, v1, i) - fp_loop(P, T, S, n, v0, enc);
        }
        const int e = cur.e[p] + de, sad = max(cur.sad[p], e);
        const int slot = atomicAdd(&s_ncand, 1);
        keys[slot] = make_ulonglong2(fp_hi(sad, e), ((unsigned long long)p << 16) | (unsigned)m);
      }
      __syncthreads();
      const int N = s_ncand;
      // 2. bitonic sort of the keys, padded to a power of two with keys above every candidate
      const long long Np = fp_pow2(N);
      for (long long y = N + tid; y < Np; y += blockDim.x) keys[y] = make_ulonglong2(~0ull, ~0ull);
      __syncthreads();
      for (long long size = 2; size <= Np; size <<= 1)
        for (long long st = size >> 1; st > 0; st >>= 1) {
          for (long long y = tid; y < Np / 2; y += blockDim.x) {
            const long long lo = 2 * st * (y / st) + (y % st), hi = lo + st;
            const ulonglong2 a = keys[lo], b = keys[hi];
            const bool up = (lo & size) == 0;
            if (fp_key_less(b, a) == up) { keys[lo] = b; keys[hi] = a; }
          }
          __syncthreads();
        }
      // 3. the first w distinct move sets in key order
      for (int c0 = 0; c0 < N; c0 += kFpChunk) {
        const int nsel = s_nsel;
        if (nsel >= w) break;
        const int c = c0 + tid;
        const bool valid = c < N;
        unsigned pm = 0;
        unsigned long long h = 0, hk = 0;
        if (valid) {
          const ulonglong2 kk = keys[c];
          pm = (unsigned)kk.y; hk = kk.x;
          h = cur.hash[pm >> 16] ^ fp_zobrist(pm & 0xffff);
        }
        s_chash[tid] = h; s_cpm[tid] = pm;
        __syncthreads();
        bool keep = valid;
        if (valid && npar > 1) {
          const int p = pm >> 16, m = pm & 0xffff;
          for (int s = 0; s < nsel && keep; s++)
            if (s_selhash[s] == h && fp_same_set(cur.bits, kw, p, m, s_selpm[s] >> 16, s_selpm[s] & 0xffff)) keep = false;
          for (int y = 0; y < tid && keep; y++)
            if (s_chash[y] == h && fp_same_set(cur.bits, kw, p, m, s_cpm[y] >> 16, s_cpm[y] & 0xffff)) keep = false;
        }
        const unsigned bal = __ballot_sync(BF_FULL, keep);
        if (lane == 0) s_wcnt[warp] = __popc(bal);
        __syncthreads();
        int off = 0, tot = 0;
        for (int y = 0; y < kFpThreads / 32; y++) { off += y < warp ? s_wcnt[y] : 0; tot += s_wcnt[y]; }
        const int pos = nsel + off + __popc(bal & ((1u << lane) - 1));
        if (keep && pos < w) { s_selhash[pos] = h; s_selpm[pos] = pm; s_selkey[pos] = hk; }
        __syncthreads();
        if (tid == 0) s_nsel = min(w, nsel + tot);
        __syncthreads();
      }
      const int nsel = s_nsel;
      // 4. the kept states of level t + 1 and their back-pointers
      for (long long y = tid; y < (long long)nsel * ps; y += blockDim.x) {
        const int s = (int)(y / ps), z = (int)(y % ps);
        nxt.pt[(size_t)s * ps + z] = cur.pt[(size_t)(s_selpm[s] >> 16) * ps + z];
      }
      for (int y = tid; y < nsel * kw; y += blockDim.x) {
        const int s = y / kw, z = y % kw, m = s_selpm[s] & 0xffff;
        nxt.bits[y] = cur.bits[(size_t)(s_selpm[s] >> 16) * kw + z] | ((m >> 6) == z ? 1ull << (m & 63) : 0ull);
      }
      __syncthreads();
      for (int s = tid; s < nsel; s += blockDim.x) {
        const int m = s_selpm[s] & 0xffff, ij = move_pair(m), i = ij >> 16, j = ij & 0xffff;
        short *pt = nxt.pt + (size_t)s * ps;
        if (m < nd) { pt[i] = 0; pt[j] = 0; }
        else { pt[i] = (short)j; pt[j] = (short)i; }
        const unsigned long long hk = s_selkey[s];
        const int e = (int)((unsigned)hk ^ 0x80000000u), sad = (int)((unsigned)(hk >> 32) ^ 0x80000000u);
        nxt.e[s] = e; nxt.sad[s] = sad; nxt.hash[s] = s_selhash[s];
        bp[(size_t)t * w + s] = make_int2((int)s_selpm[s], e);
      }
      __syncthreads();
      const FpState tmp = cur; cur = nxt; nxt = tmp;
      npar = nsel;
    }
    if (tid == 0) d.run_sad[(size_t)r * 2 * nw + x] = cur.sad[0];
  }
}

// a thread per instance: the run of least (saddle, run index), walked back from its final state
__global__ void __launch_bounds__(128) bf_k_findpath_trace(BfFindpathDev d, int *saddle, int *moves, int *path_e) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= d.n) return;
  const int W = d.width, nw = fp_nw(W), R = 2 * nw;
  const int d1 = d.nd[2 * r], d2 = d.nd[2 * r + 1], k = d1 + d2;
  int bx = 0;
  for (int x = 1; x < R; x++)
    if (d.run_sad[(size_t)r * R + x] < d.run_sad[(size_t)r * R + bx]) bx = x;
  saddle[r] = d.run_sad[(size_t)r * R + bx];
  if (!moves && !path_e) return;
  const int dir = bx & 1, w = fp_width(W, nw, bx >> 1), nd = dir ? d2 : d1;
  const int *mv = d.mv + (size_t)r * d.stride;
  int sumw = 0;
  for (int y = 0; y < bx; y++) sumw += fp_width(W, nw, y >> 1);
  const int2 *bp = d.bp + d.bp_off[r] + (long long)k * sumw;
  int *mo = moves ? moves + (size_t)r * d.stride * 2 : nullptr;
  int *pe = path_e ? path_e + (size_t)r * (d.stride + 1) : nullptr;
  int rank = 0;
  for (int t = k; t >= 1; t--) {
    const int2 b = bp[(size_t)(t - 1) * w + rank];
    const int m = b.x & 0xffff;
    rank = b.x >> 16;
    // step t of this run is step k + 1 - t of the path from s1 when the run is reverse
    const int step = dir ? k - t : t - 1;
    const int ij = dir ? mv[m < d2 ? d1 + m : m - d2] : mv[m], i = ij >> 16, j = ij & 0xffff;
    const bool del = m < nd, ins_fwd = dir ? del : !del;
    if (mo) { mo[2 * step] = ins_fwd ? i : -i; mo[2 * step + 1] = ins_fwd ? j : -j; }
    if (pe) pe[dir ? k - t : t] = b.y;
  }
  if (pe) pe[dir ? k : 0] = d.run_e0[(size_t)r * R + bx];
}

}  // namespace

size_t bf_findpath_ws_bytes(int width, int nmax, int kw, long long cap) { return fp_layout(width, nmax, kw, cap).total; }
long long bf_findpath_cap(int width, int kmax) { return fp_pow2(std::max<long long>(1, (long long)width * kmax)); }
int bf_findpath_runs(int width) { return 2 * fp_nw(width); }
int bf_findpath_width_sum(int width) {
  const int nw = fp_nw(width);
  int s = 0;
  for (int wi = 0; wi < nw; wi++) s += 2 * fp_width(width, nw, wi);
  return s;
}

cudaError_t bf_launch_findpath(const BfParams *dP, const BfFindpathDev &d, unsigned char *ws, int grid, int *work_counter, int *saddle,
                               int *moves, int *path_e, cudaStream_t st) {
  if (d.n <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  bf_k_findpath<<<grid, kFpThreads, 0, st>>>(dP, d, ws, work_counter);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  bf_k_findpath_trace<<<(d.n + 127) / 128, 128, 0, st>>>(d, saddle, moves, path_e);
  return cudaGetLastError();
}

int bf_findpath_occupancy() {
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bf_k_findpath, kFpThreads, 0) != cudaSuccess) return 1;
  return std::max(occ, 1);
}
