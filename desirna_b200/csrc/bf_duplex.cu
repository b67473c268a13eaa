// bf_duplex.cu -- RNA-RNA hybridization: the lowest-energy purely intermolecular structure of strands a and b (sm_100a).
//
// ViennaRNA's duplexfold (RNAduplex), restated from its published recurrence; no ViennaRNA output in this tree pins it.  A duplex is
// a chain of pairs (k1,l1), ..., (km,lm) of a[k] with b[l], k increasing, l decreasing, at most 30 unpaired nucleotides between
// consecutive pairs.  Its energy is the engine's two-strand eval_structure of that structure on a&b: DuplexInit, the exterior stem
// of the outermost pair, one interior loop per step, and the nick loop closed by the innermost pair.  Over cells (i,j), pair a[i]b[j]
// the innermost pair so far:
//
//   c(i,j) = DuplexInit + Ext(type(i,j), a[i-1], b[j+1])
//            min over k < i, l > j, (i-k-1) + (l-j-1) <= 30:  c(k,l) + IntLoop(i-k-1, l-j-1, type(k,l), rtype(type(i,j)), ...)
//   E(a,b) = min over (i,j) of c(i,j) + Ext(rtype(type(i,j)), b[j-1], a[i+1])            neighbours only where they exist
//
// Ties: the end cell is the first minimum in the order i ascending, then j descending; the backtrack from (i,j) takes the first
// (k,l) with c(i,j) = c(k,l) + IntLoop in the order k = i-1 downwards, then l = j+1 upwards.  tests/duplex_ref.c holds the same
// rules in plain C.
//
// Mapping: one CTA of four warps per (a, b) pair; cells are swept by anti-diagonal w = i + y, y = n2 + 1 - j, one barrier per
// diagonal.  Every dependency lies 2..32 diagonals back, so c lives in a ring of 33 diagonals in shared memory, indexed along the
// shorter strand.  A warp takes one pairable cell of the diagonal and its lanes run over the <= 496 (u1, u2) loop candidates
// (__reduce_min_sync); the end-cell minimum is kept as a packed (energy, rank) key, so the tie rule holds whatever the order in
// which warps meet the cells.  Structures: the CTA also writes its c table (n1 x n2 int32) to an HBM workspace and warp 0 walks it
// back after the sweep.  A ring that does not fit shared memory (both strands longer than ~1650 nt) lives in HBM instead.
#include <algorithm>

#include "bf_kernels.h"

#include "bf_device.cuh"

namespace {

constexpr int kDxWarps = 4;
constexpr int kRing = 33;   // diagonals w-32 .. w
constexpr long long kKeyInf = 0x7fffffffffffffffll;

__host__ __device__ inline size_t al16(size_t x) { return (x + 15) / 16 * 16; }

struct PairLens { int ia, ib; };
__device__ __forceinline__ PairLens pair_of(const BfDuplexDev &d, long long p) {
  PairLens r;
  if (d.pairs) { r.ia = d.pairs[2 * p]; r.ib = d.pairs[2 * p + 1]; }
  else { r.ia = (int)(p / d.nb); r.ib = (int)(p % d.nb); }
  return r;
}

// GRING: the ring lives in HBM (gring + blockIdx.x * ring_slot ints) instead of shared memory
template <bool GRING>
__global__ void __launch_bounds__(kDxWarps * 32, 8) bf_k_duplex(const BfParams *__restrict__ P, BfDuplexDev d, int *gring,
                                                                 size_t ring_slot, int *e_out, int *ctab, const long long *__restrict__ ctab_off,
                                                                 char *ss_out, int ss_stride) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ BfSmallI T;
  __shared__ unsigned char s_fill[BF_NCAND][2];  // s = u1 + u2 and u1, s-major: candidate x = s(s+1)/2 + u1
  __shared__ unsigned char s_bt[BF_NCAND][2];    // u1 and u2, u1-major: the backtrack's order
  __shared__ long long s_key[kDxWarps];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long p = d.p0 + blockIdx.x;
  const PairLens pl = pair_of(d, p);
  const int n1 = d.len_a[pl.ia], n2 = d.len_b[pl.ib];
  const bool by_i = n1 <= n2;           // ring index: i - 1 along a, else y - 1 along b
  const int width = by_i ? n1 : n2;
  int *ring = GRING ? gring + (size_t)blockIdx.x * ring_slot : reinterpret_cast<int *>(dyn);
  uint8_t *A = dyn + (GRING ? 0 : al16((size_t)kRing * d.ring_w * sizeof(int)));
  uint8_t *Bs = A + al16(d.amax + 2);
  const char *sa = d.seq_a + (size_t)pl.ia * d.stride_a, *sb = d.seq_b + (size_t)pl.ib * d.stride_b;
  for (int k = tid; k <= n1 + 1; k += blockDim.x) A[k] = (uint8_t)((k >= 1 && k <= n1) ? bf_base_code(sa[k - 1]) : 0);
  for (int k = tid; k <= n2 + 1; k += blockDim.x) Bs[k] = (uint8_t)((k >= 1 && k <= n2) ? bf_base_code(sb[k - 1]) : 0);
  bf_stage(&T, &P->si);
  for (int x = tid; x < BF_NCAND; x += blockDim.x) {
    int s = 0;
    while ((s + 1) * (s + 2) / 2 <= x) s++;
    s_fill[x][0] = (unsigned char)s;
    s_fill[x][1] = (unsigned char)(x - s * (s + 1) / 2);
    int u1 = 0, r = x;
    while (r >= 31 - u1) { r -= 31 - u1; u1++; }
    s_bt[x][0] = (unsigned char)u1;
    s_bt[x][1] = (unsigned char)r;
  }
  int *ct = ctab ? ctab + ctab_off[blockIdx.x] : nullptr;
  __syncthreads();

  long long best = kKeyInf;
  for (int w = 2; w <= n1 + n2; w++) {
    const int ilo = max(1, w - n2), ihi = min(n1, w - 1);
    int *rw = ring + (w % kRing) * width;
    for (int i = ilo + warp; i <= ihi; i += kDxWarps) {
      const int j = n2 + 1 - (w - i);
      const int t = bf_ptype_bases(A[i], Bs[j]);
      int c = BF_INF;
      if (t) {
        const int ai = i > 1 ? A[i - 1] : -1, bj = j < n2 ? Bs[j + 1] : -1;
        const int um1 = i - 2, um2 = n2 - j - 1;   // u1 <= i - 2 keeps k >= 1, u2 <= n2 - j - 1 keeps l <= n2
        int m = BF_INF;
        if (um1 >= 0 && um2 >= 0) {
          const int smax = min(BF_MAXLOOP, um1 + um2), ncand = (smax + 1) * (smax + 2) / 2, rt = bf_rtype(t);
          for (int x = lane; x < ncand; x += 32) {
            const int s = s_fill[x][0], u1 = s_fill[x][1], u2 = s - u1;
            if (u1 > um1 || u2 > um2) continue;
            const int k = i - 1 - u1, l = j + 1 + u2;
            const int ck = ring[((w - s - 2) % kRing) * width + (by_i ? k - 1 : n2 - l)];
            if (ck >= BF_INF) continue;
            const int tk = bf_ptype_bases(A[k], Bs[l]);
            m = min(m, ck + bf_e_intloop(P, T, u1, u2, tk, rt, A[k + 1], Bs[l - 1], ai, bj));
          }
          m = bf_warp_min(m);
        }
        c = min(T.DuplexInit + bf_e_ext(T, t, ai, bj), m);
        const int v = c + bf_e_ext(T, bf_rtype(t), j > 1 ? Bs[j - 1] : -1, i < n1 ? A[i + 1] : -1);
        best = min(best, (long long)v * 4294967296ll + (long long)((i - 1) * n2 + (n2 - j)));
      }
      if (lane == 0) {
        rw[by_i ? i - 1 : w - i - 1] = c;
        if (ct) ct[(size_t)(i - 1) * n2 + (j - 1)] = c;
      }
    }
    __syncthreads();
  }
  if (lane == 0) s_key[warp] = best;
  __syncthreads();
  best = s_key[0];
  for (int k = 1; k < kDxWarps; k++) best = min(best, s_key[k]);
  const long long q = blockIdx.x;
  if (tid == 0) e_out[q] = best == kKeyInf ? BF_INF : (int)(best >> 32);
  if (!ss_out) return;
  char *ss = ss_out + q * ss_stride;
  for (int k = tid; k < ss_stride; k += blockDim.x) ss[k] = k < n1 || (k > n1 && k <= n1 + n2) ? '.' : k == n1 ? '&' : '\0';
  __syncthreads();
  if (warp != 0 || best == kKeyInf) return;
  const int rank = (int)(best & 0xffffffffll);
  int i = rank / n2 + 1, j = n2 - rank % n2;
  while (true) {
    if (lane == 0) { ss[i - 1] = '('; ss[n1 + j] = ')'; }
    const int cij = ct[(size_t)(i - 1) * n2 + (j - 1)], rt = bf_rtype(bf_ptype_bases(A[i], Bs[j]));
    const int um1 = i - 2, um2 = n2 - j - 1;
    int found = -1;
    for (int base = 0; base < BF_NCAND && found < 0 && um1 >= 0 && um2 >= 0; base += 32) {
      const int x = base + lane;
      bool hit = false;
      if (x < BF_NCAND) {
        const int u1 = s_bt[x][0], u2 = s_bt[x][1];
        if (u1 <= um1 && u2 <= um2) {
          const int k = i - 1 - u1, l = j + 1 + u2, ck = ct[(size_t)(k - 1) * n2 + (l - 1)];
          hit = ck < BF_INF && cij == ck + bf_e_intloop(P, T, u1, u2, bf_ptype_bases(A[k], Bs[l]), rt, A[k + 1], Bs[l - 1], A[i - 1], Bs[j + 1]);
        }
      }
      const unsigned h = __ballot_sync(BF_FULL, hit);
      if (h) found = base + __ffs(h) - 1;
    }
    if (found < 0) break;
    i -= 1 + s_bt[found][0];
    j += 1 + s_bt[found][1];
  }
}

}  // namespace

namespace {
size_t duplex_smem(const BfDuplexDev &d, bool gring) {
  return (gring ? 0 : al16((size_t)kRing * d.ring_w * sizeof(int))) + al16(d.amax + 2) + al16(d.bmax + 2);
}
}  // namespace

// The static tables of bf_k_duplex (loop parameters, candidate orders) take less than 8 KB.
bool bf_duplex_gring(const BfDuplexDev &d) { return duplex_smem(d, false) > kSmemBudget - 8192; }

size_t bf_duplex_ring_slot(int ring_w) { return (size_t)kRing * ring_w; }

cudaError_t bf_launch_duplex(const BfParams *dP, const BfDuplexDev &d, bool gring, int *gring_ws, int *e_out, int *ctab,
                             const long long *ctab_off, char *ss_out, int ss_stride, cudaStream_t st) {
  if (d.np <= 0) return cudaSuccess;
  const size_t sm = duplex_smem(d, gring);
  auto kern = gring ? bf_k_duplex<true> : bf_k_duplex<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(sm, 1024));
  if (e != cudaSuccess) return e;
  kern<<<d.np, kDxWarps * 32, sm, st>>>(dP, d, gring_ws, bf_duplex_ring_slot(d.ring_w), e_out, ctab, ctab_off, ss_out, ss_stride);
  return cudaGetLastError();
}
