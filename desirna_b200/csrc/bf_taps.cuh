// bf_taps.cuh -- tap tables of the interior-loop candidates (shared by bf_fill3.cu and bf_cluster.cu).
//
// The decomposable interior-loop candidates of a cell (i,j) on diagonal d are  ring_kind[(d-2-s) mod depth][i+1+u1] + pen_kind(s,u1):
// the same 487 (row, column offset, penalty) "taps" for every cell.  Lanes run over the taps; the host assigns taps to (slot, lane)
// so that the 32 lanes of a slot hit 32 different shared-memory banks (recurrences: SURVEY.md A.4-A.6; the reference reaches them
// through fc.mfe() / fc.pf(), utils/energy_scores.py:150-151).
#pragma once
#include <cstdint>
#include <cstring>
#include <mutex>
#include <vector>

#include "bf_device.cuh"
#include "bf_kernels.h"

namespace {

constexpr int kRing = 32;
constexpr int kInfThr = BF_INF / 2;
constexpr int kNSG = 12, kNS1 = 3, kNSB = 3, kNSlot = kNSG + kNS1 + kNSB + 1;   // + the slot of the nine special candidates

__device__ __forceinline__ int ptype_sp(const uint8_t *SP, int i, int j) { return bf_ptype_bases(SP[i], SP[j]); }

// (u1, u2) of the nine non-decomposable interior candidates: stack, bulge-1 (2x), 1x1, 1x2, 2x1, 2x2, 2x3, 3x2
__host__ __device__ __forceinline__ int special_u1(int k) { return (int)((0x322211100ull >> (4 * k)) & 15); }
__host__ __device__ __forceinline__ int special_u2(int k) { return (int)((0x232121010ull >> (4 * k)) & 15); }

// slots a diagonal needs, by its largest loop size smax = min(30, d - 6) (index smax + 1); stored behind the tap words
struct TapMeta {
  unsigned char ng[32], n1[32], nb[32];
};

// ---------------------------------------------------------------------------------------------
// host: tap -> (slot, lane) assignment
// ---------------------------------------------------------------------------------------------
struct TapTable {
  uint32_t tap[kNSlot][32];   // s | u1 << 8 | valid << 16
  TapMeta meta;
  bool ok = false;
};

// M = 32: 4-byte ring entries, one bank per entry; M = 16: 8-byte entries, conflicts counted within each half-warp
TapTable build_taps(int c, int M) {
  TapTable tt;
  memset(&tt, 0, sizeof tt);
  bool ok = true;
  int first = 0;
  for (int kind = 0; kind < 3; kind++) {
    const int nslot = kind == 0 ? kNSG : kind == 1 ? kNS1 : kNSB;
    std::vector<std::pair<int, int>> T;
    if (kind == 0) { for (int s = 6; s <= 30; s++) for (int u1 = 2; u1 <= s - 2; u1++) T.push_back({s, u1}); }
    else if (kind == 1) { for (int s = 4; s <= 30; s++) { T.push_back({s, 1}); T.push_back({s, s - 1}); } }
    else { for (int s = 2; s <= 30; s++) { T.push_back({s, 0}); T.push_back({s, s}); } }
    std::vector<std::vector<int>> lanes(nslot, std::vector<int>(32, -1));   // index into T
    const int halves = M == 16 ? 2 : 1, per = 32 / halves;
    std::vector<std::pair<int, int>> left;
    for (int ti = 0; ti < (int)T.size(); ti++) {
      const int b = (((T[ti].second - T[ti].first * c) % M) + M) % M;
      bool placed = false;
      for (int k = 0; k < nslot && !placed; k++)
        for (int h = 0; h < halves && !placed; h++) {
          int free_lane = -1;
          bool clash = false;
          for (int l = h * per; l < (h + 1) * per; l++) {
            if (lanes[k][l] < 0) { if (free_lane < 0) free_lane = l; continue; }
            const auto &o = T[lanes[k][l]];
            if (((((o.second - o.first * c) % M) + M) % M) == b) clash = true;
          }
          if (!clash && free_lane >= 0) { lanes[k][free_lane] = ti; placed = true; }
        }
      if (!placed) left.push_back({ti, 0});
    }
    // what did not fit without a bank conflict goes wherever a lane is free (a two-way conflict on that slot)
    for (auto &lf : left) {
      bool placed = false;
      for (int k = nslot - 1; k >= 0 && !placed; k--)
        for (int l = 0; l < 32 && !placed; l++)
          if (lanes[k][l] < 0) { lanes[k][l] = lf.first; placed = true; }
      if (!placed) ok = false;
    }
    if (left.size() > 4) ok = false;
    unsigned char *need = kind == 0 ? tt.meta.ng : kind == 1 ? tt.meta.n1 : tt.meta.nb;
    for (int k = 0; k < nslot; k++) {
      int mins = 99;
      for (int l = 0; l < 32; l++) {
        if (lanes[k][l] < 0) continue;
        const auto &t = T[lanes[k][l]];
        tt.tap[first + k][l] = (uint32_t)t.first | ((uint32_t)t.second << 8) | (1u << 16);
        mins = std::min(mins, t.first);
      }
      for (int smax = -1; smax <= 30; smax++)
        if (mins <= smax) need[smax + 1] = (unsigned char)(k + 1);   // slots 0..k are needed
    }
    first += nslot;
  }
  // last slot: the nine non-decomposable candidates read the bulge ring at (s, u1) = (u1 + u2, u1); the other lanes read a valid
  // address and add the INF of the entry's padding
  for (int l = 0; l < 32; l++) {
    const int u1 = l < 9 ? special_u1(l) : 0, u2 = l < 9 ? special_u2(l) : 0;
    tt.tap[kNSlot - 1][l] = (uint32_t)(u1 + u2) | ((uint32_t)u1 << 8) | (1u << 16);
  }
  tt.ok = ok;
  return tt;
}

// smallest row stride >= want whose residue packs (cached per residue)
struct TapCache {
  TapTable t[2][32];
  bool have[2][32] = {};
  uint32_t *dev[2][32] = {};
  std::mutex mu;
};
TapCache g_taps;

const TapTable &taps_for(int rs, int M) {
  const int w = M == 16 ? 1 : 0, c = rs % M;
  if (!g_taps.have[w][c]) { g_taps.t[w][c] = build_taps(c, M); g_taps.have[w][c] = true; }
  return g_taps.t[w][c];
}
int pick_rs(int nmax, int M) {
  for (int rs = nmax + 2 > 40 ? nmax + 2 : 40;; rs++)   // column offsets reach 31: keep them inside one row
    if (taps_for(rs, M).ok) return rs;
}
cudaError_t taps_device(int rs, int M, const uint32_t **out) {
  const int w = M == 16 ? 1 : 0, c = rs % M;
  std::lock_guard<std::mutex> lk(g_taps.mu);
  const TapTable &t = taps_for(rs, M);
  if (!g_taps.dev[w][c]) {
    // device image: the tap words, then the slots-needed table (TapMeta)
    cudaError_t e = cudaMalloc(&g_taps.dev[w][c], sizeof t.tap + sizeof t.meta);
    if (e != cudaSuccess) return e;
    e = cudaMemcpy(g_taps.dev[w][c], t.tap, sizeof t.tap, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return e;
    e = cudaMemcpy(reinterpret_cast<unsigned char *>(g_taps.dev[w][c]) + sizeof t.tap, &t.meta, sizeof t.meta, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return e;
  }
  *out = g_taps.dev[w][c];
  return cudaSuccess;
}

}  // namespace
