// bf_design.cu -- move generator, Metropolis acceptance and replica exchange of the design loop, on the device (sm_100a).
//
// What the reference does per Monte-Carlo sub-step on the host, one Python process per replica
// (utils/replica_exchange_monte_carlo.py:176-210, utils/sequence_utils.py:926-1136), is done here for every replica of
// every design problem at once; the fold kernels (bf_fill.cu) run between bf_k_design_propose and bf_k_design_accept
// on the same stream.  One warp per batch row; the few serial pieces (bracket matching, the draw itself) run on lane 0.
//
// Random numbers: one splitmix64 stream per replica (moves and Metropolis tests) and one per job (neighbour swaps), the
// device counterpart of the reference's per-worker `random.seed(replica)` streams (:227-228) and of the parent stream
// that drives replica_exchange (:113-173).  The draws are the same KIND of draws in the same order as the reference's
// (choose range, choose position, choose letter(s), Metropolis test only when the mutant is worse); the generator is not
// Python's Mersenne twister, so trajectories agree in distribution, not bit for bit.
#include "bf_design.h"

#include "bf_device.cuh"

namespace {

constexpr int kWPB = 4;  // warps (rows) per CTA

__device__ __forceinline__ int below(unsigned long long &s, int n) {
  const int k = (int)(u01(s) * (double)n);
  return k < n ? k : n - 1;
}

__device__ __forceinline__ int letter_code(char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : 3; }
__device__ __forceinline__ char code_letter(int k) { return "ACGU"[k & 3]; }
// letters that pair with letter k (sequence_utils.py:607-622): A-U, C-G, G-{C,U}, U-{A,G}
__device__ __forceinline__ unsigned pair_mask(int k) { return k == 0 ? 8u : k == 1 ? 4u : k == 2 ? 10u : 5u; }

// k-th set bit (k < popc(m)) of a 4-bit mask
__device__ __forceinline__ int kth_bit(unsigned m, int k) {
  for (int b = 0; b < 4; b++)
    if (m >> b & 1u) { if (k == 0) return b; k--; }
  return 0;
}
// random.choice over the letters of m, or random.choices with the nucleotide weights (letters in sorted order A C G U)
__device__ int pick_letter(unsigned m, bool weighted, const BfDesignCfg &C, unsigned long long &rng) {
  if (!weighted) return kth_bit(m, below(rng, __popc(m)));
  double tot = 0.0;
  for (int b = 0; b < 4; b++) if (m >> b & 1u) tot += C.nt_weight[b];
  const double x = u01(rng) * tot;
  double cum = 0.0;
  int last = 0;
  for (int b = 0; b < 4; b++)
    if (m >> b & 1u) { cum += C.nt_weight[b]; last = b; if (x < cum) return b; }
  return last;
}

// dot-bracket -> partner table (lane 0; balanced strings as produced by bf_k_trace); characters other than ( ) are unpaired
__device__ void pair_table(const char *ss, int n, short *pt, short *stk) {
  int sp = 0;
  bool other = false;
  for (int i = 0; i < n; i++) {
    const char ch = ss[i];
    pt[i] = -1;
    if (ch == '(') stk[sp++] = (short)i;
    else if (ch == ')' && sp > 0) { const int j = stk[--sp]; pt[i] = (short)j; pt[j] = (short)i; }
    else if (ch != '.') other = true;
  }
  if (!other) return;
  // pseudoknot overlay: one more pass per bracket family present (check_dot_bracket, sequence_utils.py:74-116)
  for (int f = 0; f < 3; f++) {
    const char opn = "[<{"[f], cls = "]>}"[f];
    sp = 0;
    for (int i = 0; i < n; i++) {
      const char ch = ss[i];
      if (ch == opn) stk[sp++] = (short)i;
      else if (ch == cls && sp > 0) { const int j = stk[--sp]; pt[i] = (short)j; pt[j] = (short)i; }
    }
  }
}

struct WarpScratch { short *pt, *stk; uint8_t *fl; };
__device__ __forceinline__ WarpScratch scratch(unsigned char *dyn, int stride, int warp) {
  const size_t per = ((size_t)5 * stride + 15) / 16 * 16;
  unsigned char *b = dyn + per * warp;
  WarpScratch w;
  w.pt = reinterpret_cast<short *>(b);
  w.stk = w.pt + stride;
  w.fl = reinterpret_cast<uint8_t *>(w.stk + stride);
  return w;
}
size_t scratch_bytes(int stride) { return ((size_t)5 * stride + 15) / 16 * 16 * kWPB; }

// uniform choice among the positions v in [lo, hi] with flag(v) set; cnt = number of such positions (> 0)
template <typename F>
__device__ int choose_flagged(F flag, int lo, int hi, int cnt, unsigned long long &rng, int lane) {
  int k = below(rng, cnt);
  for (int base = lo; base <= hi; base += 32) {
    const int v = base + lane;
    const unsigned mk = __ballot_sync(BF_FULL, v <= hi && flag(v));
    const int c = __popc(mk);
    if (k < c) {
      unsigned m = mk;
      for (int t = 0; t < k; t++) m &= m - 1;
      return base + __ffs(m) - 1;
    }
    k -= c;
  }
  return lo;
}

// ------------------------------------------------------------------------------------------------ gather
// row_len / row_tgt of the active rows (after the set of active jobs changed)
__global__ void bf_k_design_gather(BfDesignDev D, int B) {
  const int lane = threadIdx.x & 31, row = blockIdx.x * kWPB + (threadIdx.x >> 5);
  if (row >= B) return;
  const int job = D.rowmap[row] / D.R;
  if (lane == 0) { D.row_len[row] = D.len[job]; D.row_cut[row] = D.len_a[job] > 0 ? D.len_a[job] + 1 : 0; }
  for (int t = 0; t < D.T; t++) {
    const char *src = (t >= 1 && t - 1 < D.n_alt[job]) ? D.alt + ((size_t)job * D.max_alt + (t - 1)) * D.stride : D.tgt + (size_t)job * D.stride;
    for (int k = lane; k < D.stride; k += 32) D.row_tgt[((size_t)row * D.T + t) * D.stride + k] = src[k];
  }
}

// ------------------------------------------------------------------------------------------------ negative design
// which rows fold into their target (1 - MCC == 0 in the accept kernel): only those need the second-best structure
__global__ void __launch_bounds__(kWPB * 32) bf_k_design_nd_flag(BfDesignDev D, int B) {
  extern __shared__ __align__(16) unsigned char dyn[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, row = blockIdx.x * kWPB + warp;
  if (row >= B) return;
  const int g = D.rowmap[row], job = g / D.R, n = D.len[job], S = D.stride;
  WarpScratch w = scratch(dyn, S, warp);
  if (lane == 0) pair_table(D.o_ss + (size_t)row * (S + 1), n, w.pt, w.stk);
  __syncwarp();
  const short *tpt = D.tpt + (size_t)job * S;
  bool same = true;
  for (int i = lane; i < n; i += 32) same = same && tpt[i] == w.pt[i];
  same = __all_sync(BF_FULL, same);
  if (lane == 0) D.nd_flag[row] = same ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------ pseudoknot overlay
__global__ void bf_k_design_pk_mask(BfDesignDev D, int B) {
  const int lane = threadIdx.x & 31, row = blockIdx.x * kWPB + (threadIdx.x >> 5);
  if (row >= B) return;
  const char *ss = D.o_ss + (size_t)row * (D.stride + 1);
  for (int k = lane; k < D.stride; k += 32) D.pk_nopair[(size_t)row * D.stride + k] = (k < D.row_len[row] && ss[k] != '.') ? 1 : 0;
}
__global__ void bf_k_design_pk_paint(BfDesignDev D, int B, int round) {
  const int lane = threadIdx.x & 31, row = blockIdx.x * kWPB + (threadIdx.x >> 5);
  if (row >= B) return;
  char *ss = D.o_ss + (size_t)row * (D.stride + 1);
  const char *s2 = D.o_ss2 + (size_t)row * (D.stride + 1);
  const char opn = "[<{"[round], cls = "]>}"[round];
  for (int k = lane; k < D.row_len[row]; k += 32) {
    if (s2[k] == '(') ss[k] = opn;
    else if (s2[k] == ')') ss[k] = cls;
  }
}

// ------------------------------------------------------------------------------------------------ propose
// avoid designs: the row's self-dimer, the finished mutant twice ('&' is the cut, n + 1, as engine.pack sets it)
__device__ __forceinline__ void self_dimer_row(const BfDesignDev &D, const BfDesignCfg &C, int row, const char *mut, int n, int lane) {
  if (C.oligo != 3) return;
  __syncwarp();
  char *d = D.dimer_seq + (size_t)row * 2 * D.stride;
  for (int k = lane; k < 2 * n; k += 32) d[k] = mut[k < n ? k : k - n];
  if (lane == 0) { D.dimer_len[row] = 2 * n; D.dimer_cut[row] = n + 1; }
}

// mutate_sequence + get_mutation_position (sequence_utils.py:926-1136) without the scoring call at its end
__global__ void __launch_bounds__(kWPB * 32) bf_k_design_propose(BfDesignDev D, BfDesignCfg C, int B, int copy_only) {
  extern __shared__ __align__(16) unsigned char dyn[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, row = blockIdx.x * kWPB + warp;
  if (row >= B) return;
  const int g = D.rowmap[row], job = g / D.R, n = D.len[job], S = D.stride;
  const char *cur = D.cur_seq + (size_t)g * S;
  char *mut = D.mut_seq + (size_t)row * S;
  for (int k = lane; k < S; k += 32) mut[k] = cur[k];
  if (lane == 0) D.row_scale[row] = D.cur_mfe[g];
  const int n_avail = D.n_avail[job];
  if (copy_only || n_avail == 0) {   // initial scoring: the "mutant" is the start sequence itself; or nothing to mutate
    self_dimer_row(D, C, row, mut, n, lane);
    return;
  }
  const short *tpt = D.tpt + (size_t)job * S;
  const uint8_t *allowed = D.allowed + (size_t)job * S;
  const unsigned short *avail = D.avail + (size_t)job * S;
  unsigned long long rng = D.rng[g];   // every lane advances an identical copy; lane 0 writes it back
  WarpScratch w = scratch(dyn, S, warp);

  int pos;
  if (!C.point_mutations) {
    pos = avail[below(rng, n_avail)];
  } else {
    if (lane == 0) pair_table(D.cur_ss + (size_t)g * (S + 1), n, w.pt, w.stk);
    __syncwarp();
    // positions of pairs present in only one of {target, MFE structure}, if mutable (sequence_utils.py:951-962)
    int nfalse = 0;
    for (int base = 0; base < n; base += 32) {
      const int i = base + lane;
      const bool f = i < n && tpt[i] != w.pt[i] && __popc(allowed[i]) > 1;
      if (i < n) w.fl[i] = f;
      nfalse += __popc(__ballot_sync(BF_FULL, f));
    }
    __syncwarp();
    bool targeted = false;
    int cnt = 0;
    // expand_cases(false_cases, len - 1, 3): every v in [1, len-1] within 3 of a flagged position (sequence_utils.py:983-1005).
    // The reference's strings carry the '&' of a two-strand design: positions are compared in those coordinates (A = index of
    // the '&'), and the '&' itself can be drawn -- a move that changes nothing (its restraint allows one letter).
    const int A = D.len_a[job];
    const int hi = A > 0 ? n : n - 1;
    auto near = [&](int v) {
      bool e = false;
      for (int o = -3; o <= 3; o++) {
        const int ua = v + o;                       // '&' coordinates
        if (ua < 0 || (A > 0 && ua == A)) continue;
        const int u = ua - (A > 0 && ua > A);       // nucleotide index
        e |= (u < n && w.fl[u]);
      }
      return e;
    };
    if (nfalse > 0) {
      for (int base = 1; base <= hi; base += 32) {
        const int v = base + lane;
        cnt += __popc(__ballot_sync(BF_FULL, v <= hi && near(v)));
      }
      // random.choices([false_cases, available_positions], weights=[p, 1-p])
      targeted = u01(rng) < D.tm_prob[D.shelf[g]];
    }
    if (targeted && cnt > 0) {
      const int va = choose_flagged(near, 1, hi, cnt, rng, lane);
      pos = (A > 0 && va == A) ? -1 : va - (A > 0 && va > A);
    } else pos = avail[below(rng, n_avail)];
  }
  __syncwarp();
  if (lane == 0 && pos < 0) D.rng[g] = rng;
  if (lane == 0 && pos >= 0) {
    const int curl = letter_code(cur[pos]);
    const unsigned a1 = allowed[pos];
    const int partner = D.mpt ? D.mpt[(size_t)job * S + pos] : tpt[pos];
    const int snake = D.snake_id ? D.snake_id[(size_t)job * S + pos] : -1;
    if (snake >= 0) {
      // a node of a conflict graph: the whole graph jumps to another of its colourings (sequence_utils.py:1085-1094)
      const char *sl = D.snake_letter + ((size_t)job * S + pos) * 4;
      int now = -1, nstates = 0;
      for (int s = 0; s < 4; s++) {
        if (sl[s]) nstates++;
        if (now < 0 && sl[s] == cur[pos]) now = s;
      }
      const int others = nstates - (now >= 0 ? 1 : 0);
      if (others > 0) {
        int k = below(rng, others), pick = -1;
        for (int s = 0; s < 4 && pick < 0; s++)
          if (sl[s] && s != now && k-- == 0) pick = s;
        const signed char *sid = D.snake_id + (size_t)job * S;
        for (int x = 0; x < n; x++)
          if (sid[x] == snake) mut[x] = D.snake_letter[((size_t)job * S + x) * 4 + pick];
      }
    } else if (partner < 0) {
      if (__popc(a1) > 1) {
        unsigned m = a1 & ~(1u << curl);
        if (!m) m = a1;
        mut[pos] = code_letter(pick_letter(m, false, C, rng));
      }
    } else {
      unsigned m1 = a1;
      if ((m1 >> curl & 1u) && __popc(m1) != 1) m1 &= ~(1u << curl);
      const int l1 = pick_letter(m1, C.acgu != 0, C, rng);
      const unsigned m2 = allowed[partner] & pair_mask(l1);
      mut[pos] = code_letter(l1);
      if (m2) mut[partner] = code_letter(pick_letter(m2, C.acgu != 0, C, rng));
    }
    D.rng[g] = rng;
    // homodimer designs keep the two strands identical (sequence_utils.py:1102-1128)
    const int A = D.len_a[job];
    if (C.oligo == 2 && A > 0 && n == 2 * A) {
      if (D.same_halves[job]) {   // identical target halves: the strand that changed is copied over the other
        bool da = false, db = false;
        for (int k = 0; k < A; k++) { da |= mut[k] != cur[k]; db |= mut[A + k] != cur[A + k]; }
        if (da) { for (int k = 0; k < A; k++) mut[A + k] = mut[k]; }
        else if (db) { for (int k = 0; k < A; k++) mut[k] = mut[A + k]; }
      } else if (partner >= 0) {  // different halves: the two letters of an inter-strand pair are mirrored onto the other strand
        const int lo = min(pos, partner), hi = max(pos, partner);
        if (lo < A && hi >= A) {
          const int in_a = lo, in_b = hi - A;
          const char ca = mut[A + in_b], cb = mut[in_a];
          mut[in_b] = ca;
          mut[A + in_a] = cb;
        } else if (hi < A) {   // both letters inside strand A: mirrored onto strand B (deliberate; see the host mirror's propose_mutation)
          mut[A + lo] = mut[lo];
          mut[A + hi] = mut[hi];
        } else {
          mut[lo - A] = mut[lo];
          mut[hi - A] = mut[hi];
        }
      }
    }
  }
  self_dimer_row(D, C, row, mut, n, lane);
}

// ------------------------------------------------------------------------------------------------ accept
// score record of the mutant (energy_scores.py:31-125 with the float32 conventions of the ViennaRNA API, sim_score.py:62-147)
// and the Metropolis test (replica_exchange_monte_carlo.py:26-77)
__global__ void __launch_bounds__(kWPB * 32) bf_k_design_accept(BfDesignDev D, BfDesignCfg C, int B, int init, int gstep) {
  extern __shared__ __align__(16) unsigned char dyn[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, row = blockIdx.x * kWPB + warp;
  if (row >= B) return;
  const int g = D.rowmap[row], job = g / D.R, n = D.len[job], S = D.stride;
  const short *tpt = D.tpt + (size_t)job * S;
  const char *nss = D.o_ss + (size_t)row * (S + 1);
  WarpScratch w = scratch(dyn, S, warp);
  if (lane == 0) pair_table(nss, n, w.pt, w.stk);
  __syncwarp();
  // per-position confusion matrix (sim_score.py:104-119)
  int tp = 0, fp = 0, fn = 0, tn = 0;
  for (int i = lane; i < n; i += 32) {
    const int r = tpt[i], q = w.pt[i];
    if (r == q) { if (r != -1) tp++; else tn++; }
    else if (r == -1) fp++;
    else fn++;
  }
  for (int o = 16; o > 0; o >>= 1) {
    tp += __shfl_xor_sync(BF_FULL, tp, o); fp += __shfl_xor_sync(BF_FULL, fp, o);
    fn += __shfl_xor_sync(BF_FULL, fn, o); tn += __shfl_xor_sync(BF_FULL, tn, o);
  }
  const bool two = D.len_a[job] > 0;
  if (two) tp += 2;   // '&' becomes the always-matching pair "Ee" for the similarity scores (energy_scores.py:79)
  // -motifs: does the motif occur in the mutant (lanes over the start positions; a window may not span the '&' of two strands)
  unsigned motif_hit = 0;
  if (C.n_motifs > 0) {
    const char *mut = D.mut_seq + (size_t)row * S;
    const int la = D.len_a[job];
    for (int m = 0; m < C.n_motifs; m++) {
      const int ml = C.motif_len[m];
      bool found = false;
      for (int p0 = 0; p0 + ml <= n && !found; p0 += 32) {
        const int p = p0 + lane;
        bool hit = p + ml <= n && !(la > 0 && p < la && p + ml > la);
        for (int k = 0; k < ml && hit; k++) hit = (C.motif_mask[m][k] >> letter_code(mut[p + k])) & 1;
        found = __any_sync(BF_FULL, hit);
      }
      if (found) motif_hit |= 1u << m;
    }
  }
  int ok = 0;
  double rec[kDesignRec];
  if (lane == 0) {
    double num, den;
    if (tp == 0 && fp == 0 && fn == 0 && tn != 0) { num = 1.0; den = 1.0; }
    else {
      num = (double)tp * tn - (double)fp * fn;
      den = sqrt((double)(tp + fp) * (double)(tp + fn) * (double)(tn + fn) * (double)(tn + fp));
    }
    const double mcc = rint(num / (den + 0.00001) * 1000.0) / 1000.0;
    const double recall = rint((double)tp / ((double)(tp + fn) + 0.001) * 1000.0) / 1000.0;
    const double precision = rint((double)tp / ((double)(tp + fp) + 0.001) * 1000.0) / 1000.0;
    const double Ed = (double)(float)((double)D.o_eval[(size_t)row * D.T] / 100.0);
    const double Epf = (double)(float)D.o_pf[(size_t)row * 5 + (two ? 3 : 4)];   // two strands: FAB (energy_scores.py:157)
    const double MFE = (double)(float)((double)D.o_mfe[row] / 100.0);
    rec[kRecEd] = Ed; rec[kRecEpf] = Epf; rec[kRecMcc] = 1.0 - mcc; rec[kRecPrecision] = 1.0 - precision; rec[kRecRecall] = 1.0 - recall;
    rec[kRecMFE] = MFE; rec[kRecEdef] = D.o_defect ? D.o_defect[row] : 0.0; rec[kRecDist] = (double)(fp + fn); rec[kRecStep] = (double)gstep;
    rec[kRecOligoFraction] = 0.0; rec[kRecOligoBonus] = 0.0; rec[kRecEd2] = 0.0; rec[kRecMotif] = 0.0; rec[kRecSubopt] = 0.0;
    double total = 0.0;
    for (int k = 0; k < C.n_terms; k++) {
      const double wgt = C.weight[k];
      switch (C.term[k]) {
        case kTermEdEpf: total += (Ed - Epf) * wgt; break;
        case kTermMcc: total += rec[kRecMcc] * 10 * wgt; break;
        case kTermSlnEpf: total += (Epf + 0.3759 * (n + (two ? 1 : 0)) + 5.7534) / 10 * wgt; break;   // len(sequence) counts the '&'
        case kTermEdMfe: total += (Ed - MFE) * wgt; break;
        case kTermPrecision: total += rec[kRecPrecision] * 10 * wgt; break;
        case kTermRecall: total += rec[kRecRecall] * 10 * wgt; break;
        case kTermEdef: total += rec[kRecEdef] * wgt; break;
      }
    }
    if (D.n_alt && D.n_alt[job] > 0) {   // alternative structures: mean of their (float32) energies minus Epf (energy_scores.py:98-102)
      double sum = 0.0;
      for (int k = 0; k < D.n_alt[job]; k++) sum += (double)(float)((double)D.o_eval[(size_t)row * D.T + 1 + k] / 100.0);
      rec[kRecEd2] = sum / D.n_alt[job];
      total += rec[kRecEd2] - Epf;
    }
    // -nd on: the mutant folds into the target (1 - mcc == 0, as the reference tests it: a fully paired duplex that folds into its
    // target has mcc 0); second-best structure within 49 kcal/mol, else 0
    if (C.subopt && D.nd_flag && D.nd_flag[row] && rec[kRecMcc] == 0.0) {
      const int e1 = D.o_e1[row], e2 = D.o_e2[row];
      rec[kRecSubopt] = (e2 < BF_INF && e2 - e1 <= 4900) ? (double)(float)((double)e2 / 100.0) : 0.0;
      total -= rec[kRecSubopt] - Epf;
    }
    const bool avoid = C.oligo == 3;   // one-strand jobs only: the fraction is the self-dimer's (energy_scores.py:118-119,412-419)
    if ((two && C.oligo >= 1) || avoid) {
      // equilibrium dimer fraction at 1 mM from FcAB - FA - FB (dimer_multichain_energy.py:36-63), float32 API values first.
      // FcAB = 999 (no inter-strand pair) gives rhs = 0 and a NaN fraction, as the host arithmetic does.
      const double *pf = (avoid ? D.o_dimer_pf : D.o_pf) + (size_t)row * 5;
      const double kT = 0.001987204259 * (273.15 + 37);
      const double dF = (double)(float)pf[2] - (double)(float)pf[0] - (double)(float)pf[1];
      const double rhs = 1e-3 / 55.14 * exp(-dF / kT);
      const double frac = 1 - (sqrt(1 + 4 * rhs) - 1) / (2 * rhs);
      rec[kRecOligoFraction] = frac;
      rec[kRecOligoBonus] = (avoid || (C.oligo == 2 && D.same_halves[job])) ? -kT * log(1 - frac) : -kT * log(frac);
      total += rec[kRecOligoBonus];
    }
    for (int m = 0; m < C.n_motifs; m++)
      if (motif_hit >> m & 1u) rec[kRecMotif] += C.motif_bonus[m];
    total += rec[kRecMotif];   // (after the oligomer terms, as in score_sequence)
    rec[kRecScore] = total;
    if (init) ok = 1;
    else {
      const double old = D.rec[(size_t)g * kDesignRec + kRecScore];
      unsigned int *cn = D.counts + (size_t)g * 3;
      if (total <= old) { ok = 1; cn[0]++; cn[1]++; }
      else {
        unsigned long long rng = D.rng[g];
        const double T = D.temps[D.shelf[g]];
        ok = exp((-C.metropolis_L / T) * (total - old)) > u01(rng);
        D.rng[g] = rng;
        if (ok) cn[0]++; else cn[2]++;
      }
    }
    if (ok) {
      for (int k = 0; k < kDesignRec; k++) D.rec[(size_t)g * kDesignRec + k] = rec[k];
      D.cur_mfe[g] = D.o_mfe[row];
    }
  }
  ok = __shfl_sync(BF_FULL, ok, 0);
  if (ok) {
    const char *mut = D.mut_seq + (size_t)row * S;
    char *cs = D.cur_seq + (size_t)g * S, *css = D.cur_ss + (size_t)g * (S + 1);
    for (int k = lane; k < S; k += 32) cs[k] = mut[k];
    for (int k = lane; k <= S; k += 32) css[k] = nss[k];
  }
}

// ------------------------------------------------------------------------------------------------ exchange
// End of a global step: record the best state of every job, then the neighbour swaps in temperature order
// (replica_exchange_monte_carlo.py:113-173: pairs (1,2),(3,4).. on even global steps, (0,1),(2,3).. on odd ones).
__global__ void bf_k_design_exchange(BfDesignDev D, BfDesignCfg C, const uint8_t *active, int gstep) {
  const int job = blockIdx.x * blockDim.x + threadIdx.x;
  if (job >= D.J || (active && !active[job])) return;
  const int R = D.R, S = D.stride;
  double *best = D.best_rec + (size_t)job * kDesignRec;
  int pick = -1;
  unsigned solved = 0;
  for (int r = 0; r < R; r++) {
    const double *rec = D.rec + (size_t)(job * R + r) * kDesignRec;
    if (rec[kRecDist] == 0.0) solved++;
    const double bm = pick < 0 ? best[kRecDist] : D.rec[(size_t)(job * R + pick) * kDesignRec + kRecDist];
    const double bs = pick < 0 ? best[kRecScore] : D.rec[(size_t)(job * R + pick) * kDesignRec + kRecScore];
    if (rec[kRecDist] < bm || (rec[kRecDist] == bm && rec[kRecScore] < bs)) pick = r;
  }
  if (pick >= 0) {
    const size_t g = (size_t)job * R + pick;
    for (int k = 0; k < kDesignRec; k++) best[k] = D.rec[g * kDesignRec + k];
    best[kRecStep] = (double)gstep;
    for (int k = 0; k < S; k++) D.best_seq[(size_t)job * S + k] = D.cur_seq[g * S + k];
    for (int k = 0; k <= S; k++) D.best_ss[(size_t)job * (S + 1) + k] = D.cur_ss[g * (S + 1) + k];
  }
  if (solved) {
    D.n_solved[job] += solved;
    if (D.solved_step[job] < 0) D.solved_step[job] = gstep;
  }
  // neighbour swaps: replicas of a job hold a permutation of the shelves
  if (gstep <= 0) return;   // initial scoring: nothing to exchange yet
  unsigned long long rng = D.job_rng[job];
  for (int a = (gstep % 2 == 0) ? 1 : 0; a + 1 < R; a += 2) {
    int ra = -1, rb = -1;
    for (int r = 0; r < R; r++) {
      const int sh = D.shelf[job * R + r];
      if (sh == a) ra = r;
      if (sh == a + 1) rb = r;
    }
    if (ra < 0 || rb < 0) continue;
    const double e0 = D.rec[(size_t)(job * R + ra) * kDesignRec + kRecScore], e1 = D.rec[(size_t)(job * R + rb) * kDesignRec + kRecScore];
    bool ok = e1 <= e0;
    unsigned int *rc = D.re_counts + (size_t)job * 3;
    if (ok) rc[1]++;
    else {
      const double T0 = D.temps[a], T1 = D.temps[a + 1];
      ok = exp(C.metropolis_L * (1.0 / T0 - 1.0 / T1) * (e0 - e1)) > u01(rng);
    }
    if (ok) { D.shelf[job * R + ra] = a + 1; D.shelf[job * R + rb] = a; rc[0]++; }
    else rc[2]++;
  }
  D.job_rng[job] = rng;
}

}  // namespace

cudaError_t bf_launch_design_nd_flag(const BfDesignDev &D, int B, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  bf_k_design_nd_flag<<<(B + kWPB - 1) / kWPB, kWPB * 32, scratch_bytes(D.stride), st>>>(D, B);
  return cudaGetLastError();
}
cudaError_t bf_launch_design_pk_mask(const BfDesignDev &D, int B, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  bf_k_design_pk_mask<<<(B + kWPB - 1) / kWPB, kWPB * 32, 0, st>>>(D, B);
  return cudaGetLastError();
}
cudaError_t bf_launch_design_pk_paint(const BfDesignDev &D, int B, int round, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  bf_k_design_pk_paint<<<(B + kWPB - 1) / kWPB, kWPB * 32, 0, st>>>(D, B, round);
  return cudaGetLastError();
}
cudaError_t bf_launch_design_gather(const BfDesignDev &D, int B, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  bf_k_design_gather<<<(B + kWPB - 1) / kWPB, kWPB * 32, 0, st>>>(D, B);
  return cudaGetLastError();
}
cudaError_t bf_launch_design_propose(const BfDesignDev &D, const BfDesignCfg &C, int B, bool copy_only, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  bf_k_design_propose<<<(B + kWPB - 1) / kWPB, kWPB * 32, scratch_bytes(D.stride), st>>>(D, C, B, copy_only ? 1 : 0);
  return cudaGetLastError();
}
cudaError_t bf_launch_design_accept(const BfDesignDev &D, const BfDesignCfg &C, int B, bool init, int gstep, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  bf_k_design_accept<<<(B + kWPB - 1) / kWPB, kWPB * 32, scratch_bytes(D.stride), st>>>(D, C, B, init ? 1 : 0, gstep);
  return cudaGetLastError();
}
cudaError_t bf_launch_design_exchange(const BfDesignDev &D, const BfDesignCfg &C, const uint8_t *active, int gstep, cudaStream_t st) {
  if (D.J <= 0) return cudaSuccess;
  bf_k_design_exchange<<<(D.J + 63) / 64, 64, 0, st>>>(D, C, active, gstep);
  return cudaGetLastError();
}
