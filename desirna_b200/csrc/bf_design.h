// bf_design.h -- device side of the Replica-Exchange Monte-Carlo design loop (bf_design.cu).
//
// The reference runs this loop on the host: utils/replica_exchange_monte_carlo.py:176-271 (Metropolis sub-steps and
// neighbour swaps) around utils/sequence_utils.py:926-1136 (move generator).  Here the state of every replica of every
// design problem ("job") stays in HBM; one sub-step is  propose -> MFE fill + backtrack -> PF fill + exterior -> eval ->
// accept  on one stream, with no host round trip.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

constexpr int kDesignRec = 15;   // doubles per replica record
// record slots (names of the reference's ScoreSeq fields, utils/energy_scores.py:176-195)
enum { kRecScore = 0, kRecEd = 1, kRecEpf = 2, kRecMcc = 3, kRecPrecision = 4, kRecRecall = 5, kRecMFE = 6, kRecEdef = 7, kRecDist = 8, kRecStep = 9, kRecOligoFraction = 10, kRecOligoBonus = 11, kRecEd2 = 12, kRecMotif = 13, kRecSubopt = 14 };
// scoring terms (-sf), in the order of ScoreSeq.get_scoring_function (utils/energy_scores.py:376-398)
enum { kTermEdEpf = 0, kTermMcc = 1, kTermSlnEpf = 2, kTermEdMfe = 3, kTermPrecision = 4, kTermRecall = 5, kTermEdef = 6 };

struct BfDesignCfg {
  int n_terms;
  int term[8];
  double weight[8];
  double metropolis_L;   // sim_options.L
  int point_mutations;   // -tm on/off
  int acgu;              // -acgu on: paired letters drawn with nt_weight
  double nt_weight[4];   // A C G U
  int oligo;             // two-strand jobs: 1 heterodimer, adds -kT ln(dimer fraction); 2 homodimer, strands kept identical and
                         // -kT ln(dimer fraction) (different target halves) or -kT ln(1 - fraction) (identical halves)
                         // (energy_scores.py:120-125,421-441, dimer_multichain_energy.py:36-76, sequence_utils.py:1102-1128)
  int subopt;            // -nd on: Epf - E(second-best structure) for mutants that fold into the target (energy_scores.py:104-107)
  int n_motifs;          // -motifs: IUPAC motifs, bonus added when the motif occurs in the sequence (sequence_utils.py:1231-1256)
  int motif_len[8];
  double motif_bonus[8];
  unsigned char motif_mask[8][32];
};

struct BfDesignDev {
  int J, R, stride;
  // per job
  const char *tgt;               // J x stride   target dot-bracket
  const short *tpt;              // J x stride   partner in the target (0-based) or -1
  const uint8_t *allowed;        // J x stride   letters_allowed, bit 0..3 = A C G U  (sequence_utils.py:454-525)
  const int *len;                // J            nucleotides (both strands, no '&')
  const int *len_a;              // J            length of strand A, 0 = single strand ('&' sits after it in the reference's strings)
  const uint8_t *same_halves;    // J            1: the two halves of the target are the same string (homodimer designs)
  const short *mpt;              // J x stride   partner for the move generator (Nucleotide.pairs_with), or null = tpt
  const signed char *snake_id;   // J x stride   conflict graph of the position, -1 none; or null
  const char *snake_letter;      // J x stride x 4   letter of the position in each colouring of its graph (0 = absent)
  const char *alt;               // J x max_alt x stride   alternative structures (energy_scores.py:98-102), or null
  const int *n_alt;              // J
  int max_alt, T;                // T = 1 + max_alt targets per batch row
  const unsigned short *avail;   // J x stride   positions with more than one allowed letter (sequence_utils.py:1026-1029)
  const int *n_avail;            // J
  unsigned long long *job_rng;   // J            stream of the neighbour swaps
  char *best_seq, *best_ss;      // J x stride, J x (stride+1)
  double *best_rec;              // J x kDesignRec
  int *solved_step;              // J            first global step at whose end a replica folds into the target, -1 before
  unsigned int *n_solved;        // J            replica states (at global-step ends) that fold into the target
  unsigned int *re_counts;       // J x 3        neighbour swaps accepted, accepted because not worse, rejected (Stats, :671-792)
  // per replica g = job * R + r
  char *cur_seq, *cur_ss;        // G x stride, G x (stride+1)
  double *rec;                   // G x kDesignRec
  int *shelf;                    // G            index into temps
  int *cur_mfe;                  // G            MFE (dcal/mol) of the current sequence: scale of its mutant's partition function
  unsigned long long *rng;       // G
  unsigned int *counts;          // G x 3        accepted, accepted because not worse, rejected
  const double *temps;           // R            temperature shelves, ascending
  const double *tm_prob;         // R            probability of a targeted move per shelf (sequence_utils.py:963)
  // per batch row (active jobs only)
  const int *rowmap;             // B -> g
  char *mut_seq;                 // B x stride
  int *row_len;                  // B
  int *row_cut;                  // B            1-based first nucleotide of strand B, 0 = single strand (bf_batch_t.cut)
  int *row_scale;                // B            cur_mfe of the row's replica (written by bf_k_design_propose)
  char *row_tgt;                 // B x T x stride   target, then the alternative structures (rows beyond n_alt repeat the target)
  int *o_mfe;                    // B
  char *o_ss;                    // B x (stride+1)
  double *o_pf;                  // B x 5
  int *o_eval;                   // B x T
  double *o_defect;              // B (only with the Edef term)
  // pseudoknot overlay (sequence_utils.py:1166-1228): constrained refolds of the rows
  uint8_t *pk_nopair;            // B x stride      positions already paired
  int *o_mfe2;                   // B
  char *o_ss2;                   // B x (stride+1)  structure of the constrained refold
  // negative design: rows whose structure equals the target, and their (best, second-best) energies from bf_k_mfe2
  uint8_t *nd_flag;              // B
  int *o_e1, *o_e2;              // B
};

cudaError_t bf_launch_design_gather(const BfDesignDev &D, int B, cudaStream_t st);
cudaError_t bf_launch_design_nd_flag(const BfDesignDev &D, int B, cudaStream_t st);                 // nd_flag: does o_ss equal the target
cudaError_t bf_launch_design_pk_mask(const BfDesignDev &D, int B, cudaStream_t st);                 // pk_nopair from the overlay so far (o_ss)
cudaError_t bf_launch_design_pk_paint(const BfDesignDev &D, int B, int round, cudaStream_t st);     // pairs of o_ss2 into o_ss as [] <> {}
cudaError_t bf_launch_design_propose(const BfDesignDev &D, const BfDesignCfg &C, int B, bool copy_only, cudaStream_t st);
cudaError_t bf_launch_design_accept(const BfDesignDev &D, const BfDesignCfg &C, int B, bool init, int gstep, cudaStream_t st);
cudaError_t bf_launch_design_exchange(const BfDesignDev &D, const BfDesignCfg &C, const uint8_t *active, int gstep, cudaStream_t st);
