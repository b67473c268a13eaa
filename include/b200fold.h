/*
 * b200fold.h -- C-ABI of the B200-native batched RNA folding engine.
 *
 * DesiRNA has no FFI of its own: its hot path enters native code through ViennaRNA's
 * SWIG module `RNA`.  Each entry point below names the reference call site it replaces
 * (paths relative to the DesiRNA tree).  All functions return 0 on success, a BF_ERR_*
 * code otherwise; bf_last_error() gives the message.  No allocation crosses the boundary:
 * every buffer is caller-owned, strings are fixed-stride char arrays.
 *
 * Threading: one engine per process (one process per GPU, as in the reference's one
 * worker per replica: utils/replica_exchange_monte_carlo.py:248).  Calls are serialised
 * by the caller.
 */
#ifndef B200FOLD_H
#define B200FOLD_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

enum {
  BF_OK = 0,
  BF_ERR_CUDA = 1,         /* CUDA runtime failure (no GPU, launch error, out of memory) */
  BF_ERR_NOT_INIT = 2,     /* bf_init not called / no parameters loaded */
  BF_ERR_PARAMS = 3,       /* parameter file missing or malformed */
  BF_ERR_UNAVAILABLE = 4,  /* e.g. Turner 2004 tables are not packaged */
  BF_ERR_ARG = 5           /* bad argument (null buffer, length > stride, ...) */
};

/* what to compute for every sequence of a batch */
enum {
  BF_WANT_MFE = 1u,    /* Zuker MFE energy                        fc.mfe()[1], RNA.fold()[1]   energy_scores.py:354 */
  BF_WANT_SS = 2u,     /* + backtracked MFE structure             fc.mfe()[0], fc.mfe_dimer()[0] energy_scores.py:151,156 */
  BF_WANT_PF = 4u,     /* McCaskill inside: ensemble free energy  fc.pf()[1], fc.pf_dimer()     energy_scores.py:150,157 */
  BF_WANT_EVAL = 8u,   /* energy of the given target structures   fc.eval_structure()          energy_scores.py:75,99 */
  BF_WANT_BPP = 16u,   /* base-pair probabilities (outside pass)  md.compute_bpp=1 + fc.pf()    energy_scores.py:369-373 */
  BF_WANT_DEFECT = 32u /* ensemble defect of target 0             fc.ensemble_defect()          energy_scores.py:374 */
};

typedef struct {
  int32_t B;             /* sequences in the batch */
  int32_t stride;        /* bytes between consecutive rows of seq / nopair / each target; >= max length */
  const char *seq;       /* B x stride, ASCII ACGU (T accepted), '&' removed by the caller */
  const int32_t *len;    /* B lengths */
  const int32_t *cut;    /* B or NULL: 1-based index of the first nucleotide of strand B, 0 = one strand
                            (RNA.fold_compound("A&B"): energy_scores.py:147, dimer_multichain_energy.py:89,104) */
  const uint8_t *nopair; /* B x stride or NULL: 1 = position may not pair -- fc.hc_add_from_db with 'x'
                            (sequence_utils.py:1181,1198,1214).  Applies to the MFE only. */
  const char *targets;   /* B x n_targets x stride dot-bracket strings or NULL; only '(' ')' pair */
  int32_t n_targets;
  uint32_t want;         /* OR of BF_WANT_* */
} bf_batch_t;

typedef struct {
  int32_t *mfe_dcal;  /* B: MFE in dcal/mol (ViennaRNA returns kcal/mol as C float = value/100) */
  char *mfe_ss;       /* B x (stride+1): NUL-terminated dot-bracket, no '&' (as fc.mfe_dimer) */
  double *pf;         /* B x 5: FA, FB, FcAB, FAB, F0AB in kcal/mol; one strand: [4] = ensemble free energy */
  int32_t *eval_dcal; /* B x n_targets: energy of each target in dcal/mol (>= 10000000: malformed / forbidden loop) */
  double *defect;     /* B: ensemble defect of target 0 */
  double *bpp;        /* B x stride x stride (row i-1, col j-1, i<j) or NULL */
} bf_result_t;

/* engine life cycle */
int bf_init(int device);
int bf_shutdown(void);
const char *bf_last_error(void);

/* RNA.params_load(path)                                                    DesiRNA.py:455-456 */
int bf_params_load(const char *par_path);
/* `-p 2004` keeps ViennaRNA's compiled-in defaults; `-p 1999` loads the vendored file (DesiRNA.py:455).
 * year 1999 -> table set at `builtin_dir`/turner1999_37C.par; 2004 -> BF_ERR_UNAVAILABLE (not packaged). */
int bf_params_builtin(int year, const char *builtin_dir);
/* read back one integer parameter (loader cross-checks): name as in bf_params.h, up to 6 indices */
int bf_params_get(const char *name, int i0, int i1, int i2, int i3, int i4, int i5, int32_t *out);

/* Score a batch whose buffers live in HOST memory: copies in, runs the kernels, copies out, synchronises.
 * This is the call behind score_sequence()/get_mfe_e_ss() (energy_scores.py:31-159). */
int bf_score_batch(const bf_batch_t *batch, bf_result_t *result);

/* Same, but every pointer in batch/result is a DEVICE pointer; work is enqueued on `cuda_stream`
 * (a cudaStream_t handle; NULL = the legacy default stream, as in the CUDA runtime) and NOT synchronised. */
int bf_score_batch_device(const bf_batch_t *batch, bf_result_t *result, void *cuda_stream);

/* fc.subopt_cb(delta, cb, data) with RNA.cvar.uniq_ML = 1                     energy_scores.py:465-474, sequence_utils.py:783
 * Every secondary structure of ONE single-strand sequence whose energy is within delta_dcal of the MFE, each exactly once,
 * sorted by energy.  The O(N^3) tables come from the GPU MFE fill; the output-sensitive walk over them runs on the host.
 * ss_out: max_out x (len+1) chars, e_out: max_out energies in dcal/mol, *n_out: structures written (<= max_out),
 * *truncated: 1 if the band holds more than max_out structures.  nopair: optional len bytes (hard constraint 'x'). */
/* Energies (dcal/mol) of the best and of the second-best secondary structure of every sequence of the batch (seq, len, cut,
 * nopair, stride as in bf_score_batch), by one DP over (best, second best) pairs on the unambiguous grammar -- what
 * get_first_suboptimal_structure_and_energy(seq, fc, 1)[1] reads off fc.subopt_cb's enumeration (utils/energy_scores.py:453-488,
 * RNA.cvar.uniq_ML = 1).  e2 >= 10000000: there is no second structure.  Two structures of equal energy count twice (e2 == e1).
 * Rows with cut > 0 are two strands under the loop model of bf_score_batch's two-strand MFE and eval: unconnected structures
 * count, a connected one pays DuplexInit once; e1 equals that MFE. */
int bf_second_best(const bf_batch_t *batch, int32_t *e1_dcal, int32_t *e2_dcal);
int bf_subopt(const char *seq, int32_t len, const uint8_t *nopair, int32_t delta_dcal, int32_t max_out, char *ss_out, int32_t *e_out,
              int32_t *n_out, int32_t *truncated);

/* device time (ms, CUDA events on the launch stream) of the mfe, pf and eval kernels of the most recent
 * bf_score_batch[_device] call; -1 for a kernel that did not run.  Blocks until those kernels finished. */
int bf_last_kernel_ms(double out[3]);
/* micro-benchmarks for the roofline denominators: out[0] INT32 add+min op/s, out[1] FP64 flop/s (DFMA),
 * out[2] shared-memory load bytes/s, whole chip */
int bf_microbench(double out[3]);

/* number of kernels launched by this process since bf_init (bench.py "gpu_launches") */
int64_t bf_kernel_launches(void);
/* SM count of the device in use */
int bf_sm_count(void);
/* Test / measurement hook.  Kernel variants are chosen per call by default rules that a few BF_* environment variables override;
 * this sets the variable BF_<KEY> from the host program (value < 0: remove it, back to the default rule).  The keys:
 *   "cl" 0 / 1: never / always use the cluster-per-sequence fill kernels where they cover the length; "cl_c" 4 | 8 | 16: their
 *   cluster size; "cl_bw" 16 | 32: their block width;
 *   "ext_wide" 0 / 1: exterior recursions by one warp / one CTA per sequence;
 *   "wide" 0: no 16-warp variants for small batches;
 *   "fill3" 0: the round-1 fill kernels instead of the third-generation ones; "fill3_small" 0: small batches on the 16-warp round-1
 *   kernels instead of the 16-warp third-generation ones;
 *   "blk_min" / "blk_min_pf" N: the round-1 MFE / PF fills use the blocked split from N nt on (default 280 / 250);
 *   "force_generic" 1: single strands on the generic kernels too (read by bf_init);
 *   "design_overlap" 0: the device design loop always folds MFE, then PF.
 * Any other key is refused with BF_ERR_ARG. */
int bf_set_option(const char *key, int value);
/* Test hook: copy one engine-internal DP table of the most recent call to host memory.
 * which: 0 = c (int32), 1 = fML (int32), 2 = qb (double); layout: per sequence a packed, diagonal-major triangle of
 * *slot_entries entries (entry (i,j), d=j-i>=4, at (d-4)*n - (d*(d-1)/2-6) + i-1).  host may be NULL to query the size. */
int bf_debug_copy_table(int which, int32_t n_seq, void *host, size_t host_bytes, size_t *slot_entries);


/* ---------------------------------------------------------------------------------------------------------
 * Device-resident Replica-Exchange Monte-Carlo design loop: many design problems ("jobs") x replicas advance
 * in lock step with sequences, scores, temperature shelves and random streams resident in HBM.  Replaces,
 * for targets made of . ( ), one strand (with or without avoiding self-dimers) or two (heterodimer, homodimer):
 *   remc.mutate_sequence_re / single_replica_design / mc_delta      utils/replica_exchange_monte_carlo.py:26-110,176-271
 *   remc.replica_exchange / replica_exchange_attempt                utils/replica_exchange_monte_carlo.py:80-173
 *   seq_utils.mutate_sequence / get_mutation_position / expand_cases  utils/sequence_utils.py:926-1136
 *   es.score_sequence arithmetic (Ed-Epf, 1-MCC, sln_Epf, Ed-MFE, 1-precision, 1-recall, Edef)  utils/energy_scores.py:31-125,376-398
 * The random generator is per-replica splitmix64, not Python's: trajectories match in distribution only.
 * All jobs of one loop share `stride`; callers bucket jobs of similar length into one loop each. */
typedef struct {
  int32_t n_jobs, replicas, stride;
  const char *target;      /* n_jobs x stride dot-bracket, only . ( )                          input_file.sec_struct */
  const int32_t *len;      /* n_jobs: nucleotides (both strands) */
  const int32_t *len_a;    /* n_jobs or NULL: length of strand A of a two-strand job (the reference's 'A&B' strings), 0 = one strand */
  const uint8_t *allowed;  /* n_jobs x stride: Nucleotide.letters_allowed as bits A=1 C=2 G=4 U=8  sequence_utils.py:454-525 */
  const char *init_seq;    /* n_jobs x replicas x stride start sequences                         sequence_utils.py:862-888 */
  const double *temps;     /* replicas: temperature shelves, ascending                           sequence_utils.py:811-859 */
  const double *tm_prob;   /* replicas: probability of a targeted move on each shelf             sequence_utils.py:963 */
  int32_t n_terms;         /* scoring function terms in -sf order */
  int32_t term[8];         /* 0 Ed-Epf, 1 1-MCC, 2 sln_Epf, 3 Ed-MFE, 4 1-precision, 5 1-recall, 6 Edef */
  double weight[8];
  double metropolis_L;     /* sim_options.L (DesiRNA.py:568) */
  int32_t point_mutations; /* -tm on: targeted mutations */
  int32_t re_attempt;      /* Monte-Carlo sub-steps per global step (-e) */
  int32_t acgu;            /* -acgu on: paired letters drawn with nt_weight */
  double nt_weight[4];     /* A C G U */
  int32_t oligo;           /* two-strand jobs: 1 heterodimer (-kT ln(dimer fraction)), 2 homodimer (strands kept identical;
                              -kT ln(fraction) or, for identical target halves, -kT ln(1 - fraction))   energy_scores.py:120-125,421-441;
                              one-strand jobs: 3 avoid (-o on): every mutant's self-dimer seq&seq is folded too (partition function
                              only, default scale) and -kT ln(1 - fraction) of that dimer is added; BF_ERR_ARG with a two-strand job
                                                                                                energy_scores.py:118-119,412-419 */
  uint64_t seed;
  /* optional scenario terms (all zero = absent) */
  const char *alt_targets;   /* n_jobs x max_alt x stride: alternative structures (input_file.alt_sec_structs), only . ( );
                                adds mean(eval(alt)) - Epf to the scoring function                    energy_scores.py:98-102 */
  const int32_t *n_alt;      /* n_jobs: alternative structures of each job, 0..max_alt */
  int32_t max_alt;
  int32_t n_motifs;          /* -motifs: up to 8 IUPAC motifs of up to 32 letters, bonus added when the motif occurs   sequence_utils.py:1231-1256 */
  const uint8_t *motif_mask; /* n_motifs x 32: letters allowed at each motif position (A=1 C=2 G=4 U=8), 0 beyond its length */
  const int32_t *motif_len;  /* n_motifs */
  const double *motif_bonus; /* n_motifs */
  int32_t pks;               /* 1: pseudoknot overlay (targets may use the bracket families () [] <> {}): after the MFE fold the
                                paired positions are forbidden, the sequence is folded again and the new pairs painted with the next
                                family, up to three rounds                                  sequence_utils.py:1166-1228 */
  const int16_t *move_partner; /* n_jobs x stride or NULL: partner of each position FOR THE MOVE GENERATOR (Nucleotide.pairs_with,
                                sequence_utils.py:486-505), -1 = none; NULL = the target's partner.  Differs from the target's with
                                alternative structures: their clash-free pairs are pair restraints too */
  const int8_t *snake_id;    /* n_jobs x stride or NULL: index of the conflict graph ("snake") a position belongs to, -1 = none
                                sequence_utils.py:119-396 */
  const char *snake_letter;  /* n_jobs x stride x 4: letter of the position in each colouring of its graph, 0 = colouring absent;
                                a move on a graph node sets every node of the graph to another colouring   :1085-1094 */
  int32_t subopt;            /* 1: negative design (-nd on): a mutant that folds into its target also pays Epf - E(second-best
                                structure), the latter from bf_second_best's DP (two-strand jobs too; not with pks)
                                                                                                energy_scores.py:104-107,453-488 */
} bf_design_t;

enum { BF_DESIGN_REC = 15 }; /* doubles per record: scoring_function, edesired, Epf, 1-mcc, 1-precision, 1-recall, MFE,
                                ensemble_defect, positions whose partner differs from the target's (0 = solved), global step,
                                oligo_fraction, oligomer_bonus (avoid designs: the monomer bonus), edesired2 (mean energy of the
                                alternative structures), motif bonus, subopt_e */

/* Allocates the loop on the engine's GPU, scores the start sequences (global step 0). */
int bf_design_create(const bf_design_t *cfg, void **handle);
/* Enqueue `global_steps` global steps (each: re_attempt sub-steps of propose/fold/accept, then neighbour swaps) on the
 * loop's own stream and return without waiting; loops of different handles overlap on the GPU. */
int bf_design_run(void *handle, int32_t global_steps);
int bf_design_sync(void *handle);
/* *busy = 1 while enqueued steps are still running (does not wait): lets a host advance many loops at their own pace. */
int bf_design_busy(void *handle, int32_t *busy);
/* active[j] = 0 drops job j from the following steps (-sws on: stop when solved); waits for enqueued steps first. */
int bf_design_set_active(void *handle, const uint8_t *active);
/* Best state per job seen at global-step ends (fewest mismatching positions, then lowest scoring function):
 * best_seq n_jobs x stride, best_ss n_jobs x (stride+1), best_rec n_jobs x BF_DESIGN_REC, solved_step (first global step
 * that ended with a replica folding into the target, -1 = none), n_solved (such replica states so far).  NULL = skip. */
int bf_design_read_jobs(void *handle, char *best_seq, char *best_ss, double *best_rec, int32_t *solved_step, uint32_t *n_solved);
/* Current state of every replica (job-major): seq G x stride, ss G x (stride+1), rec G x BF_DESIGN_REC, shelf G,
 * counts G x 3 (accepted, accepted because not worse, rejected).  NULL = skip. */
int bf_design_read_replicas(void *handle, char *seq, char *ss, double *rec, int32_t *shelf, uint32_t *counts);
/* Neighbour-swap counters per job, n_jobs x 3: accepted, accepted because not worse, rejected (stats_inputs_outputs.py:740-756). */
int bf_design_read_swaps(void *handle, uint32_t *re_counts);
/* Test hook: run the move generator once for every active replica without scoring; mut_seq: rows x stride. */
int bf_design_propose_only(void *handle, char *mut_seq);
int bf_design_destroy(void *handle);

#ifdef __cplusplus
}
#endif
#endif
