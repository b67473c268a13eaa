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
/* fc.pbacktrack(num_samples) (vrna_pbacktrack, RNAsubopt -p): stochastic backtracking.  n_samples secondary structures of every
 * sequence of the batch (seq, len, stride as in bf_score_batch), each drawn independently from the Boltzmann ensemble of the
 * partition function bf_score_batch computes (the MFE sets its scale, as for BF_WANT_BPP).  HOST buffers, synchronous.
 * ss_out: B x n_samples x (stride+1) chars, sample-major within a row; sample k of row r at (r * n_samples + k) * (stride+1),
 * len[r] characters of . ( ) and a NUL (the rest of the slot is NUL too).  The samples are a function of (seed, r, k) alone: the
 * same call repeats, and the first k samples of a call with n > k are those of a call with k.
 * BF_ERR_UNAVAILABLE: a row with cut > 0, a nopair mask (the partition function ignores constraints), a stride outside the fill
 * path (> 2000) or BF_FORCE_GENERIC.  BF_ERR_ARG: n_samples < 1, null buffers, len > stride. */
int bf_sample(const bf_batch_t *batch, int32_t n_samples, uint64_t seed, char *ss_out);
/* E_pair: for every base pair (i,j) of every sequence of the batch (seq, len, nopair, stride as in bf_score_batch), the lowest
 * free energy of any secondary structure that contains it -- the MFE fill, then an outside pass in the minimum-free-energy
 * semiring over the fill's tables (RNAsubopt -z computes the same matrix).  Same energy model as BF_WANT_MFE: a nopair mask is
 * honoured as the MFE honours it.  HOST buffers, synchronous.
 * e_pair_out: B x stride x stride int32 in dcal/mol, entry [i-1][j-1] for i < j (the layout of bpp); 10000000 where (i,j)
 * cannot pair (not canonical, j - i <= 3, a masked position) or no structure contains it, on and below the diagonal and
 * beyond len.
 * BF_ERR_UNAVAILABLE: a row with cut > 0, a stride outside the fill path (> 2000) or BF_FORCE_GENERIC.
 * BF_ERR_ARG: null buffers, len > stride. */
int bf_pair_mfe(const bf_batch_t *batch, int32_t *e_pair_out);
/* fc.subopt_zuker() (vrna_subopt_zuker, RNAsubopt -z): Zuker suboptimals of ONE single-strand sequence.  The pairs with a finite
 * E_pair (bf_pair_mfe) are taken in order of (E_pair, i, j); for each pair no structure listed so far contains, one structure of
 * energy E_pair that contains it is appended (inside part traced back from the fill's c table, outside part from the outside
 * pass).  Every pair with a finite E_pair is therefore in some listed structure.  Output sorted by (energy, structure string);
 * ss_out: max_out x (len+1) chars, e_out: max_out energies in dcal/mol, *n_out: structures written, *truncated: 1 if pairs were
 * left uncovered after max_out structures.  nopair: optional len bytes (hard constraint 'x').
 * Which of several structures of equal energy is listed for a pair is a choice of the traceback; ViennaRNA may list another one
 * (no ViennaRNA output pins it).
 * BF_ERR_UNAVAILABLE: len outside the fill path (> 2000) or BF_FORCE_GENERIC.  BF_ERR_ARG: null buffers, len <= 0, max_out <= 0. */
int bf_subopt_zuker(const char *seq, int32_t len, const uint8_t *nopair, int32_t max_out, char *ss_out, int32_t *e_out, int32_t *n_out,
                    int32_t *truncated);

/* RNA.duplexfold(s1, s2) / RNAduplex: RNA-RNA hybridization, counting intermolecular pairs only (not called by DesiRNA).
 * For every requested (a, b) pair of strands, the lowest energy of a duplex structure: a chain of pairs a[k]-b[l], canonical,
 * k increasing and l decreasing, with at most 30 unpaired nucleotides between consecutive pairs, scored as bf_score_batch's
 * two-strand eval scores that structure on a&b (DuplexInit, the outer exterior stem, interior loops, the nick loop closed by the
 * innermost pair).  This is ViennaRNA's duplexfold recurrence as published; no ViennaRNA output pins it here.
 * Ties: the innermost pair is the first minimum in the order i (in a) ascending, then j (in b) descending; the backtrack from
 * (i,j) takes the first (k,l) that reproduces the energy, k = i-1 downwards, then l = j+1 upwards.
 * pairs: n_pairs x 2 (index into a, index into b), or NULL for the full grid a.n x b.n, a-major (n_pairs is then ignored).
 * e_dcal: one energy per pair in dcal/mol; 10000000 where no intermolecular pair is possible.
 * ss_out: NULL (energies only) or per pair a.stride + b.stride + 2 chars: a's len characters, '&', b's len characters, NUL
 * (the rest of the slot NUL too).  Pairs are '(' in a and ')' in b, full length, not trimmed; all dots where there is no pair.
 * HOST buffers, synchronous.  BF_ERR_ARG: null buffers, len < 0 or > stride, a strand longer than 2000 nt, a pair index out of
 * range, n_pairs < 0, a stride above 65536. */
typedef struct {
  int32_t n;           /* strands */
  int32_t stride;      /* bytes between consecutive rows of seq, >= every len, <= 65536 */
  const char *seq;     /* n x stride ASCII ACGU (T accepted) */
  const int32_t *len;  /* n lengths, 0 .. 2000 */
} bf_strands_t;
typedef struct {
  bf_strands_t a, b;
  int32_t n_pairs;
  const int32_t *pairs;
} bf_duplex_t;
int bf_duplex(const bf_duplex_t *q, int32_t *e_dcal, char *ss_out);

/* Accessibility-aware RNA-RNA interaction (RNAup / RNAplex -a / IntaRNA's site model; not called by DesiRNA).  HOST buffers,
 * synchronous.
 * A site of strands a and b is a duplex chain as in bf_duplex: pairs (k1,l1), ..., (km,lm) of a[k] with b[l], k increasing, l
 * decreasing, at most 30 unpaired nucleotides between consecutive pairs, with both spans km - k1 + 1 and l1 - lm + 1 at most
 * max_span (1 .. 64).  Its hybridization energy H (dcal/mol) is bf_duplex's energy of that chain: the engine's two-strand eval of
 * the structure on a&b (DuplexInit, the outer exterior stem, the interior loops, the nick loop closed by the innermost pair, with
 * neighbours only where they exist).  Its opening energies are
 *   ED_a = -(kT/1000) ln P_u^a(k1, km - k1 + 1),   ED_b = -(kT/1000) ln P_u^b(lm, l1 - lm + 1)     (kcal/mol)
 * with kT the loaded parameter set's, in cal/mol (the partition function's), and P_u from each side's accessibility mode:
 *   acc = -1: none, ED = 0;  acc = 0: global, bf_unpaired's ensemble of the whole strand;  acc = W > 0: bf_plfold's window average
 *   with span = W (W >= max_span).  Where P_u <= 0 the site does not exist.
 * Its score is E = (double)H / 100.0 + ED_a + ED_b, evaluated in that order in double.  For each requested pair of strands the
 * result is the site of least E; ties go to the first site in the order k1 ascending, l1 descending, km ascending, lm descending.
 * The structure is traced back inside the table of that start with bf_duplex's rule (the first (k,l) reproducing the cell, k = i-1
 * downwards, then l = j+1 upwards).  With no accessibility on either side and max_span >= both lengths, 100 E is bf_duplex's energy.
 * The accessibility of each side is computed once per call on the device (once for both when a and b are the same strand set and
 * mode); P_u and ED stay on the device.
 * Outputs per pair (pairs: n_pairs x 2 (index into a, index into b), or NULL for the full grid a.n x b.n, a-major):
 *   e:      E in kcal/mol, +inf where no site exists;
 *   h_dcal: NULL or H, 10000000 where no site exists;
 *   ed:     NULL or 2 doubles, ED_a and ED_b (0 where no site exists);
 *   site:   NULL or 4 ints, 1-based k1, km, lm, l1 (0 where no site exists);
 *   ss_out: NULL or a.stride + b.stride + 2 chars in bf_duplex's layout, all dots where no site exists.
 * This is not RNAup's partition-function interaction (RNAup -b): a single best site, no intramolecular structure inside it.
 * BF_ERR_ARG: null q or e, a bad strand set (as bf_duplex), max_span outside 1 .. 64, acc < -1, a window below max_span,
 * n_pairs < 0, a pair index out of range.  BF_ERR_UNAVAILABLE: global accessibility of a strand longer than the PF fill path covers,
 * a window longer than the fill path covers, accessibility under BF_FORCE_GENERIC. */
typedef struct {
  bf_strands_t a, b;       /* as bf_duplex; strands <= 2000 nt */
  int32_t n_pairs;         /* with pairs == NULL: the full a-major grid */
  const int32_t *pairs;
  int32_t max_span;        /* 1 .. 64 */
  int32_t acc_a, acc_b;    /* -1 none, 0 global, W > 0 RNAplfold window W (W >= max_span) */
} bf_interact_t;
int bf_interact(const bf_interact_t *q, double *e, int32_t *h_dcal, double *ed, int32_t *site, char *ss_out);

/* Direct refolding paths (ViennaRNA's findpath: fc.path_findpath_saddle / fc.path_findpath; not called by DesiRNA).  HOST buffers,
 * synchronous.
 * Each instance r has a single-strand sequence (ACGU, T accepted, len[r] <= stride <= 2000), two structures s1 and s2 of len[r]
 * characters ('.', '(' and ')' only, balanced, every pair with j - i >= 4; pairs need not be canonical) and the call's width W,
 * 1 .. 1024.
 * E(x) is the energy of structure x exactly as bf_score_batch with BF_WANT_EVAL returns it: int dcal/mol, non-standard pairs
 * scored as type 7.
 * One run (a -> b, width w): the moves are the deletions D = pairs of a not in b, ascending i, then the insertions I = pairs of b
 * not in a, ascending i, indexed 0 .. k-1 with k = |D| + |I|.  A state is a set of moves done; its structure is a minus the
 * deleted pairs plus the inserted pairs, and it is valid when no position is in two pairs and no two pairs cross.
 *   Level 0 is {a}, with saddle E(a).
 *   Level t+1 holds every valid one-move successor of the states kept at level t, with saddle = max(parent saddle, E(child)).
 *   Successors with the same move set are one state; it keeps the least (saddle, parent rank, move index).
 *   States are ordered by (saddle, E, parent rank, move index); the first w are kept, and their positions are their ranks.
 * A level is never empty (while a deletion remains it is valid; once all are done every remaining insertion is compatible), so
 * level k is exactly {b}.
 * Runs of a call: w = 1, 2, 4, ... (the powers of two below W), then W; each w runs forward (s1 -> s2), then reverse (s2 -> s1).
 * The result is the run with the least saddle; ties go to the first run in that order.
 * The path is reported from s1 to s2 (a reverse run's path is reversed, so its deletions become insertions):
 *   saddle_dcal: n saddles (dcal/mol), = max(path_e);
 *   n_moves:     NULL or n counts k;
 *   moves:       NULL or n x stride x 2: move m of instance r is (i, j), 1-based, positive for an insertion and negative for a
 *                deletion (ViennaRNA's vrna_move_t sign convention); 0 past k;
 *   path_e:      NULL or n x (stride + 1): E of the k + 1 structures of the path, E(s1) first; 0 past k.
 * Every intermediate is a valid secondary structure.  The saddle does not increase from W' to W for every power of two W' <= W (the
 * runs of W' are a subset of those of W), and when W is at least the largest level it is the optimum over all direct paths.
 * Not pinned: ViennaRNA's exact width schedule, direction alternation and tie order are recalled; no ViennaRNA output in the tree
 * pins them.
 * BF_ERR_ARG: null q or saddle_dcal, n < 0, stride < 1 or > 2000, len < 0 or > stride, width outside 1 .. 1024, a sequence
 * character other than ACGUT, an unbalanced structure, another character, a pair with j - i < 4.  BF_ERR_NOT_INIT before bf_init or
 * before parameters are loaded. */
typedef struct {
  int32_t n, stride;       /* instances; bytes between rows of seq, s1 and s2 */
  const char *seq;         /* n x stride */
  const int32_t *len;      /* n */
  const char *s1, *s2;     /* n x stride dot-bracket */
  int32_t width;           /* W, 1 .. 1024 */
} bf_findpath_t;
int bf_findpath(const bf_findpath_t *q, int32_t *saddle_dcal, int32_t *n_moves, int32_t *moves, int32_t *path_e);

/* Folding kinetics (Kinfold-style trajectories; not called by DesiRNA).  HOST buffers, synchronous.
 * States: the secondary structures of one strand whose pairs are all canonical (AU, CG, GU either way) with j - i >= 4, no position
 * in two pairs, no two pairs crossing.  E(x) is the energy of x exactly as bf_score_batch with BF_WANT_EVAL returns it (int dcal/mol).
 * Moves of x: deleting any pair of x; inserting a canonical pair (i, j), j - i >= 4, i and j unpaired, crossing no pair of x (both
 * in the same loop).  No shift moves.  The canonical move order is (i, j) ascending; a pair is in x or not, so one list holds both.
 * Rate of a move x -> y: k(dE), dE = E(y) - E(x), kT = the loaded parameter set's kT (cal/mol), taken from a table over integer
 * dE in [-32768, 32767] built on the host in double:
 *   rule 0, Kawasaki:   k = exp(-dE * 10 / (2 kT));
 *   rule 1, Metropolis: k = min(1, exp(-dE * 10 / kT)).
 * Stochastic step (Gillespie's direct method), at state x and time t:
 *   the valid moves in canonical order are cut into consecutive groups of 32.  Within a group the rates v[0 .. 31] (0 past the last
 *   move) are combined by a 5-step inclusive scan: for o = 1, 2, 4, 8, 16, v[l] += v[l - o] for l >= o, all at once.  A running
 *   double R starts at 0 and adds each group's v[31] in group order; K is the final R, and the running prefix of move l of group g
 *   is R(before g) + v[l].
 *   Each step draws u1, then u2, from the trajectory's splitmix64 stream, seeded from (seed, instance r, trajectory k) alone as
 *   bf_sample seeds (seed, row, sample).  dt = -ln(1 - u1) / K.  If t + dt > t_max, the trajectory ends at t_max in x.  Otherwise
 *   t += dt and the move taken is the first whose running prefix exceeds u2 K (the last valid move if none does, by rounding).
 *   K = 0 (no move): x is absorbing until t_max.
 * Steepest descent (rule 2): each step takes the move of least dE, ties to the first in canonical order, and only if dE < 0; the
 * walk ends at a local minimum.  t stays 0; seed, t_max and the snapshot times are not read.
 * Stop structure (optional, per instance): absorbing; reaching it ends the trajectory with status 1 at that time.
 * max_steps moves end a trajectory with status 2 (unless its last move reached the stop structure).
 * Inputs: n instances (seq, len, stride as in bf_findpath, len <= stride <= 2000); start (NULL: the open chain) and stop (NULL:
 * none), n x stride dot-brackets; n_traj trajectories per instance; rule; t_max; seed; max_steps; n_snap ascending snapshot times
 * in [0, t_max].
 * Outputs, per trajectory u = r * n_traj + k (caller-owned, NULL to skip, except status):
 *   status:  0 t_max reached (rule 2: a local minimum), 1 stop structure reached, 2 max_steps moves;
 *   t_end:   the time the trajectory ended (t_max, the time of the hit or of the last move; 0 for rule 2);
 *   steps:   moves made;
 *   e_end, ss_end: E and the structure at the end, ss_end stride + 1 chars per trajectory, NUL-padded;
 *   e_snap, ss_snap: n_snap per trajectory, the state occupied at t_s (the state entered at the last move at or before t_s).  After
 *   a hit that is the stop structure; after a cap, and for rule 2, 10000000 and an empty string.
 * Device workspaces and outputs stay within a fixed budget (1 GB; bf_set_option "kinfold_mb"); a call that does not fit runs in
 * several launches and its results do not depend on the split.
 * Not reproduced: Kinfold's defaults -- shift moves, its multiloop and dangle options, --noLP, growth (--grow), energy cutoffs.  Its
 * time unit (k0 = 1) and default --time 500 are recalled; no Kinfold output in the tree pins them.
 * BF_ERR_ARG: null q or status, n < 0, n_traj < 1, stride outside 1 .. 2000, len < 0 or > stride, a sequence character other than
 * ACGUT, an unbalanced start or stop structure or another character, a non-canonical pair or one with j - i < 4, rule outside
 * 0 .. 2, t_max not finite or <= 0 (rules 0, 1), n_snap < 0, snapshot times not ascending or outside [0, t_max] (rules 0, 1),
 * max_steps < 1.  BF_ERR_NOT_INIT before bf_init or before parameters are loaded. */
typedef struct {
  int32_t n, stride;       /* instances; bytes between rows of seq, start and stop */
  const char *seq;         /* n x stride */
  const int32_t *len;      /* n */
  const char *start;       /* n x stride dot-bracket, or NULL: the open chain */
  const char *stop;        /* n x stride dot-bracket, or NULL: none */
  int32_t n_traj;          /* trajectories per instance, >= 1 */
  int32_t rule;            /* 0 Kawasaki, 1 Metropolis, 2 steepest descent */
  double t_max;
  uint64_t seed;
  int64_t max_steps;
  int32_t n_snap;
  const double *t_snap;    /* n_snap ascending times */
} bf_kinfold_t;
int bf_kinfold(const bf_kinfold_t *q, int32_t *status, double *t_end, int64_t *steps, int32_t *e_end, char *ss_end, int32_t *e_snap,
               char *ss_snap);

/* Accessibility (not called by DesiRNA; RNAplfold -u, RNA.pfl_fold_up).  HOST buffers, synchronous.
 * Global: for a sequence of length n, P_u(i, u) is the probability that none of positions i .. i+u-1 is paired, in exactly the
 * ensemble of bf_score_batch's BF_WANT_PF / BF_WANT_BPP (loaded parameters, dangles = 2, pf_smooth, the per-nucleotide scale taken
 * from the MFE).  Equivalently P_u(i, u) = Z(positions i .. i+u-1 may not pair) / Z.  Values are clamped to [0, 1] against rounding.
 * pu_out: B x stride x max_u doubles, [r][i-1][u-1] = P_u(i, u); 0 where i+u-1 > len.
 * BF_ERR_UNAVAILABLE: a row with cut > 0, a nopair mask (the partition function ignores constraints), a stride the PF fill path does
 * not cover (as for BF_WANT_BPP; at present above 668) or BF_FORCE_GENERIC.  BF_ERR_ARG: null buffers, len > stride, max_u outside
 * 1 .. stride. */
int bf_unpaired(const bf_batch_t *batch, int32_t max_u, double *pu_out);
/* RNAplfold with span = window size (RNA.pfl_fold / RNA.pfl_fold_up).  For a strand of length n let W' = min(winsize, n); the windows
 * are the substrings s .. s+W'-1, s = 1 .. n-W'+1, each folded as an isolated sequence under the global model above (its end
 * nucleotides have no outside neighbours).
 *   pbar(i, j):    the mean, over the windows that contain both i and j, of that window's pair probability;
 *   pbar_u(i, u):  the mean, over the windows that contain i .. i+u-1, of that window's P_u.
 * All windows of all strands of s run through one pipeline, in chunks of consecutive windows within a fixed memory budget; every chunk
 * runs the kernels chosen for the whole call and each average is summed in window order, so the result does not depend on the
 * chunking.  Not pinned by any ViennaRNA output here: whether
 * ViennaRNA's window folds let exterior-loop dangles see the nucleotides just outside the window, and the shim's output conventions.
 * A maximum base-pair span smaller than the window is not supported.
 * bpp_out: NULL or n x stride x winsize doubles, [r][i-1][d] = pbar(i, i+d); 0 where d < 4, i+d > len or d >= W'.
 * pu_out:  NULL or n x stride x max_u doubles, [r][i-1][u-1] = pbar_u(i, u); 0 where i+u-1 > len.
 * BF_ERR_ARG: both outputs NULL, null strands, len < 0 or > stride, winsize < 1, max_u outside 1 .. winsize.
 * BF_ERR_UNAVAILABLE: winsize > 2000, a window W' longer than the PF fill path covers (as for bf_unpaired), or BF_FORCE_GENERIC. */
int bf_plfold(const bf_strands_t *s, int32_t winsize, int32_t max_u, double *bpp_out, double *pu_out);

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
 *   "plfold_mb" N: memory budget of one bf_plfold chunk in MB (default 1024); the result does not depend on it.
 *   "kinfold_mb" N: memory budget of bf_kinfold's device workspaces and outputs in MB (default 1024); the result does not depend on it.
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
