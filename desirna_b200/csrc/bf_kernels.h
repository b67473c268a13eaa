// bf_kernels.h -- host-visible planners and launchers of the fold kernels.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "bf_params.h"

struct BfBatchDev;

// Switches that override a default kernel-selection rule, read from the environment variable of that name at call time
// (bf_capi.cu holds the list; bf_set_option sets them from the host program).  Unset or empty: dflt.
int bf_opt(const char *name, int dflt);

// The per-call switches (include/b200fold.h), read once by each bf_plan_* call; each field holds the default when unset.
struct BfOpts {
  int wide, fill3, fill3_small, blk_min, blk_min_pf, cl, cl_c, cl_bw, ext_wide;
};
BfOpts bf_opts();

// ---- one fold pass of one call: which kernel runs it, with what grid, shared memory and workspace.  bf_plan_* decides once per
// pass; the launchers follow the plan and choose nothing.
enum BfFamily {
  BF_FAM_GENERIC,   // bf_kernels.cu: W x W tables per CTA (two strands, lengths the fill path does not cover, BF_FORCE_GENERIC)
  BF_FAM_CLUSTER,   // bf_cluster.cu: a thread-block cluster per sequence
  BF_FAM_TAP,       // bf_fill3.cu: flat tap tables
  BF_FAM_ROUND1,    // bf_fill.cu: diagonal-major round-1 fills
};
enum BfExtRoute {
  BF_EXT_IN_FILL,   // the fill kernel runs the exterior recursion itself (16-warp round-1 fills; the generic kernels)
  BF_EXT_CTA,       // bf_ext.cu: one CTA per sequence
  BF_EXT_WARP,      // bf_k_trace / bf_k_pf_ext: one warp per sequence
};
struct BfPlan {
  BfFamily family;
  int key;              // instantiation within the family (its kernel table's index; cluster: C; outside pass: version)
  int bw;               // cluster: block width
  int grid;             // CTAs (cluster family: clusters)
  size_t smem;          // dynamic shared memory per CTA
  size_t ws;            // HBM workspace per CTA / cluster: ints (MFE), doubles (PF, outside pass)
  unsigned tables_off;  // generic: shared-memory offset of the DP tables (0: in HBM)
  BfExtRoute ext;
};

cudaError_t bf_plan_mfe(int stride, int B, bool two, bool force_generic, int sms, BfPlan *p);
cudaError_t bf_plan_pf(int stride, int B, bool two, bool force_generic, int sms, BfPlan *p);
cudaError_t bf_plan_out(int stride, int B, int sms, BfPlan *p, bool keep = false);   // keep: for bf_launch_pf_out's keep
cudaError_t bf_plan_mfe_out(int stride, int B, int sms, BfPlan *p);   // p->ws: ints per CTA

cudaError_t bf_upload_constants();

// ---- generic kernels (bf_kernels.cu)
cudaError_t bf_gen_mfe_plan(int stride, int B, bool two, const BfOpts &o, int sms, BfPlan *p);
cudaError_t bf_gen_pf_plan(int stride, int B, bool two, const BfOpts &o, int sms, BfPlan *p);
cudaError_t bf_launch_mfe(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, int *ws, int *work_counter, int *out_mfe, char *out_ss,
                          int ss_stride, cudaStream_t st);
cudaError_t bf_launch_pf(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, double *ws, int *work_counter, const int *mfe_for_scale,
                         double *out5, cudaStream_t st);
cudaError_t bf_launch_eval(const BfParams *dP, const BfBatchDev &b, const char *targets, int n_targets, int tstride, int *out_e,
                           cudaStream_t st);

// ---- diagonal-major fill path for single-strand batches (bf_fill.cu, and the routing of bf_plan_mfe / bf_plan_pf)
size_t bf_tri_slot(int nmax);      // entries of one packed triangular table (per sequence)
int bf_fill_mfe_mode(int nmax);    // 0: length not covered (the generic kernels take it); else 1 + placement flags
int bf_fill_pf_mode(int nmax);
// f5_out (B x (stride + 4) ints): written by the fill when p.ext == BF_EXT_IN_FILL, else unused
cudaError_t bf_launch_mfe_fill(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, int *ctri, int *ftri, int *ws, int *work_counter,
                               int *f5_out, cudaStream_t st);
cudaError_t bf_launch_trace(const BfParams *dP, const BfBatchDev &b, const int *ctri, const int *ftri, int *out_mfe, char *out_ss,
                            int ss_stride, cudaStream_t st, const int *f5_in = nullptr);
// qmseq: optional per-sequence qm/qm1 storage (2 x bf_tri_slot doubles per sequence) for the outside pass
// out5: written by the fill when p.ext == BF_EXT_IN_FILL, else unused
cudaError_t bf_launch_pf_fill(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, double *qbtri, double *qmws, double *qmseq,
                              const int *mfe_for_scale, double *lnscale, int *work_counter, double *out5, cudaStream_t st);
cudaError_t bf_launch_pf_ext(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *lnscale, double *out5,
                             cudaStream_t st);

// ---- third-generation fill kernels (bf_fill3.cu): flat tap tables, rings always on chip
// small: the batch leaves SMs idle -- 16-warp CTAs with the whole shared memory of their SM.  Not covered: p is left as it is.
cudaError_t bf_fill3_mfe_plan(int nmax, int B, bool small, const BfOpts &o, int sms, BfPlan *p);
cudaError_t bf_launch_mfe_fill3(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, int *ctri, int *ftri, int *ws, int *work_counter,
                                cudaStream_t st);
cudaError_t bf_fill3_pf_plan(int nmax, int B, bool small, const BfOpts &o, int sms, BfPlan *p);
cudaError_t bf_launch_pf_fill3(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, double *qbtri, double *ws, double *qmseq,
                               const int *mfe_for_scale, double *lnscale, int *work_counter, cudaStream_t st);

// ---- cluster-per-sequence fill kernels (bf_cluster.cu): tables partitioned over the shared memories of a thread-block cluster
// true: the cluster kernel takes this batch (default rule, BF_CL=0/1 override) and p holds its plan
bool bf_cl_mfe_plan(int nmax, int B, const BfOpts &o, BfPlan *p);
cudaError_t bf_launch_mfe_cl(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, int *ctri, int *ftri, int *ws, int *work_counter,
                             cudaStream_t st);
bool bf_cl_pf_plan(int nmax, int B, const BfOpts &o, BfPlan *p);
cudaError_t bf_launch_pf_cl(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, double *qbtri, double *ws, double *qmseq,
                            const int *mfe_for_scale, double *lnscale, int *work_counter, cudaStream_t st);

// ---- second-best structure energy by a 2-best DP on the unambiguous grammar (bf_twobest.cu)
size_t bf_twobest_slot(int wstride);   // int2 entries of HBM workspace per CTA
cudaError_t bf_launch_twobest(const BfParams *dP, const BfBatchDev &b, int2 *ws, int wstride, int grid, int *work_counter, int *out_e1, int *out_e2,
                              cudaStream_t st, const uint8_t *only = nullptr,    // only: optional per-sequence flags, 0 = skip
                              bool two = false);                                 // two: some row has a cut (b.cut), nick-aware grammar

// ---- exterior recursions for small batches (bf_ext.cu): one CTA per sequence
bool bf_ext_wide_ok(int nmax);
cudaError_t bf_launch_f5_wide(const BfParams *dP, const BfBatchDev &b, const int *ctri, int *f5_out, cudaStream_t st);   // f5_out: B x (stride + 4)
cudaError_t bf_launch_q5_wide(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *lnscale, double *out5, cudaStream_t st);

// ---- outside pass: base-pair probabilities and ensemble defect (bf_outside.cu)
// keep (plan made with keep): B x 3 x bf_tri_slot doubles, per sequence the packed bqb, bqm and qm1-outside triangles (bf_unpaired.cu)
cudaError_t bf_launch_pf_out(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *qmseq, double *ws,
                             const double *lnscale, const char *targets, int n_targets, int tstride, double *out_defect, double *out_bpp,
                             int *work_counter, cudaStream_t st, double *keep = nullptr);

// ---- accessibility (bf_unpaired.cu): probabilities of unpaired stretches from the tables of a PF fill (qb, qm / qm1 kept) and of the
// outside pass with keep.  pu_out: B x stride x max_u doubles, [r][i-1][u-1] = P(i .. i+u-1 unpaired), 0 where i+u-1 > len.
cudaError_t bf_launch_unpaired(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *qmseq, const double *keep,
                               const double *lnscale, double *ws, size_t ws_bytes, int max_u, double *pu_out, int *work_counter, int sms,
                               cudaStream_t st);
size_t bf_unpaired_ws_bytes(int stride);   // HBM workspace of one CTA of bf_k_unpaired
// RNAplfold window averages: windows w0 .. w0 + nw - 1 of the call (strand-major, window s of strand r is global window win0[r] + s - 1)
// have been folded as rows 0 .. nw - 1 of a batch of stride wstride (qb, keep; pu: nw x wstride x max_u).  Strands r0 .. r1 - 1 hold
// them.  Each output element adds its windows of this chunk in ascending order to its running sum and divides by its window count in
// the chunk that holds its last window, so the result does not depend on where the chunks end.
struct BfPlfoldDev {
  const int *len, *win0, *wlen;   // per strand: length, first global window, window length min(W, len)
  int stride;                      // of the strands and of the outputs
  int winsize, max_u;              // bpp row width W, pu row width
  int r0, r1;                      // strands of this chunk
  long long w0;                    // first global window of this chunk
  int nw, wstride;
};
cudaError_t bf_launch_plfold_avg(const BfPlfoldDev &d, const double *qbtri, const double *keep, const double *pu, double *bpp_acc,
                                 double *pu_acc, cudaStream_t st);

// ---- minimum-free-energy outside pass (bf_outside.cu): over the c / fML triangles an MFE fill of the same batch left behind.
// e_pair: B x stride x stride ints, [i-1][j-1] = lowest energy of a structure containing (i,j), BF_INF elsewhere.
cudaError_t bf_launch_mfe_out(const BfPlan &p, const BfParams *dP, const BfBatchDev &b, const int *ctri, const int *ftri, int *ws, int *e_pair,
                              int *work_counter, cudaStream_t st);

// ---- stochastic backtracking (bf_sample.cu): n_samples structures per sequence drawn from the tables a PF fill with qmseq kept left
// behind.  q5: B x (stride + 1) doubles of scratch; ss_out: B x n_samples x (stride + 1) chars, sample-major within a row.
cudaError_t bf_launch_sample(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *qmseq, const double *lnscale, double *q5,
                             int n_samples, unsigned long long seed, char *ss_out, int sms, cudaStream_t st);

// ---- RNA-RNA hybridization (bf_duplex.cu): duplex MFE of np pairs (a strand, b strand), pairs p0 .. p0 + np - 1 of the call
struct BfDuplexDev {
  const char *seq_a, *seq_b;   // strands, rows of stride_a / stride_b bytes
  int stride_a, stride_b;
  const int *len_a, *len_b;
  const int *pairs;            // 2 per pair (index into a, index into b), or null: the grid, pair p = (p / nb, p % nb)
  int nb;
  long long p0;
  int np;
  int amax, bmax;              // longest a / b strand of the launch
  int ring_w;                  // largest min(len a, len b) of the launch: the ring's width
};
// true: the c ring of this launch does not fit shared memory and lives in HBM, bf_duplex_ring_slot(ring_w) ints per pair
bool bf_duplex_gring(const BfDuplexDev &d);
size_t bf_duplex_ring_slot(int ring_w);
// e_out: np energies (BF_INF: no pair possible).  ss_out (null: energies only): np x ss_stride chars, a's characters, '&', b's, NUL;
// then ctab holds each pair's n1 x n2 c table at ctab_off[pair - p0] ints.
cudaError_t bf_launch_duplex(const BfParams *dP, const BfDuplexDev &d, bool gring, int *gring_ws, int *e_out, int *ctab,
                             const long long *ctab_off, char *ss_out, int ss_stride, cudaStream_t st);

// ---- accessibility-aware RNA-RNA interaction (bf_interact.cu): the best site of np pairs, pairs p0 .. p0 + np - 1 of the call
struct BfInteractDev {
  const char *seq_a, *seq_b;   // strands, rows of stride_a / stride_b bytes
  int stride_a, stride_b;
  const int *len_a, *len_b;
  const int *pairs;            // as BfDuplexDev
  int nb;
  long long p0;
  int ia0, ib0;                // the grid's pair p0: (p0 / nb, p0 % nb)
  int np;
  int amax, bmax;              // longest a / b strand of the call: units per pair, staging sizes
  int span;                    // max_span, 1 .. 64
  const double *ed_a, *ed_b;   // opening energies [strand][k-1][u-1], rows_a / rows_b positions x span; null: no accessibility
  int rows_a, rows_b;
};
struct BfInteractSlot { double e; long long rank; int h, pad; };   // best site of one (pair, k1) unit; rank -1: none
// per pair of the launch: E, H (BF_INF: no site), packed rank (-1: no site); ed (2 per pair) and site (k1, km, lm, l1) or null
struct BfInteractOut {
  double *e;
  int *h;
  long long *rank;
  double *ed;
  int *site;
};
// slots: np x amax.  ss_out (null: energies only): np x ss_stride chars in bf_duplex's layout.
cudaError_t bf_launch_interact(const BfParams *dP, const BfInteractDev &d, BfInteractSlot *slots, const BfInteractOut &out, char *ss_out,
                               int ss_stride, int *work_counter, int sms, cudaStream_t st);
// ed[x] = -(kT / 1000) ln pu[x] (kcal/mol), +inf where pu[x] <= 0; kT in cal/mol
cudaError_t bf_launch_interact_ed(const double *pu, double *ed, size_t n, double kT, cudaStream_t st);

// ---- direct refolding paths (bf_findpath.cu): the breadth-limited findpath search of n instances, all runs of width W
#define BF_FINDPATH_MAX_LEN 2000
#define BF_FINDPATH_MAX_WIDTH 1024
struct BfFindpathDev {
  int n, stride;               // instances of the launch; row stride of seq and mv (pair tables: stride + 2)
  const char *seq;             // n x stride
  const int *len;              // n
  const short *pt1, *pt2;      // pair tables of s1 / s2, n x (stride + 2), index 0 .. len + 1, 0 = unpaired
  const int *mv;               // n x stride: (i << 16 | j) of the pairs of s1 not in s2 (ascending i), then of s2 not in s1
  const int *nd;               // n x 2: the two counts
  int width, nmax, kw;         // W; workspace shape: longest strand, 64-bit words of the longest move bitset
  long long cap;               // candidate keys per CTA (a power of two >= W x the most moves)
  int2 *bp;                    // back-pointers (parent rank << 16 | move, E) of every run, level-major, from bp_off[r]
  const long long *bp_off;     // n
  int *run_sad, *run_e0;       // n x bf_findpath_runs(W): saddle and start energy of each run
};
size_t bf_findpath_ws_bytes(int width, int nmax, int kw, long long cap);   // one CTA's workspace
long long bf_findpath_cap(int width, int kmax);
int bf_findpath_runs(int width);
int bf_findpath_width_sum(int width);   // sum of w over the runs: back-pointers per instance = moves x this
int bf_findpath_occupancy();
// ws: grid x bf_findpath_ws_bytes.  saddle: n; moves (n x stride x 2) and path_e (n x (stride + 1)) or null.
cudaError_t bf_launch_findpath(const BfParams *dP, const BfFindpathDev &d, unsigned char *ws, int grid, int *work_counter, int *saddle,
                               int *moves, int *path_e, cudaStream_t st);

// ---- folding kinetics (bf_kinfold.cu): trajectories u0 .. u0 + nu - 1 of the call, trajectory u = r x T + k
#define BF_KINFOLD_MAX_LEN 2000
struct BfKinfoldDev {
  int stride, T;               // row stride of seq (pair tables: stride + 2); trajectories per instance
  const char *seq;             // instances x stride
  const int *len;              // per instance
  const short *start, *stop;   // pair tables, instances x (stride + 2), index 0 .. len + 1; stop may be null
  const double *rate;          // 65536 rates, k(dE) at [dE + 32768]
  int rule;                    // 0 Kawasaki, 1 Metropolis, 2 steepest descent
  double t_max;
  unsigned long long seed;
  long long max_steps;
  int n_snap;
  const double *t_snap;        // n_snap ascending times
  long long u0;
  int nu;
  int nmax, gmax;              // longest strand of the call; groups of one warp's workspace
  // outputs of the launch's trajectories, indexed by u - u0
  int *status;
  double *t_end;
  long long *steps;
  int *e_end;
  char *ss_end;                // (stride + 1) per trajectory
  int *e_snap;                 // n_snap per trajectory
  char *ss_snap;               // n_snap x (stride + 1) per trajectory
};
size_t bf_kinfold_smem(int nmax);       // dynamic shared memory of one CTA
size_t bf_kinfold_ws_bytes(int gmax, int nmax);   // HBM workspace of one CTA
int bf_kinfold_occupancy(int nmax);
// ws: grid x bf_kinfold_ws_bytes(d.gmax, d.nmax)
cudaError_t bf_launch_kinfold(const BfParams *dP, const BfKinfoldDev &d, unsigned char *ws, int grid, int *work_counter, cudaStream_t st);

// ---- suboptimal structures (bf_subopt.cu): host walk over the c / fML tables of the GPU fill
#ifdef __cplusplus
#include <string>
#include <utility>
#include <vector>
int bf_wuchty_host(const BfParams *P, int n, const uint8_t *S, const uint8_t *SP, const int *c, const int *fm, int delta, int cap,
                   std::vector<std::pair<int, std::string>> *out, int *mfe_out, bool *truncated);
// Zuker suboptimals: e_pair (n x n, [i-1][j-1]) from bf_launch_mfe_out over the same tables.  Returns the number of structures
// (<= cap; *truncated when more pairs were left uncovered), or -1 if e_pair and the tables disagree.
int bf_zuker_host(const BfParams *P, int n, const uint8_t *S, const uint8_t *SP, const int *c, const int *fm, const int *e_pair, int cap,
                  std::vector<std::pair<int, std::string>> *out, bool *truncated);
#endif
