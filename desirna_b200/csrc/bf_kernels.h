// bf_kernels.h -- host-visible launchers of the fold kernels (bf_kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "bf_params.h"

struct BfBatchDev;

// Switches that override a default kernel-selection rule, read from the environment variable of that name at call time
// (bf_capi.cu holds the list; bf_set_option sets them from the host program).  Unset or empty: dflt.
int bf_opt(const char *name, int dflt);

cudaError_t bf_upload_constants();
size_t bf_mfe_slot_ints(int wstride);
size_t bf_pf_slot_doubles(int wstride);
int bf_occupancy_mfe(bool two, int wstride);
int bf_occupancy_pf(bool two, int wstride);

cudaError_t bf_launch_mfe(const BfParams *dP, const BfBatchDev &b, bool two, int *ws, int wstride, int grid, int *work_counter,
                          int *out_mfe, char *out_ss, int ss_stride, cudaStream_t st);
cudaError_t bf_launch_pf(const BfParams *dP, const BfBatchDev &b, bool two, double *ws, int wstride, int grid, int *work_counter,
                         const int *mfe_for_scale, double *out5, cudaStream_t st);
cudaError_t bf_launch_eval(const BfParams *dP, const BfBatchDev &b, const char *targets, int n_targets, int tstride, int *out_e,
                           cudaStream_t st);

// ---- diagonal-major fill path for single-strand batches (bf_fill.cu)
size_t bf_tri_slot(int nmax);      // entries of one packed triangular table (per sequence)
int bf_fill_mfe_mode(int nmax);    // 0: length not covered (the generic kernels take it); else 1 + placement flags
int bf_fill_pf_mode(int nmax);
size_t bf_mfe_ws_slot(int nmax, int B);   // ints of per-CTA HBM workspace of the MFE fill (B: batch size, selects the 16-warp variant)
size_t bf_pf_ws_slot(int nmax, int B);    // doubles of per-CTA HBM workspace of the PF fill
void bf_fill_set_sms(int sms);    // SM count of the device (batches of at most that many sequences use 16-warp CTAs)
cudaError_t bf_mfe_fill_grid(const BfBatchDev &b, int sms, int *grid);
cudaError_t bf_pf_fill_grid(const BfBatchDev &b, int sms, int *grid);
// f5_out / f5_in (B x (stride + 4) ints): the 16-warp fill variants run the exterior recursion themselves (bf_mfe_fill_does_ext)
cudaError_t bf_launch_mfe_fill(const BfParams *dP, const BfBatchDev &b, int *ctri, int *ftri, int *ws, int sms, int *work_counter,
                               cudaStream_t st, int *f5_out = nullptr);
bool bf_mfe_fill_does_ext(int nmax, int B);
cudaError_t bf_launch_trace(const BfParams *dP, const BfBatchDev &b, const int *ctri, const int *ftri, int *out_mfe, char *out_ss,
                            int ss_stride, cudaStream_t st, const int *f5_in = nullptr);
// qmseq: optional per-sequence qm/qm1 storage (2 x bf_tri_slot doubles per sequence) for the outside pass
cudaError_t bf_launch_pf_fill(const BfParams *dP, const BfBatchDev &b, double *qbtri, double *qmws, double *qmseq, const int *mfe_for_scale,
                              double *lnscale, int sms, int *work_counter, cudaStream_t st, double *out5 = nullptr);
// true: the fill kernel chosen for (nmax, B) runs the exterior recursion itself and writes out5 (16-warp variants)
bool bf_pf_fill_does_ext(int nmax, int B);
cudaError_t bf_launch_pf_ext(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *lnscale, double *out5,
                             cudaStream_t st);

// ---- third-generation fill kernels (bf_fill3.cu): flat tap tables, rings always on chip
// small: the batch leaves SMs idle -- 16-warp CTAs with the whole shared memory of their SM (the caller decides, see bf_fill.cu)
bool bf_fill3_mfe_ok(int nmax, bool small);
size_t bf_fill3_mfe_ws_slot(int nmax);   // ints of per-CTA HBM workspace (per-cell constants of one sequence)
cudaError_t bf_fill3_mfe_grid(const BfBatchDev &b, int sms, int *grid, bool small);
cudaError_t bf_launch_mfe_fill3(const BfParams *dP, const BfBatchDev &b, int *ctri, int *ftri, int *ws, int sms, int *work_counter,
                                cudaStream_t st, bool small);

bool bf_fill3_pf_ok(int nmax, bool small);
size_t bf_fill3_pf_ws_slot(int nmax);    // doubles of per-CTA HBM workspace
cudaError_t bf_fill3_pf_grid(const BfBatchDev &b, int sms, int *grid, bool small);
cudaError_t bf_launch_pf_fill3(const BfParams *dP, const BfBatchDev &b, double *qbtri, double *ws, double *qmseq, const int *mfe_for_scale,
                               double *lnscale, int sms, int *work_counter, cudaStream_t st, bool small);

// ---- cluster-per-sequence fill kernels (bf_cluster.cu): tables partitioned over the shared memories of a thread-block cluster
bool bf_cl_mfe_use(int nmax, int B);           // does the cluster kernel take this batch (default rule, BF_CL=0/1 override)
int bf_cl_mfe_csize(int nmax, int B);          // cluster size it would use (0: length not covered)
size_t bf_cl_mfe_ws_slot(int nmax, int B);     // ints of HBM workspace per cluster
cudaError_t bf_cl_mfe_grid(const BfBatchDev &b, int sms, int *nclusters);
cudaError_t bf_launch_mfe_cl(const BfParams *dP, const BfBatchDev &b, int *ctri, int *ftri, int *ws, int sms, int *work_counter,
                             cudaStream_t st);
bool bf_cl_pf_use(int nmax, int B);
int bf_cl_pf_csize(int nmax, int B);
size_t bf_cl_pf_ws_slot(int nmax, int B);      // doubles of HBM workspace per cluster
cudaError_t bf_cl_pf_grid(const BfBatchDev &b, int sms, int *nclusters);
cudaError_t bf_launch_pf_cl(const BfParams *dP, const BfBatchDev &b, double *qbtri, double *ws, double *qmseq, const int *mfe_for_scale,
                            double *lnscale, int sms, int *work_counter, cudaStream_t st);

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
size_t bf_out_ws_slot(int nmax);   // doubles of per-CTA HBM workspace
cudaError_t bf_out_grid(const BfBatchDev &b, int sms, int *grid);
cudaError_t bf_launch_pf_out(const BfParams *dP, const BfBatchDev &b, const double *qbtri, const double *qmseq, double *ws,
                             const double *lnscale, const char *targets, int n_targets, int tstride, double *out_defect, double *out_bpp,
                             int grid, int *work_counter, cudaStream_t st);

// ---- suboptimal structures (bf_subopt.cu): host walk over the c / fML tables of the GPU fill
#ifdef __cplusplus
#include <string>
#include <utility>
#include <vector>
int bf_wuchty_host(const BfParams *P, int n, const uint8_t *S, const uint8_t *SP, const int *c, const int *fm, int delta, int cap,
                   std::vector<std::pair<int, std::string>> *out, int *mfe_out, bool *truncated);
#endif
