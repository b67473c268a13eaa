// bf_capi.cu -- engine state and the C-ABI declared in include/b200fold.h.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/b200fold.h"
#include "bf_design.h"
#include "bf_device.cuh"
#include "bf_kernels.h"
#include "bf_params.h"

// The switches that override a default kernel-selection rule (include/b200fold.h lists what each does).  They are read where the
// choice is made (BF_FORCE_GENERIC at bf_init, BF_DESIGN_OVERLAP at bf_design_create, the others at every call), so that a host
// program can flip them between calls on one engine.
static const char *const kOptions[] = {"BF_CL", "BF_CL_C", "BF_CL_BW", "BF_EXT_WIDE", "BF_WIDE", "BF_FILL3", "BF_FILL3_SMALL",
                                       "BF_BLK_MIN", "BF_BLK_MIN_PF", "BF_FORCE_GENERIC", "BF_DESIGN_OVERLAP", "BF_PLFOLD_MB",
                                       "BF_FINDPATH_MB", "BF_KINFOLD_MB"};

int bf_opt(const char *name, int dflt) {
  const char *v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
}

BfOpts bf_opts() {
  BfOpts o;
  o.wide = bf_opt("BF_WIDE", 1);
  o.fill3 = bf_opt("BF_FILL3", 1);
  o.fill3_small = bf_opt("BF_FILL3_SMALL", 1);
  o.blk_min = bf_opt("BF_BLK_MIN", 280);
  o.blk_min_pf = bf_opt("BF_BLK_MIN_PF", 250);
  o.cl = bf_opt("BF_CL", -1);
  o.cl_c = bf_opt("BF_CL_C", 0);
  o.cl_bw = bf_opt("BF_CL_BW", 32);
  o.ext_wide = bf_opt("BF_EXT_WIDE", -1);
  return o;
}

namespace {

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// Engine-internal device memory of one pipeline invocation (DP tables, per-CTA workspaces, work counters, timing events).
// The engine owns one for the bf_score_batch* entry points; every design loop (bf_design_*) owns its own, so that loops
// running on different streams never share tables.
struct Workspace {
  int *d_counters = nullptr;  // work counters (one per kernel kind)
  DevBuf ws_mfe, ws_pf, d_mfe_scratch;
  DevBuf tri_c, tri_f, tri_qb, ws_qm, ws_ring, d_lnscale, qm_seq, ws_out;  // diagonal-major fill path (bf_fill.cu)
  DevBuf f5buf;  // f5 of every sequence when the fill kernel runs the exterior recursion (16-warp variants)
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // begin/end of mfe, pf, eval in the last call
  bool ran[3] = {false, false, false};
  // the partition function of a small batch can run beside the MFE fill on SMs of its own (run_device: scale_override)
  cudaStream_t st2 = nullptr, st3 = nullptr;   // st3: eval_structure of a small batch (it reads the sequence and the targets only)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join3 = nullptr;
  cudaError_t create() {
    cudaError_t e = cudaMalloc(&d_counters, 8 * sizeof(int));
    for (int k = 0; k < 6 && e == cudaSuccess; k++) e = cudaEventCreate(&ev[k]);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st3, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev_join3, cudaEventDisableTiming);
    return e;
  }
  void destroy() {
    for (DevBuf *b : {&ws_mfe, &ws_pf, &d_mfe_scratch, &tri_c, &tri_f, &tri_qb, &ws_qm, &ws_ring, &d_lnscale, &qm_seq, &ws_out, &f5buf}) b->release();
    if (d_counters) cudaFree(d_counters);
    d_counters = nullptr;
    for (int k = 0; k < 6; k++) { if (ev[k]) cudaEventDestroy(ev[k]); ev[k] = nullptr; }
    if (ev_fork) cudaEventDestroy(ev_fork);
    if (ev_join) cudaEventDestroy(ev_join);
    if (ev_join3) cudaEventDestroy(ev_join3);
    if (st2) cudaStreamDestroy(st2);
    if (st3) cudaStreamDestroy(st3);
    ev_fork = ev_join = ev_join3 = nullptr; st2 = st3 = nullptr;
  }
};

struct Engine {
  bool inited = false, have_params = false;
  int device = 0, sm_count = 0;
  cudaStream_t stream = nullptr;
  BfParams *hP = nullptr;  // host image
  BfParams *dP = nullptr;  // device image
  Workspace w;             // tables and workspaces of the bf_score_batch* entry points
  bool force_generic = false;                     // BF_FORCE_GENERIC=1: route single strands through the generic kernels too
  // staging for the host-buffer entry point
  DevBuf d_seq, d_len, d_cut, d_nopair, d_targets, d_mfe, d_ss, d_pf, d_eval, d_defect, d_bpp;
  DevBuf d_q5, d_samples;  // bf_sample: exterior prefixes, drawn structures
  DevBuf d_epair;          // bf_pair_mfe: E_pair of every sequence
  // bf_unpaired / bf_plfold: kept outside triangles, bf_k_unpaired's workspace, P_u of every row; per-strand window tables, averages
  DevBuf d_keep, d_upws, d_pu, d_pfstr, d_pfbpp, d_pfpu;
  // bf_duplex: strands, pair list, per-pair c-table offsets, c tables / HBM rings, energies, structures
  DevBuf d_dxa, d_dxb, d_dxlen, d_dxpairs, d_dxoff, d_dxws, d_dxe, d_dxss;
  // bf_interact (strands and pair list in the bf_duplex buffers above): opening-energy tables of each side, per-unit slots, results
  DevBuf d_ixeda, d_ixedb, d_ixslot, d_ixres;
  // bf_findpath: sequences, lengths, pair tables, move lists and counts, back-pointer offsets, per-CTA workspaces, back-pointers, per-run
  // saddles and start energies, results
  DevBuf d_fpseq, d_fplen, d_fppt, d_fpmv, d_fpnd, d_fpoff, d_fpws, d_fpbp, d_fprun, d_fpout;
  // bf_kinfold: sequences, lengths, start / stop pair tables, rate table, snapshot times, per-CTA workspaces, outputs of one launch
  DevBuf d_kfseq, d_kflen, d_kfpt, d_kfrate, d_kfsnap, d_kfws, d_kfout;
  // small batches (a replica-exchange sub-step scored through the host-buffer call): inputs packed into one pinned block and one H2D
  // copy, results into one device block and one D2H copy
  DevBuf d_in, d_out, d_zero;
  void *h_in = nullptr, *h_out = nullptr;
  size_t h_in_cap = 0, h_out_cap = 0, zero_cap = 0;
  int64_t launches = 0;
  int last_stride = 0;
  std::string err;
};

Engine g;

int fail(int code, const std::string &msg) { g.err = msg; return code; }
int cuda_fail(cudaError_t e, const char *what) { return fail(BF_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e)); }

#define CU(call, what)                                  \
  do {                                                  \
    cudaError_t e_ = (call);                            \
    if (e_ != cudaSuccess) return cuda_fail(e_, what);  \
  } while (0)

int upload_params() {
  if (!g.dP) CU(cudaMalloc(&g.dP, sizeof(BfParams)), "cudaMalloc(params)");
  CU(cudaMemcpy(g.dP, g.hP, sizeof(BfParams), cudaMemcpyHostToDevice), "upload parameter image");
  g.have_params = true;
  return BF_OK;
}

int validate(const bf_batch_t *b, const bf_result_t *r) {
  if (!b || !r) return fail(BF_ERR_ARG, "null batch/result");
  if (b->B < 0 || b->stride <= 0) return fail(BF_ERR_ARG, "bad batch shape");
  if (b->B && (!b->seq || !b->len)) return fail(BF_ERR_ARG, "seq/len missing");
  if (b->stride > 4000) return fail(BF_ERR_ARG, "stride > 4000 not supported");
  if ((b->want & BF_WANT_SS) && !r->mfe_ss) return fail(BF_ERR_ARG, "BF_WANT_SS without mfe_ss buffer");
  if ((b->want & BF_WANT_MFE) && !r->mfe_dcal) return fail(BF_ERR_ARG, "BF_WANT_MFE without mfe_dcal buffer");
  if ((b->want & BF_WANT_PF) && !r->pf) return fail(BF_ERR_ARG, "BF_WANT_PF without pf buffer");
  if ((b->want & BF_WANT_EVAL) && (!r->eval_dcal || !b->targets || b->n_targets <= 0)) return fail(BF_ERR_ARG, "BF_WANT_EVAL without targets/eval_dcal");
  if ((b->want & BF_WANT_DEFECT) && (!r->defect || !b->targets || b->n_targets <= 0)) return fail(BF_ERR_ARG, "BF_WANT_DEFECT without targets/defect buffer");
  if ((b->want & BF_WANT_BPP) && !r->bpp) return fail(BF_ERR_ARG, "BF_WANT_BPP without bpp buffer");
  if ((b->want & (BF_WANT_BPP | BF_WANT_DEFECT)) && !r->pf) return fail(BF_ERR_ARG, "BF_WANT_BPP/DEFECT need the pf buffer too");
  return BF_OK;
}

// all pointers are device pointers
// scale_override (device, B ints, dcal/mol): energies that set the partition function's per-nucleotide scale instead of this
// call's own MFE.  The result does not depend on the scale beyond rounding, and without that dependency the partition function
// runs on the workspace's second stream beside the MFE fill -- worth it when both grids fit the GPU together (small batches).
// keep_qm: keep the per-sequence qm / qm1 tables (w.qm_seq) of the PF fill for a pass that reads them after this call (bf_sample);
// the outside pass (BF_WANT_BPP / BF_WANT_DEFECT) keeps them in any case.
// keep_out (device, B x 3 x bf_tri_slot doubles): run the outside pass and keep its bqb / bqm / qm1-outside triangles (bf_unpaired).
// plan_B > 0: choose the kernels as for a batch of plan_B rows (bf_plfold: every chunk of a call runs the same kernels).
int run_device(Workspace &w, const bf_batch_t *b, const bf_result_t *r, bool two, cudaStream_t st, const int *scale_override = nullptr,
               bool timing = true, bool keep_qm = false, double *keep_out = nullptr, int plan_B = 0) {
  if (b->B == 0) return BF_OK;
  BfBatchDev db;
  db.B = b->B; db.stride = b->stride; db.seq = b->seq; db.len = b->len; db.cut = b->cut; db.nopair = b->nopair;
  if (&w == &g.w) g.last_stride = b->stride;
  if (scale_override) CU(cudaEventRecord(w.ev_fork, st), "fork");   // what the second stream has to wait for: the work before this call
  const int *mfe_for_scale = nullptr;
  w.ran[0] = w.ran[1] = w.ran[2] = false;
  bool eval_done = false;
  if (scale_override && (b->want & BF_WANT_EVAL) && (b->want & BF_WANT_PF) && !(b->want & (BF_WANT_BPP | BF_WANT_DEFECT)) && !b->nopair) {
    // side-by-side fills: eval_structure on a stream of its own from the start (the SMs the two fills leave free take it)
    CU(cudaStreamWaitEvent(w.st3, w.ev_fork, 0), "fork eval");
    if (timing) cudaEventRecord(w.ev[4], w.st3);
    CU(bf_launch_eval(g.dP, db, b->targets, b->n_targets, b->stride, r->eval_dcal, w.st3), "launch bf_k_eval");
    if (timing) cudaEventRecord(w.ev[5], w.st3);
    CU(cudaEventRecord(w.ev_join3, w.st3), "join eval");
    w.ran[2] = true;
    g.launches++;
    eval_done = true;
  }
  if (b->want & (BF_WANT_MFE | BF_WANT_SS)) {
    int *out_mfe = r->mfe_dcal;
    if (!out_mfe) { CU(w.d_mfe_scratch.reserve((size_t)b->B * sizeof(int)), "cudaMalloc(mfe scratch)"); out_mfe = (int *)w.d_mfe_scratch.p; }
    char *out_ss = (b->want & BF_WANT_SS) ? r->mfe_ss : nullptr;
    BfPlan p;
    CU(bf_plan_mfe(b->stride, plan_B > 0 ? plan_B : b->B, two, g.force_generic, g.sm_count, &p), "plan the MFE fill");
    if (timing) cudaEventRecord(w.ev[0], st);
    if (p.family != BF_FAM_GENERIC) {
      const size_t slot = bf_tri_slot(b->stride) * sizeof(int);
      CU(w.tri_c.reserve((size_t)b->B * slot), "cudaMalloc(c table)");
      CU(w.tri_f.reserve((size_t)b->B * slot), "cudaMalloc(fML table)");
      CU(w.ws_ring.reserve((size_t)p.grid * p.ws * sizeof(int)), "cudaMalloc(ring workspace)");
      int *f5 = nullptr;
      if (p.ext != BF_EXT_WARP) {
        CU(w.f5buf.reserve((size_t)b->B * (b->stride + 4) * sizeof(int)), "cudaMalloc(f5)");
        f5 = (int *)w.f5buf.p;
      }
      CU(bf_launch_mfe_fill(p, g.dP, db, (int *)w.tri_c.p, (int *)w.tri_f.p, (int *)w.ws_ring.p, w.d_counters + 0,
                            p.ext == BF_EXT_IN_FILL ? f5 : nullptr, st), "launch bf_k_mfe_fill");
      if (p.ext == BF_EXT_CTA) {
        CU(bf_launch_f5_wide(g.dP, db, (const int *)w.tri_c.p, f5, st), "launch bf_k_f5_wide");
        g.launches++;
      }
      CU(bf_launch_trace(g.dP, db, (const int *)w.tri_c.p, (const int *)w.tri_f.p, out_mfe, out_ss, b->stride + 1, st, f5), "launch bf_k_trace");
      g.launches += 2;
    } else {
      CU(w.ws_mfe.reserve((size_t)p.grid * p.ws * sizeof(int)), "cudaMalloc(mfe workspace)");
      CU(bf_launch_mfe(p, g.dP, db, (int *)w.ws_mfe.p, w.d_counters + 0, out_mfe, out_ss, b->stride + 1, st), "launch bf_k_mfe");
      g.launches++;
    }
    if (timing) cudaEventRecord(w.ev[1], st);
    w.ran[0] = timing;
    mfe_for_scale = out_mfe;
  }
  const bool want_out = (b->want & (BF_WANT_BPP | BF_WANT_DEFECT)) != 0 || keep_out;
  const bool want_qm = want_out || keep_qm;
  if ((b->want & BF_WANT_PF) || want_out) {
    BfPlan p;
    CU(bf_plan_pf(b->stride, plan_B > 0 ? plan_B : b->B, two, g.force_generic, g.sm_count, &p), "plan the PF fill");
    if (want_qm && p.family == BF_FAM_GENERIC)
      return fail(BF_ERR_UNAVAILABLE, want_out ? "base-pair probabilities / ensemble defect: single-strand sequences within the fill path's length range only"
                                               : "sampling: single-strand sequences within the fill path's length range only");
    BfBatchDev dbp = db;
    dbp.nopair = nullptr;  // hard constraints are added after fc.pf() in the reference (sequence_utils.py:1181)
    // a constrained MFE is not a bound on the unconstrained ensemble: only use it for scaling when unconstrained
    const bool beside = scale_override && !want_out && !b->nopair;
    cudaStream_t sp = beside ? w.st2 : st;
    if (beside) CU(cudaStreamWaitEvent(sp, w.ev_fork, 0), "fork");
    const int *scale_src = beside ? scale_override : (b->nopair ? nullptr : mfe_for_scale);
    if (timing) cudaEventRecord(w.ev[2], sp);
    if (p.family != BF_FAM_GENERIC) {
      const size_t slot = bf_tri_slot(b->stride) * sizeof(double);
      CU(w.tri_qb.reserve((size_t)b->B * slot), "cudaMalloc(qb table)");
      CU(w.d_lnscale.reserve((size_t)b->B * sizeof(double)), "cudaMalloc(lnscale)");
      CU(w.ws_qm.reserve((size_t)p.grid * p.ws * sizeof(double)), "cudaMalloc(qm workspace)");
      double *qmseq = nullptr;
      if (want_qm) {
        CU(w.qm_seq.reserve((size_t)b->B * 2 * slot), "cudaMalloc(per-sequence qm/qm1)");
        qmseq = (double *)w.qm_seq.p;
      }
      CU(bf_launch_pf_fill(p, g.dP, dbp, (double *)w.tri_qb.p, (double *)w.ws_qm.p, qmseq, scale_src, (double *)w.d_lnscale.p, w.d_counters + 1,
                           p.ext == BF_EXT_IN_FILL ? r->pf : nullptr, sp), "launch bf_k_pf_fill");
      g.launches++;
      if (p.ext == BF_EXT_CTA) {
        CU(bf_launch_q5_wide(g.dP, dbp, (const double *)w.tri_qb.p, (const double *)w.d_lnscale.p, r->pf, sp), "launch bf_k_q5_wide");
        g.launches++;
      } else if (p.ext == BF_EXT_WARP) {
        CU(bf_launch_pf_ext(g.dP, dbp, (const double *)w.tri_qb.p, (const double *)w.d_lnscale.p, r->pf, sp), "launch bf_k_pf_ext");
        g.launches++;
      }
      if (want_out) {
        BfPlan po;
        CU(bf_plan_out(b->stride, plan_B > 0 ? plan_B : b->B, g.sm_count, &po, keep_out != nullptr), "plan bf_k_pf_out");
        CU(w.ws_out.reserve((size_t)po.grid * po.ws * sizeof(double)), "cudaMalloc(outside workspace)");
        if (b->want & BF_WANT_BPP) CU(cudaMemsetAsync(r->bpp, 0, (size_t)b->B * b->stride * b->stride * sizeof(double), st), "clear bpp");
        CU(bf_launch_pf_out(po, g.dP, dbp, (const double *)w.tri_qb.p, qmseq, (double *)w.ws_out.p, (const double *)w.d_lnscale.p,
                            (b->want & BF_WANT_DEFECT) ? b->targets : nullptr, b->n_targets, b->stride,
                            (b->want & BF_WANT_DEFECT) ? r->defect : nullptr, (b->want & BF_WANT_BPP) ? r->bpp : nullptr,
                            w.d_counters + 2, st, keep_out), "launch bf_k_pf_out");
        g.launches++;
      }
    } else {
      CU(w.ws_pf.reserve((size_t)p.grid * p.ws * sizeof(double)), "cudaMalloc(pf workspace)");
      CU(bf_launch_pf(p, g.dP, dbp, (double *)w.ws_pf.p, w.d_counters + 1, scale_src, r->pf, sp), "launch bf_k_pf");
      g.launches++;
    }
    if (timing) cudaEventRecord(w.ev[3], sp);
    if (beside) { CU(cudaEventRecord(w.ev_join, sp), "join"); CU(cudaStreamWaitEvent(st, w.ev_join, 0), "join"); }
    w.ran[1] = timing;
  }
  if (eval_done) CU(cudaStreamWaitEvent(st, w.ev_join3, 0), "join eval");
  if ((b->want & BF_WANT_EVAL) && !eval_done) {
    if (timing) cudaEventRecord(w.ev[4], st);
    CU(bf_launch_eval(g.dP, db, b->targets, b->n_targets, b->stride, r->eval_dcal, st), "launch bf_k_eval");
    if (timing) cudaEventRecord(w.ev[5], st);
    w.ran[2] = true;
    g.launches++;
  }
  return BF_OK;
}

// A small batch asked for both the MFE and the ensemble energy: the partition function does not wait for the MFE (which would set
// its per-nucleotide scale) but runs beside it with ViennaRNA's default scale estimate (a zero in scale_override selects it; the
// result depends on the scale through rounding only).  Both grids are one CTA per sequence, so they overlap while 2 B <= SM count;
// up to 400 nt the default scale keeps every scaled quantity far inside the double range (|E| <= 0.9 kcal/mol/nt: < 1e201).
int overlap_scale(const bf_batch_t *b, const int **ov) {
  *ov = nullptr;
  if (!(b->want & (BF_WANT_MFE | BF_WANT_SS)) || !(b->want & BF_WANT_PF) || (b->want & (BF_WANT_BPP | BF_WANT_DEFECT)) || b->nopair) return BF_OK;
  if (2 * b->B > g.sm_count || b->stride > 400) return BF_OK;
  if (g.zero_cap < (size_t)b->B) {
    const size_t n = std::max<size_t>(256, (size_t)b->B);
    CU(g.d_zero.reserve(n * sizeof(int)), "cudaMalloc(zero scale)");
    CU(cudaMemset(g.d_zero.p, 0, n * sizeof(int)), "clear zero scale");
    g.zero_cap = n;
  }
  *ov = (const int *)g.d_zero.p;
  return BF_OK;
}

cudaError_t reserve_pinned(void **p, size_t *cap, size_t n) {
  if (n <= *cap) return cudaSuccess;
  if (*p) cudaFreeHost(*p);
  *p = nullptr; *cap = 0;
  const size_t want = std::max<size_t>(n, 64 << 10);
  cudaError_t e = cudaMallocHost(p, want);
  if (e == cudaSuccess) *cap = want;
  return e;
}

bool any_cut(const bf_batch_t *b, const int32_t *host_cut) {
  if (!host_cut) return false;
  for (int i = 0; i < b->B; i++) if (host_cut[i] > 0) return true;
  return false;
}

}  // namespace

extern "C" {

const char *bf_last_error(void) { return g.err.c_str(); }

int bf_init(int device) {
  if (g.inited) return BF_OK;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) return fail(BF_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e));
  if (device < 0 || device >= count) return fail(BF_ERR_ARG, "device index out of range");
  CU(cudaSetDevice(device), "cudaSetDevice");
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
  if (prop.major < 10) return fail(BF_ERR_CUDA, std::string("built for sm_100a, found ") + prop.name);
  g.device = device;
  g.force_generic = bf_opt("BF_FORCE_GENERIC", 0) == 1;
  g.sm_count = prop.multiProcessorCount;
  CU(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking), "cudaStreamCreate");
  CU(g.w.create(), "create engine workspace");
  CU(bf_upload_constants(), "upload candidate table");
  if (!g.hP) g.hP = new BfParams;
  g.inited = true;
  if (g.have_params) return upload_params();
  return BF_OK;
}

int bf_shutdown(void) {
  if (!g.inited) return BF_OK;
  cudaStreamSynchronize(g.stream);
  for (DevBuf *b : {&g.d_defect, &g.d_bpp, &g.d_seq, &g.d_len, &g.d_cut, &g.d_nopair, &g.d_targets, &g.d_mfe, &g.d_ss, &g.d_pf, &g.d_eval, &g.d_in, &g.d_out, &g.d_zero,
                    &g.d_q5, &g.d_samples, &g.d_epair, &g.d_dxa, &g.d_dxb, &g.d_dxlen, &g.d_dxpairs, &g.d_dxoff, &g.d_dxws, &g.d_dxe,
                    &g.d_dxss}) b->release();
  if (g.h_in) cudaFreeHost(g.h_in);
  if (g.h_out) cudaFreeHost(g.h_out);
  g.h_in = g.h_out = nullptr; g.h_in_cap = g.h_out_cap = g.zero_cap = 0;
  g.w.destroy();
  if (g.dP) cudaFree(g.dP);
  cudaStreamDestroy(g.stream);
  g.dP = nullptr; g.stream = nullptr;
  g.inited = false;
  return BF_OK;
}

int bf_params_load(const char *par_path) {
  if (!par_path) return fail(BF_ERR_ARG, "null path");
  if (!g.hP) g.hP = new BfParams;
  std::string err;
  if (bf_params_parse_file(par_path, g.hP, &err)) { g.have_params = false; return fail(BF_ERR_PARAMS, err); }
  g.hP->year = 0;
  g.have_params = true;
  if (g.inited) return upload_params();
  return BF_OK;
}

int bf_params_builtin(int year, const char *builtin_dir) {
  if (year == 2004)
    return fail(BF_ERR_UNAVAILABLE, "Turner 2004 tables are compiled into ViennaRNA, not shipped with DesiRNA; load rna_turner2004.par with bf_params_load");
  if (year != 1999) return fail(BF_ERR_ARG, "year must be 1999 or 2004");
  if (!builtin_dir) return fail(BF_ERR_ARG, "null builtin_dir");
  std::string p = std::string(builtin_dir) + "/turner1999_37C.par";
  int rc = bf_params_load(p.c_str());
  if (rc == BF_OK) g.hP->year = 1999;
  return rc;
}

int bf_params_get(const char *name, int i0, int i1, int i2, int i3, int i4, int i5, int32_t *out) {
  if (!g.have_params || !g.hP) return fail(BF_ERR_NOT_INIT, "no parameters loaded");
  if (!name || !out) return fail(BF_ERR_ARG, "null argument");
  const BfParams &P = *g.hP;
  auto in = [](int v, int hi) { return v >= 0 && v < hi; };
  std::string n(name);
#define T3(tab) if (n == #tab) { if (!in(i0, 8) || !in(i1, 5) || !in(i2, 5)) return fail(BF_ERR_ARG, "index"); *out = P.si.tab[i0][i1][i2]; return BF_OK; }
  T3(mmH) T3(mmI) T3(mm1nI) T3(mm23I) T3(mmM) T3(mmE)
#undef T3
  if (n == "stack") { if (!in(i0, 8) || !in(i1, 8)) return fail(BF_ERR_ARG, "index"); *out = P.si.stack[i0][i1]; return BF_OK; }
  if (n == "dangle5") { if (!in(i0, 8) || !in(i1, 5)) return fail(BF_ERR_ARG, "index"); *out = P.si.dangle5[i0][i1]; return BF_OK; }
  if (n == "dangle3") { if (!in(i0, 8) || !in(i1, 5)) return fail(BF_ERR_ARG, "index"); *out = P.si.dangle3[i0][i1]; return BF_OK; }
  if (n == "int11") { if (!in(i0, 8) || !in(i1, 8) || !in(i2, 5) || !in(i3, 5)) return fail(BF_ERR_ARG, "index"); *out = P.int11[i0][i1][i2][i3]; return BF_OK; }
  if (n == "int21") { if (!in(i0, 8) || !in(i1, 8) || !in(i2, 5) || !in(i3, 5) || !in(i4, 5)) return fail(BF_ERR_ARG, "index"); *out = P.int21[i0][i1][i2][i3][i4]; return BF_OK; }
  if (n == "int22") { if (!in(i0, 8) || !in(i1, 8) || !in(i2, 5) || !in(i3, 5) || !in(i4, 5) || !in(i5, 5)) return fail(BF_ERR_ARG, "index"); *out = P.int22[i0][i1][i2][i3][i4][i5]; return BF_OK; }
  if (n == "hairpin" || n == "bulge" || n == "interior") {
    if (!in(i0, 31)) return fail(BF_ERR_ARG, "index");
    *out = n == "hairpin" ? P.si.hairpin[i0] : n == "bulge" ? P.si.bulge[i0] : P.si.interior[i0];
    return BF_OK;
  }
  if (n == "ninio_m") { *out = P.si.ninio_m; return BF_OK; }
  if (n == "ninio_max") { *out = P.si.ninio_max; return BF_OK; }
  if (n == "MLbase") { *out = P.si.MLbase; return BF_OK; }
  if (n == "MLclosing") { *out = P.si.MLclosing; return BF_OK; }
  if (n == "MLintern") { *out = P.si.MLintern; return BF_OK; }
  if (n == "DuplexInit") { *out = P.si.DuplexInit; return BF_OK; }
  if (n == "TerminalAU") { *out = P.si.TerminalAU; return BF_OK; }
  if (n == "lxc1000") { *out = (int32_t)(P.lxc * 1000.0 + 0.5); return BF_OK; }
  if (n == "n_tetra") { *out = P.n_tetra; return BF_OK; }
  if (n == "n_tri") { *out = P.n_tri; return BF_OK; }
  if (n == "n_hexa") { *out = P.n_hexa; return BF_OK; }
  if (n == "tetra_e") { if (!in(i0, 4096)) return fail(BF_ERR_ARG, "index"); *out = P.tetra_e[i0]; return BF_OK; }
  return fail(BF_ERR_ARG, "unknown parameter name: " + n);
}

int bf_score_batch_device(const bf_batch_t *b, bf_result_t *r, void *cuda_stream) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  int rc = validate(b, r);
  if (rc) return rc;
  // the cut array lives on the device: the two-strand kernels handle cut == 0 rows as single strands
  const int *ov = nullptr;
  rc = overlap_scale(b, &ov);
  if (rc) return rc;
  return run_device(g.w, b, r, b->cut != nullptr, (cudaStream_t)cuda_stream, ov);
}

int bf_score_batch(const bf_batch_t *b, bf_result_t *r) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  int rc = validate(b, r);
  if (rc) return rc;
  if (b->B == 0) return BF_OK;
  for (int i = 0; i < b->B; i++) {
    if (b->len[i] < 0 || b->len[i] > b->stride) return fail(BF_ERR_ARG, "sequence length exceeds stride");
    if (b->cut && (b->cut[i] < 0 || b->cut[i] > b->len[i])) return fail(BF_ERR_ARG, "cut point outside sequence");
  }
  cudaStream_t st = g.stream;
  const size_t B = b->B, S = b->stride;
  const bool two = any_cut(b, b->cut);
  bf_batch_t db = *b;
  bf_result_t dr;
  std::memset(&dr, 0, sizeof dr);
  const int *ov = nullptr;
  rc = overlap_scale(b, &ov);
  if (rc) return rc;
  const size_t T = (b->want & (BF_WANT_EVAL | BF_WANT_DEFECT)) ? (size_t)b->n_targets : 0;
  auto up = [](size_t x) { return (x + 15) / 16 * 16; };
  // ---- small batches: one pinned block in, one out
  const size_t o_len = up(B * S), o_cut = o_len + up(B * sizeof(int)), o_np = o_cut + (two ? up(B * sizeof(int)) : 0),
               o_tg = o_np + (b->nopair ? up(B * S) : 0), in_bytes = o_tg + up(B * T * S);
  const size_t p_ss = up(B * sizeof(int)), p_pf = p_ss + up(B * (S + 1)), p_ev = p_pf + up(B * 5 * sizeof(double)),
               p_df = p_ev + up(B * std::max<size_t>(T, 1) * sizeof(int)), out_bytes = p_df + up(B * sizeof(double));
  if (in_bytes <= ((size_t)256 << 10) && out_bytes <= ((size_t)256 << 10)) {
    CU(reserve_pinned(&g.h_in, &g.h_in_cap, in_bytes), "cudaMallocHost(inputs)");
    CU(reserve_pinned(&g.h_out, &g.h_out_cap, out_bytes), "cudaMallocHost(results)");
    CU(g.d_in.reserve(in_bytes), "cudaMalloc(inputs)");
    CU(g.d_out.reserve(out_bytes), "cudaMalloc(results)");
    char *hi = (char *)g.h_in, *di = (char *)g.d_in.p, *dou = (char *)g.d_out.p;
    std::memcpy(hi, b->seq, B * S);
    std::memcpy(hi + o_len, b->len, B * sizeof(int));
    if (two) std::memcpy(hi + o_cut, b->cut, B * sizeof(int));
    if (b->nopair) std::memcpy(hi + o_np, b->nopair, B * S);
    if (T) std::memcpy(hi + o_tg, b->targets, B * T * S);
    CU(cudaMemcpyAsync(di, hi, in_bytes, cudaMemcpyHostToDevice, st), "H2D inputs");
    db.seq = di; db.len = (const int32_t *)(di + o_len);
    db.cut = two ? (const int32_t *)(di + o_cut) : nullptr;
    db.nopair = b->nopair ? (const uint8_t *)(di + o_np) : nullptr;
    db.targets = T ? di + o_tg : nullptr;
    if (b->want & (BF_WANT_MFE | BF_WANT_SS)) dr.mfe_dcal = (int32_t *)dou;
    if (b->want & BF_WANT_SS) dr.mfe_ss = dou + p_ss;
    if (b->want & (BF_WANT_PF | BF_WANT_BPP | BF_WANT_DEFECT)) dr.pf = (double *)(dou + p_pf);
    if (b->want & BF_WANT_EVAL) dr.eval_dcal = (int32_t *)(dou + p_ev);
    if (b->want & BF_WANT_DEFECT) dr.defect = (double *)(dou + p_df);
    if (b->want & BF_WANT_BPP) { CU(g.d_bpp.reserve(B * S * S * sizeof(double)), "cudaMalloc(bpp)"); dr.bpp = (double *)g.d_bpp.p; }
    rc = run_device(g.w, &db, &dr, two, st, ov);
    if (rc) return rc;
    CU(cudaMemcpyAsync(g.h_out, dou, out_bytes, cudaMemcpyDeviceToHost, st), "D2H results");
    if (b->want & BF_WANT_BPP) CU(cudaMemcpyAsync(r->bpp, dr.bpp, B * S * S * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H bpp");
    CU(cudaStreamSynchronize(st), "bf_score_batch");
    const char *ho = (const char *)g.h_out;
    if ((b->want & BF_WANT_MFE) && r->mfe_dcal) std::memcpy(r->mfe_dcal, ho, B * sizeof(int));
    if (b->want & BF_WANT_SS) std::memcpy(r->mfe_ss, ho + p_ss, B * (S + 1));
    if ((b->want & (BF_WANT_PF | BF_WANT_BPP | BF_WANT_DEFECT)) && r->pf) std::memcpy(r->pf, ho + p_pf, B * 5 * sizeof(double));
    if (b->want & BF_WANT_EVAL) std::memcpy(r->eval_dcal, ho + p_ev, B * T * sizeof(int));
    if (b->want & BF_WANT_DEFECT) std::memcpy(r->defect, ho + p_df, B * sizeof(double));
    return BF_OK;
  }
  CU(g.d_seq.reserve(B * S), "cudaMalloc(seq)");
  CU(g.d_len.reserve(B * sizeof(int)), "cudaMalloc(len)");
  CU(cudaMemcpyAsync(g.d_seq.p, b->seq, B * S, cudaMemcpyHostToDevice, st), "H2D seq");
  CU(cudaMemcpyAsync(g.d_len.p, b->len, B * sizeof(int), cudaMemcpyHostToDevice, st), "H2D len");
  db.seq = (const char *)g.d_seq.p; db.len = (const int32_t *)g.d_len.p; db.cut = nullptr; db.nopair = nullptr; db.targets = nullptr;
  if (two) {
    CU(g.d_cut.reserve(B * sizeof(int)), "cudaMalloc(cut)");
    CU(cudaMemcpyAsync(g.d_cut.p, b->cut, B * sizeof(int), cudaMemcpyHostToDevice, st), "H2D cut");
    db.cut = (const int32_t *)g.d_cut.p;
  }
  if (b->nopair) {
    CU(g.d_nopair.reserve(B * S), "cudaMalloc(nopair)");
    CU(cudaMemcpyAsync(g.d_nopair.p, b->nopair, B * S, cudaMemcpyHostToDevice, st), "H2D nopair");
    db.nopair = (const uint8_t *)g.d_nopair.p;
  }
  if (b->want & (BF_WANT_EVAL | BF_WANT_DEFECT)) {
    size_t tb = B * (size_t)b->n_targets * S;
    CU(g.d_targets.reserve(tb), "cudaMalloc(targets)");
    CU(cudaMemcpyAsync(g.d_targets.p, b->targets, tb, cudaMemcpyHostToDevice, st), "H2D targets");
    db.targets = (const char *)g.d_targets.p;
    CU(g.d_eval.reserve(B * b->n_targets * sizeof(int)), "cudaMalloc(eval)");
    dr.eval_dcal = (int32_t *)g.d_eval.p;
  }
  if (b->want & BF_WANT_DEFECT) { CU(g.d_defect.reserve(B * sizeof(double)), "cudaMalloc(defect)"); dr.defect = (double *)g.d_defect.p; }
  if (b->want & BF_WANT_BPP) { CU(g.d_bpp.reserve(B * S * S * sizeof(double)), "cudaMalloc(bpp)"); dr.bpp = (double *)g.d_bpp.p; }
  if (b->want & (BF_WANT_MFE | BF_WANT_SS)) { CU(g.d_mfe.reserve(B * sizeof(int)), "cudaMalloc(mfe)"); dr.mfe_dcal = (int32_t *)g.d_mfe.p; }
  if (b->want & BF_WANT_SS) { CU(g.d_ss.reserve(B * (S + 1)), "cudaMalloc(ss)"); dr.mfe_ss = (char *)g.d_ss.p; }
  if (b->want & (BF_WANT_PF | BF_WANT_BPP | BF_WANT_DEFECT)) { CU(g.d_pf.reserve(B * 5 * sizeof(double)), "cudaMalloc(pf)"); dr.pf = (double *)g.d_pf.p; }
  rc = run_device(g.w, &db, &dr, two, st, ov);
  if (rc) return rc;
  if ((b->want & BF_WANT_MFE) && r->mfe_dcal) CU(cudaMemcpyAsync(r->mfe_dcal, dr.mfe_dcal, B * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H mfe");
  if (b->want & BF_WANT_SS) CU(cudaMemcpyAsync(r->mfe_ss, dr.mfe_ss, B * (S + 1), cudaMemcpyDeviceToHost, st), "D2H ss");
  if ((b->want & (BF_WANT_PF | BF_WANT_BPP | BF_WANT_DEFECT)) && r->pf) CU(cudaMemcpyAsync(r->pf, dr.pf, B * 5 * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H pf");
  if (b->want & BF_WANT_EVAL) CU(cudaMemcpyAsync(r->eval_dcal, dr.eval_dcal, B * b->n_targets * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H eval");
  if (b->want & BF_WANT_DEFECT) CU(cudaMemcpyAsync(r->defect, dr.defect, B * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H defect");
  if (b->want & BF_WANT_BPP) CU(cudaMemcpyAsync(r->bpp, dr.bpp, B * S * S * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H bpp");
  CU(cudaStreamSynchronize(st), "bf_score_batch");
  return BF_OK;
}

int bf_second_best(const bf_batch_t *b, int32_t *e1_dcal, int32_t *e2_dcal) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!b || !e1_dcal || !e2_dcal || b->B < 0 || b->stride <= 0 || (b->B && (!b->seq || !b->len))) return fail(BF_ERR_ARG, "bf_second_best: bad argument");
  if (b->stride > 2000) return fail(BF_ERR_ARG, "bf_second_best: stride > 2000 not supported");
  if (b->B == 0) return BF_OK;
  const bool two = any_cut(b, b->cut);
  cudaStream_t st = g.stream;
  const size_t B = b->B, S = b->stride;
  CU(g.d_seq.reserve(B * S), "cudaMalloc(seq)");
  CU(g.d_len.reserve(B * sizeof(int)), "cudaMalloc(len)");
  CU(g.d_mfe.reserve(2 * B * sizeof(int)), "cudaMalloc(second best)");
  CU(cudaMemcpyAsync(g.d_seq.p, b->seq, B * S, cudaMemcpyHostToDevice, st), "H2D seq");
  CU(cudaMemcpyAsync(g.d_len.p, b->len, B * sizeof(int), cudaMemcpyHostToDevice, st), "H2D len");
  BfBatchDev db;
  db.B = b->B; db.stride = b->stride; db.seq = (const char *)g.d_seq.p; db.len = (const int *)g.d_len.p; db.cut = nullptr; db.nopair = nullptr;
  if (two) {
    CU(g.d_cut.reserve(B * sizeof(int)), "cudaMalloc(cut)");
    CU(cudaMemcpyAsync(g.d_cut.p, b->cut, B * sizeof(int), cudaMemcpyHostToDevice, st), "H2D cut");
    db.cut = (const int32_t *)g.d_cut.p;
  }
  if (b->nopair) {
    CU(g.d_nopair.reserve(B * S), "cudaMalloc(nopair)");
    CU(cudaMemcpyAsync(g.d_nopair.p, b->nopair, B * S, cudaMemcpyHostToDevice, st), "H2D nopair");
    db.nopair = (const uint8_t *)g.d_nopair.p;
  }
  const int wstride = b->stride + 2;
  const int grid = std::min(b->B, 2 * g.sm_count);
  CU(g.w.ws_mfe.reserve((size_t)grid * bf_twobest_slot(wstride) * sizeof(int2)), "cudaMalloc(second-best workspace)");
  int *d_e = (int *)g.d_mfe.p;
  CU(bf_launch_twobest(g.dP, db, (int2 *)g.w.ws_mfe.p, wstride, grid, g.w.d_counters + 0, d_e, d_e + B, st, nullptr, two), "launch bf_k_mfe2");
  g.launches++;
  CU(cudaMemcpyAsync(e1_dcal, d_e, B * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H e1");
  CU(cudaMemcpyAsync(e2_dcal, d_e + B, B * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H e2");
  CU(cudaStreamSynchronize(st), "bf_second_best");
  return BF_OK;
}

int bf_sample(const bf_batch_t *b, int32_t n_samples, uint64_t seed, char *ss_out) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!b || !ss_out || n_samples < 1 || b->B < 0 || b->stride <= 0 || (b->B && (!b->seq || !b->len))) return fail(BF_ERR_ARG, "bf_sample: bad argument");
  if (any_cut(b, b->cut)) return fail(BF_ERR_UNAVAILABLE, "bf_sample: single strands only");
  if (b->nopair) return fail(BF_ERR_UNAVAILABLE, "bf_sample: the partition function does not honour hard constraints");
  if (g.force_generic || bf_fill_pf_mode(b->stride) == 0) return fail(BF_ERR_UNAVAILABLE, "bf_sample: stride outside the fill path");
  for (int i = 0; i < b->B; i++)
    if (b->len[i] < 0 || b->len[i] > b->stride) return fail(BF_ERR_ARG, "sequence length exceeds stride");
  if (b->B == 0) return BF_OK;
  cudaStream_t st = g.stream;
  const size_t B = b->B, S = b->stride, out_bytes = B * (size_t)n_samples * (S + 1);
  CU(g.d_seq.reserve(B * S), "cudaMalloc(seq)");
  CU(g.d_len.reserve(B * sizeof(int)), "cudaMalloc(len)");
  CU(g.d_mfe.reserve(B * sizeof(int)), "cudaMalloc(mfe)");
  CU(g.d_pf.reserve(B * 5 * sizeof(double)), "cudaMalloc(pf)");
  CU(g.d_q5.reserve(B * (S + 1) * sizeof(double)), "cudaMalloc(q5)");
  CU(g.d_samples.reserve(out_bytes), "cudaMalloc(samples)");
  CU(cudaMemcpyAsync(g.d_seq.p, b->seq, B * S, cudaMemcpyHostToDevice, st), "H2D seq");
  CU(cudaMemcpyAsync(g.d_len.p, b->len, B * sizeof(int), cudaMemcpyHostToDevice, st), "H2D len");
  // the MFE sets the partition function's scale, as for base-pair probabilities; the fill keeps qm / qm1 for the walk
  bf_batch_t db;
  memset(&db, 0, sizeof(db));
  db.B = b->B; db.stride = b->stride; db.seq = (const char *)g.d_seq.p; db.len = (const int32_t *)g.d_len.p;
  db.want = BF_WANT_MFE | BF_WANT_PF;
  bf_result_t dr;
  memset(&dr, 0, sizeof(dr));
  dr.mfe_dcal = (int32_t *)g.d_mfe.p; dr.pf = (double *)g.d_pf.p;
  int rc = run_device(g.w, &db, &dr, false, st, nullptr, true, true);
  if (rc) return rc;
  BfBatchDev dev;
  dev.B = b->B; dev.stride = b->stride; dev.seq = db.seq; dev.len = db.len; dev.cut = nullptr; dev.nopair = nullptr;
  CU(bf_launch_sample(g.dP, dev, (const double *)g.w.tri_qb.p, (const double *)g.w.qm_seq.p, (const double *)g.w.d_lnscale.p, (double *)g.d_q5.p,
                      n_samples, seed, (char *)g.d_samples.p, g.sm_count, st), "launch bf_k_sample");
  g.launches += 2;
  CU(cudaMemcpyAsync(ss_out, g.d_samples.p, out_bytes, cudaMemcpyDeviceToHost, st), "D2H samples");
  CU(cudaStreamSynchronize(st), "bf_sample");
  return BF_OK;
}

int bf_pair_mfe(const bf_batch_t *b, int32_t *e_pair_out) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!b || !e_pair_out || b->B < 0 || b->stride <= 0 || (b->B && (!b->seq || !b->len))) return fail(BF_ERR_ARG, "bf_pair_mfe: bad argument");
  if (any_cut(b, b->cut)) return fail(BF_ERR_UNAVAILABLE, "bf_pair_mfe: single strands only");
  if (g.force_generic || bf_fill_mfe_mode(b->stride) == 0) return fail(BF_ERR_UNAVAILABLE, "bf_pair_mfe: stride outside the fill path");
  for (int i = 0; i < b->B; i++)
    if (b->len[i] < 0 || b->len[i] > b->stride) return fail(BF_ERR_ARG, "sequence length exceeds stride");
  if (b->B == 0) return BF_OK;
  cudaStream_t st = g.stream;
  const size_t B = b->B, S = b->stride;
  CU(g.d_seq.reserve(B * S), "cudaMalloc(seq)");
  CU(g.d_len.reserve(B * sizeof(int)), "cudaMalloc(len)");
  CU(g.d_mfe.reserve(B * sizeof(int)), "cudaMalloc(mfe)");
  CU(g.d_epair.reserve(B * S * S * sizeof(int)), "cudaMalloc(e_pair)");
  CU(cudaMemcpyAsync(g.d_seq.p, b->seq, B * S, cudaMemcpyHostToDevice, st), "H2D seq");
  CU(cudaMemcpyAsync(g.d_len.p, b->len, B * sizeof(int), cudaMemcpyHostToDevice, st), "H2D len");
  bf_batch_t db;
  memset(&db, 0, sizeof(db));
  db.B = b->B; db.stride = b->stride; db.seq = (const char *)g.d_seq.p; db.len = (const int32_t *)g.d_len.p;
  if (b->nopair) {
    CU(g.d_nopair.reserve(B * S), "cudaMalloc(nopair)");
    CU(cudaMemcpyAsync(g.d_nopair.p, b->nopair, B * S, cudaMemcpyHostToDevice, st), "H2D nopair");
    db.nopair = (const uint8_t *)g.d_nopair.p;
  }
  db.want = BF_WANT_MFE;
  bf_result_t dr;
  memset(&dr, 0, sizeof(dr));
  dr.mfe_dcal = (int32_t *)g.d_mfe.p;
  int rc = run_device(g.w, &db, &dr, false, st);
  if (rc) return rc;
  BfBatchDev dev;
  dev.B = b->B; dev.stride = b->stride; dev.seq = db.seq; dev.len = db.len; dev.cut = nullptr; dev.nopair = db.nopair;
  BfPlan p;
  CU(bf_plan_mfe_out(b->stride, b->B, g.sm_count, &p), "plan bf_k_mfe_out");
  CU(g.w.ws_out.reserve((size_t)p.grid * p.ws * sizeof(int)), "cudaMalloc(outside workspace)");
  CU(bf_launch_mfe_out(p, g.dP, dev, (const int *)g.w.tri_c.p, (const int *)g.w.tri_f.p, (int *)g.w.ws_out.p, (int *)g.d_epair.p,
                       g.w.d_counters + 2, st), "launch bf_k_mfe_out");
  g.launches++;
  CU(cudaMemcpyAsync(e_pair_out, g.d_epair.p, B * S * S * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H e_pair");
  CU(cudaStreamSynchronize(st), "bf_pair_mfe");
  return BF_OK;
}

namespace {
// The accessibility pipeline on a batch already on the device (seq, len, stride): MFE (it sets the scale), PF fill with qm / qm1 kept,
// the outside pass keeping its triangles in g.d_keep, then bf_k_unpaired into d_pu when d_pu is not null.  plan_B: as for run_device.
int unpaired_device(const bf_batch_t *db, int max_u, double *d_pu, cudaStream_t st, int plan_B = 0) {
  const size_t B = db->B, S = db->stride;
  CU(g.d_mfe.reserve(B * sizeof(int)), "cudaMalloc(mfe)");
  CU(g.d_pf.reserve(B * 5 * sizeof(double)), "cudaMalloc(pf)");
  CU(g.d_keep.reserve(B * 3 * bf_tri_slot(db->stride) * sizeof(double)), "cudaMalloc(outside triangles)");
  bf_result_t dr;
  memset(&dr, 0, sizeof(dr));
  dr.mfe_dcal = (int32_t *)g.d_mfe.p; dr.pf = (double *)g.d_pf.p;
  int rc = run_device(g.w, db, &dr, false, st, nullptr, true, true, (double *)g.d_keep.p, plan_B);
  if (rc || !d_pu) return rc;
  const size_t slot = bf_unpaired_ws_bytes(db->stride);
  const size_t ws = std::min<size_t>(std::min<size_t>(B, 8 * (size_t)g.sm_count) * slot, std::max<size_t>(slot, (size_t)1 << 30));
  CU(g.d_upws.reserve(ws), "cudaMalloc(unpaired workspace)");
  CU(cudaMemsetAsync(d_pu, 0, B * S * max_u * sizeof(double), st), "clear pu");
  BfBatchDev dev;
  dev.B = db->B; dev.stride = db->stride; dev.seq = db->seq; dev.len = db->len; dev.cut = nullptr; dev.nopair = nullptr;
  CU(bf_launch_unpaired(g.dP, dev, (const double *)g.w.tri_qb.p, (const double *)g.w.qm_seq.p, (const double *)g.d_keep.p,
                        (const double *)g.w.d_lnscale.p, (double *)g.d_upws.p, ws, max_u, d_pu, g.w.d_counters + 3, g.sm_count, st),
     "launch bf_k_unpaired");
  g.launches++;
  return BF_OK;
}
}  // namespace

int bf_unpaired(const bf_batch_t *b, int32_t max_u, double *pu_out) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!b || !pu_out || b->B < 0 || b->stride <= 0 || (b->B && (!b->seq || !b->len))) return fail(BF_ERR_ARG, "bf_unpaired: bad argument");
  if (max_u < 1 || max_u > b->stride) return fail(BF_ERR_ARG, "bf_unpaired: max_u outside 1 .. stride");
  if (any_cut(b, b->cut)) return fail(BF_ERR_UNAVAILABLE, "bf_unpaired: single strands only");
  if (b->nopair) return fail(BF_ERR_UNAVAILABLE, "bf_unpaired: the partition function does not honour hard constraints");
  if (g.force_generic || bf_fill_pf_mode(b->stride) == 0) return fail(BF_ERR_UNAVAILABLE, "bf_unpaired: stride outside the fill path");
  for (int i = 0; i < b->B; i++)
    if (b->len[i] < 0 || b->len[i] > b->stride) return fail(BF_ERR_ARG, "sequence length exceeds stride");
  if (b->B == 0) return BF_OK;
  cudaStream_t st = g.stream;
  const size_t B = b->B, S = b->stride;
  CU(g.d_seq.reserve(B * S), "cudaMalloc(seq)");
  CU(g.d_len.reserve(B * sizeof(int)), "cudaMalloc(len)");
  CU(g.d_pu.reserve(B * S * max_u * sizeof(double)), "cudaMalloc(pu)");
  CU(cudaMemcpyAsync(g.d_seq.p, b->seq, B * S, cudaMemcpyHostToDevice, st), "H2D seq");
  CU(cudaMemcpyAsync(g.d_len.p, b->len, B * sizeof(int), cudaMemcpyHostToDevice, st), "H2D len");
  bf_batch_t db;
  memset(&db, 0, sizeof(db));
  db.B = b->B; db.stride = b->stride; db.seq = (const char *)g.d_seq.p; db.len = (const int32_t *)g.d_len.p;
  db.want = BF_WANT_MFE | BF_WANT_PF;
  int rc = unpaired_device(&db, max_u, (double *)g.d_pu.p, st);
  if (rc) return rc;
  CU(cudaMemcpyAsync(pu_out, g.d_pu.p, B * S * max_u * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H pu");
  CU(cudaStreamSynchronize(st), "bf_unpaired");
  return BF_OK;
}

namespace {
// The RNAplfold pipeline on host strands s (checked by the caller): leaves the window averages in g.d_pfbpp (want_bpp: n x stride x
// winsize) and g.d_pfpu (want_pu: n x stride x max_u) on the device.
int plfold_device(const bf_strands_t *s, int32_t winsize, int32_t max_u, bool want_bpp, bool want_pu) {
  if (winsize > 2000) return fail(BF_ERR_UNAVAILABLE, "bf_plfold: window longer than 2000 nt");
  if (g.force_generic) return fail(BF_ERR_UNAVAILABLE, "bf_plfold: BF_FORCE_GENERIC");
  const int n = s->n, S = s->stride;
  // windows: strand r has nwin = len - W' + 1 of length W' = min(W, len), global indices win0[r] .. win0[r] + nwin - 1
  std::vector<int> tab(3 * (size_t)n);   // len, win0, wlen
  long long total = 0;
  int wstride = 1;
  for (int r = 0; r < n; r++) {
    const int len = s->len[r], wl = std::min<int>(winsize, len);
    if (total > INT32_MAX - len) return fail(BF_ERR_ARG, "bf_plfold: more than 2^31 windows");
    tab[r] = len; tab[n + r] = (int)total; tab[2 * n + r] = wl;
    total += len > 0 ? len - wl + 1 : 0;
    wstride = std::max(wstride, wl);
  }
  if (bf_fill_pf_mode(wstride) == 0) return fail(BF_ERR_UNAVAILABLE, "bf_plfold: window longer than the PF fill path covers");
  if (n == 0) return BF_OK;
  cudaStream_t st = g.stream;
  const size_t bpp_bytes = (size_t)n * S * winsize * sizeof(double), pu_bytes = (size_t)n * S * max_u * sizeof(double);
  CU(g.d_pfstr.reserve(tab.size() * sizeof(int)), "cudaMalloc(plfold strands)");
  CU(cudaMemcpyAsync(g.d_pfstr.p, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice, st), "H2D plfold strands");
  if (want_bpp) { CU(g.d_pfbpp.reserve(bpp_bytes), "cudaMalloc(plfold bpp)"); CU(cudaMemsetAsync(g.d_pfbpp.p, 0, bpp_bytes, st), "clear plfold bpp"); }
  if (want_pu) { CU(g.d_pfpu.reserve(pu_bytes), "cudaMalloc(plfold pu)"); CU(cudaMemsetAsync(g.d_pfpu.p, 0, pu_bytes, st), "clear plfold pu"); }
  // chunks of consecutive windows within the memory budget: per window the fill's c / fML (ints) and qb / qm / qm1 triangles, the three
  // kept outside triangles, P_u and the sequence
  const size_t per = bf_tri_slot(wstride) * (2 * sizeof(int) + 6 * sizeof(double)) + (size_t)wstride * (1 + (want_pu ? max_u * sizeof(double) : 0));
  const size_t budget = (size_t)std::max(1, bf_opt("BF_PLFOLD_MB", 1024)) << 20;
  const long long cap = std::max<long long>(1, std::min<long long>(1 << 16, (long long)(budget / per)));
  const long long chunk = std::min<long long>(cap, std::max<long long>(total, 1));
  CU(g.d_seq.reserve((size_t)chunk * wstride), "cudaMalloc(seq)");
  CU(g.d_len.reserve((size_t)chunk * sizeof(int)), "cudaMalloc(len)");
  if (want_pu) CU(g.d_pu.reserve((size_t)chunk * wstride * max_u * sizeof(double)), "cudaMalloc(pu)");
  std::vector<char> hseq((size_t)chunk * wstride, 0);
  std::vector<int> hlen((size_t)chunk);
  const int *dstr = (const int *)g.d_pfstr.p;
  int r = 0;
  for (long long w0 = 0; w0 < total; w0 += chunk) {
    const int nw = (int)std::min<long long>(chunk, total - w0);
    while (tab[n + r] + (long long)(tab[r] > 0 ? tab[r] - tab[2 * n + r] + 1 : 0) <= w0) r++;   // strand of window w0
    const int r0 = r;
    int rr = r0;
    for (int k = 0; k < nw; k++) {
      const long long gw = w0 + k;
      while (tab[n + rr] + (long long)(tab[rr] > 0 ? tab[rr] - tab[2 * n + rr] + 1 : 0) <= gw) rr++;
      const int sidx = (int)(gw - tab[n + rr]), wl = tab[2 * n + rr];
      memcpy(&hseq[(size_t)k * wstride], s->seq + (size_t)rr * S + sidx, wl);
      memset(&hseq[(size_t)k * wstride + wl], 0, wstride - wl);
      hlen[k] = wl;
    }
    CU(cudaMemcpyAsync(g.d_seq.p, hseq.data(), (size_t)nw * wstride, cudaMemcpyHostToDevice, st), "H2D windows");
    CU(cudaMemcpyAsync(g.d_len.p, hlen.data(), (size_t)nw * sizeof(int), cudaMemcpyHostToDevice, st), "H2D window lengths");
    bf_batch_t db;
    memset(&db, 0, sizeof(db));
    db.B = nw; db.stride = wstride; db.seq = (const char *)g.d_seq.p; db.len = (const int32_t *)g.d_len.p;
    db.want = BF_WANT_MFE | BF_WANT_PF;
    // planned for the whole call, so that the kernels -- and with them every window's values -- do not depend on the chunking
    int rc = unpaired_device(&db, max_u, want_pu ? (double *)g.d_pu.p : nullptr, st, (int)std::max<long long>(total, 1));
    if (rc) return rc;
    BfPlfoldDev d;
    d.len = dstr; d.win0 = dstr + n; d.wlen = dstr + 2 * n;
    d.stride = S; d.winsize = winsize; d.max_u = max_u;
    d.r0 = r0; d.r1 = rr + 1; d.w0 = w0; d.nw = nw; d.wstride = wstride;
    CU(bf_launch_plfold_avg(d, (const double *)g.w.tri_qb.p, (const double *)g.d_keep.p, want_pu ? (const double *)g.d_pu.p : nullptr,
                            want_bpp ? (double *)g.d_pfbpp.p : nullptr, want_pu ? (double *)g.d_pfpu.p : nullptr, st),
       "launch bf_k_plfold_avg");
    g.launches++;
    // the host staging buffers are rewritten for the next chunk: the copies above must have read them
    CU(cudaStreamSynchronize(st), "bf_plfold chunk");
  }
  return BF_OK;
}
}  // namespace

int bf_plfold(const bf_strands_t *s, int32_t winsize, int32_t max_u, double *bpp_out, double *pu_out) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!s || (!bpp_out && !pu_out) || s->n < 0 || s->stride <= 0 || (s->n && (!s->seq || !s->len))) return fail(BF_ERR_ARG, "bf_plfold: bad argument");
  for (int r = 0; r < s->n; r++)
    if (s->len[r] < 0 || s->len[r] > s->stride) return fail(BF_ERR_ARG, "bf_plfold: strand length exceeds stride");
  if (winsize < 1 || max_u < 1 || max_u > winsize) return fail(BF_ERR_ARG, "bf_plfold: winsize < 1 or max_u outside 1 .. winsize");
  int rc = plfold_device(s, winsize, max_u, bpp_out != nullptr, pu_out != nullptr);
  if (rc || s->n == 0) return rc;
  cudaStream_t st = g.stream;
  const size_t bpp_bytes = (size_t)s->n * s->stride * winsize * sizeof(double), pu_bytes = (size_t)s->n * s->stride * max_u * sizeof(double);
  if (bpp_out) CU(cudaMemcpyAsync(bpp_out, g.d_pfbpp.p, bpp_bytes, cudaMemcpyDeviceToHost, st), "D2H plfold bpp");
  if (pu_out) CU(cudaMemcpyAsync(pu_out, g.d_pfpu.p, pu_bytes, cudaMemcpyDeviceToHost, st), "D2H plfold pu");
  CU(cudaStreamSynchronize(st), "bf_plfold");
  return BF_OK;
}

namespace {
constexpr int kDuplexMaxLen = 2000;                   // per strand, as for the fill path
constexpr int kDuplexMaxStride = 1 << 16;             // bytes per strand row: keeps a structure slot far below the per-launch budget
constexpr long long kDuplexChunk = 1 << 16;           // pairs per launch at most
constexpr size_t kDuplexWsInts = (size_t)64 << 20;    // c tables / HBM rings of one launch: 256 MB
constexpr size_t kDuplexSsBytes = (size_t)256 << 20;  // structures of one launch

int check_strands(const bf_strands_t &s) {
  if (s.n < 0 || s.stride <= 0 || s.stride > kDuplexMaxStride || (s.n && (!s.seq || !s.len))) return fail(BF_ERR_ARG, "bf_duplex: bad strand set");
  for (int k = 0; k < s.n; k++) {
    if (s.len[k] < 0 || s.len[k] > s.stride) return fail(BF_ERR_ARG, "bf_duplex: strand length exceeds stride");
    if (s.len[k] > kDuplexMaxLen) return fail(BF_ERR_ARG, "bf_duplex: strand longer than 2000 nt");
  }
  return BF_OK;
}
}  // namespace

int bf_duplex(const bf_duplex_t *q, int32_t *e_dcal, char *ss_out) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!q || !e_dcal || (q->pairs && q->n_pairs < 0)) return fail(BF_ERR_ARG, "bf_duplex: bad argument");
  int rc = check_strands(q->a);
  if (!rc) rc = check_strands(q->b);
  if (rc) return rc;
  const long long P = q->pairs ? q->n_pairs : (long long)q->a.n * q->b.n;
  if (q->pairs)
    for (long long p = 0; p < P; p++)
      if (q->pairs[2 * p] < 0 || q->pairs[2 * p] >= q->a.n || q->pairs[2 * p + 1] < 0 || q->pairs[2 * p + 1] >= q->b.n)
        return fail(BF_ERR_ARG, "bf_duplex: pair index out of range");
  if (P == 0) return BF_OK;
  const bool want_ss = ss_out != nullptr;
  const int sa = q->a.stride, sb = q->b.stride, ss_stride = sa + sb + 2;
  auto len_of = [&](long long p, int *n1, int *n2) {
    const int ia = q->pairs ? q->pairs[2 * p] : (int)(p / q->b.n), ib = q->pairs ? q->pairs[2 * p + 1] : (int)(p % q->b.n);
    *n1 = q->a.len[ia]; *n2 = q->b.len[ib];
  };
  BfDuplexDev d;
  d.stride_a = sa; d.stride_b = sb; d.nb = q->b.n;
  d.amax = *std::max_element(q->a.len, q->a.len + q->a.n);
  d.bmax = *std::max_element(q->b.len, q->b.len + q->b.n);
  if (q->pairs) {
    d.ring_w = 0;
    for (long long p = 0; p < P; p++) { int n1, n2; len_of(p, &n1, &n2); d.ring_w = std::max(d.ring_w, std::min(n1, n2)); }
  } else {
    d.ring_w = std::min(d.amax, d.bmax);
  }
  const bool gring = bf_duplex_gring(d);
  const size_t ring_slot = bf_duplex_ring_slot(d.ring_w);
  cudaStream_t st = g.stream;
  CU(g.d_dxa.reserve((size_t)q->a.n * sa), "cudaMalloc(duplex a)");
  CU(g.d_dxb.reserve((size_t)q->b.n * sb), "cudaMalloc(duplex b)");
  CU(g.d_dxlen.reserve((size_t)(q->a.n + q->b.n) * sizeof(int)), "cudaMalloc(duplex len)");
  CU(cudaMemcpyAsync(g.d_dxa.p, q->a.seq, (size_t)q->a.n * sa, cudaMemcpyHostToDevice, st), "H2D duplex a");
  CU(cudaMemcpyAsync(g.d_dxb.p, q->b.seq, (size_t)q->b.n * sb, cudaMemcpyHostToDevice, st), "H2D duplex b");
  int *dlen = (int *)g.d_dxlen.p;
  CU(cudaMemcpyAsync(dlen, q->a.len, q->a.n * sizeof(int), cudaMemcpyHostToDevice, st), "H2D duplex len a");
  CU(cudaMemcpyAsync(dlen + q->a.n, q->b.len, q->b.n * sizeof(int), cudaMemcpyHostToDevice, st), "H2D duplex len b");
  d.seq_a = (const char *)g.d_dxa.p; d.seq_b = (const char *)g.d_dxb.p;
  d.len_a = dlen; d.len_b = dlen + q->a.n;
  d.pairs = nullptr;
  if (q->pairs) {
    CU(g.d_dxpairs.reserve((size_t)P * 2 * sizeof(int)), "cudaMalloc(duplex pairs)");
    CU(cudaMemcpyAsync(g.d_dxpairs.p, q->pairs, (size_t)P * 2 * sizeof(int), cudaMemcpyHostToDevice, st), "H2D duplex pairs");
    d.pairs = (const int *)g.d_dxpairs.p;
  }
  // chunks of consecutive pairs whose c tables (structures) or HBM rings fit the workspace budget
  const long long cap = want_ss ? std::min<long long>(kDuplexChunk, (long long)(kDuplexSsBytes / ss_stride)) : kDuplexChunk;
  std::vector<long long> off;
  for (long long p0 = 0; p0 < P;) {
    long long p1 = p0;
    size_t ws = 0, used = 0;   // c-table ints; c tables and rings
    off.clear();
    if (want_ss || gring) {
      while (p1 < P && p1 - p0 < cap) {
        int n1, n2;
        len_of(p1, &n1, &n2);
        const size_t tab = want_ss ? (size_t)n1 * n2 : 0, need = tab + (gring ? ring_slot : 0);
        if (p1 > p0 && used + need > kDuplexWsInts) break;
        if (want_ss) off.push_back((long long)ws);
        ws += tab;
        used += need;
        p1++;
      }
    } else {
      p1 = std::min(P, p0 + cap);
    }
    const int np = (int)(p1 - p0);
    int *ctab = nullptr, *gws = nullptr;
    const long long *doff = nullptr;
    if (want_ss || gring) {
      CU(g.d_dxws.reserve((ws + (gring ? (size_t)np * ring_slot : 0)) * sizeof(int)), "cudaMalloc(duplex workspace)");
      gws = (int *)g.d_dxws.p;
      if (want_ss) {
        ctab = gws + (gring ? (size_t)np * ring_slot : 0);
        CU(g.d_dxoff.reserve(off.size() * sizeof(long long)), "cudaMalloc(duplex offsets)");
        CU(cudaMemcpyAsync(g.d_dxoff.p, off.data(), off.size() * sizeof(long long), cudaMemcpyHostToDevice, st), "H2D duplex offsets");
        doff = (const long long *)g.d_dxoff.p;
      }
    }
    CU(g.d_dxe.reserve((size_t)np * sizeof(int)), "cudaMalloc(duplex energies)");
    if (want_ss) CU(g.d_dxss.reserve((size_t)np * ss_stride), "cudaMalloc(duplex structures)");
    d.p0 = p0; d.np = np;
    CU(bf_launch_duplex(g.dP, d, gring, gws, (int *)g.d_dxe.p, ctab, doff, want_ss ? (char *)g.d_dxss.p : nullptr, ss_stride, st),
       "launch bf_k_duplex");
    g.launches++;
    CU(cudaMemcpyAsync(e_dcal + p0, g.d_dxe.p, (size_t)np * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H duplex energies");
    if (want_ss)
      CU(cudaMemcpyAsync(ss_out + (size_t)p0 * ss_stride, g.d_dxss.p, (size_t)np * ss_stride, cudaMemcpyDeviceToHost, st), "D2H duplex structures");
    p0 = p1;
  }
  CU(cudaStreamSynchronize(st), "bf_duplex");
  return BF_OK;
}

namespace {
constexpr int kInteractMaxSpan = 64;
constexpr long long kInteractSlots = 8 << 20;          // (pair, k1) slots of one launch: 192 MB
constexpr size_t kInteractSsBytes = (size_t)256 << 20;  // structures of one launch

int max_len(const bf_strands_t &s) { return s.n ? *std::max_element(s.len, s.len + s.n) : 0; }

// Accessibility mode acc (-1 none, 0 global, W > 0 window) of strand set s with max_u = span, when it is available
int interact_acc_check(const bf_strands_t &s, int acc, int span) {
  if (acc < -1) return fail(BF_ERR_ARG, "bf_interact: accessibility mode below -1");
  if (acc > 0 && acc < span) return fail(BF_ERR_ARG, "bf_interact: window shorter than max_span");
  if (acc < 0) return BF_OK;
  if (g.force_generic) return fail(BF_ERR_UNAVAILABLE, "bf_interact: accessibility under BF_FORCE_GENERIC");
  const int m = acc == 0 ? max_len(s) : std::min(acc, max_len(s));
  if (acc > 2000 || (m > 0 && bf_fill_pf_mode(m) == 0)) return fail(BF_ERR_UNAVAILABLE, "bf_interact: strand or window longer than the PF fill path covers");
  return BF_OK;
}

// The opening energies of one side on the device, [strand][k-1][u-1], *rows positions x span per strand: P_u from bf_k_unpaired
// (global) or the RNAplfold pipeline (window), turned into ED by bf_k_interact_ed.
int interact_ed(const bf_strands_t &s, int acc, int span, DevBuf &ed, int *rows, cudaStream_t st) {
  const size_t n = s.n;
  const double *pu;
  if (acc == 0) {
    const int S = std::max(1, max_len(s));
    std::vector<char> h(n * S, 0);
    for (size_t r = 0; r < n; r++) memcpy(&h[r * S], s.seq + r * s.stride, s.len[r]);
    CU(g.d_seq.reserve(n * S), "cudaMalloc(seq)");
    CU(g.d_len.reserve(n * sizeof(int)), "cudaMalloc(len)");
    CU(g.d_pu.reserve(n * S * span * sizeof(double)), "cudaMalloc(pu)");
    CU(cudaMemcpyAsync(g.d_seq.p, h.data(), n * S, cudaMemcpyHostToDevice, st), "H2D seq");
    CU(cudaMemcpyAsync(g.d_len.p, s.len, n * sizeof(int), cudaMemcpyHostToDevice, st), "H2D len");
    bf_batch_t db;
    memset(&db, 0, sizeof(db));
    db.B = s.n; db.stride = S; db.seq = (const char *)g.d_seq.p; db.len = (const int32_t *)g.d_len.p;
    db.want = BF_WANT_MFE | BF_WANT_PF;
    int rc = unpaired_device(&db, span, (double *)g.d_pu.p, st);
    if (rc) return rc;
    pu = (const double *)g.d_pu.p;
    *rows = S;
  } else {
    int rc = plfold_device(&s, acc, span, false, true);
    if (rc) return rc;
    pu = (const double *)g.d_pfpu.p;
    *rows = s.stride;
  }
  const size_t cnt = n * *rows * span;
  CU(ed.reserve(cnt * sizeof(double)), "cudaMalloc(opening energies)");
  CU(bf_launch_interact_ed(pu, (double *)ed.p, cnt, g.hP->kT, st), "launch bf_k_interact_ed");
  g.launches++;
  // the host staging vector above goes out of scope
  CU(cudaStreamSynchronize(st), "bf_interact accessibility");
  return BF_OK;
}
}  // namespace

int bf_interact(const bf_interact_t *q, double *e, int32_t *h_dcal, double *ed, int32_t *site, char *ss_out) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!q || !e || (q->pairs && q->n_pairs < 0)) return fail(BF_ERR_ARG, "bf_interact: bad argument");
  int rc = check_strands(q->a);
  if (!rc) rc = check_strands(q->b);
  if (rc) return rc;
  const int span = q->max_span;
  if (span < 1 || span > kInteractMaxSpan) return fail(BF_ERR_ARG, "bf_interact: max_span outside 1 .. 64");
  const long long P = q->pairs ? q->n_pairs : (long long)q->a.n * q->b.n;
  if (q->pairs)
    for (long long p = 0; p < P; p++)
      if (q->pairs[2 * p] < 0 || q->pairs[2 * p] >= q->a.n || q->pairs[2 * p + 1] < 0 || q->pairs[2 * p + 1] >= q->b.n)
        return fail(BF_ERR_ARG, "bf_interact: pair index out of range");
  if ((rc = interact_acc_check(q->a, q->acc_a, span)) || (rc = interact_acc_check(q->b, q->acc_b, span))) return rc;
  if (P == 0) return BF_OK;
  cudaStream_t st = g.stream;
  BfInteractDev d;
  d.span = span;
  d.ed_a = d.ed_b = nullptr;
  d.rows_a = d.rows_b = 0;
  if (q->acc_a >= 0) {
    if ((rc = interact_ed(q->a, q->acc_a, span, g.d_ixeda, &d.rows_a, st))) return rc;
    d.ed_a = (const double *)g.d_ixeda.p;
  }
  if (q->acc_b >= 0) {
    const bool same = q->acc_b == q->acc_a && q->b.n == q->a.n && q->b.stride == q->a.stride && q->b.seq == q->a.seq && q->b.len == q->a.len;
    if (same) {
      d.ed_b = d.ed_a; d.rows_b = d.rows_a;
    } else {
      if ((rc = interact_ed(q->b, q->acc_b, span, g.d_ixedb, &d.rows_b, st))) return rc;
      d.ed_b = (const double *)g.d_ixedb.p;
    }
  }
  const int sa = q->a.stride, sb = q->b.stride, ss_stride = sa + sb + 2;
  CU(g.d_dxa.reserve((size_t)q->a.n * sa), "cudaMalloc(interact a)");
  CU(g.d_dxb.reserve((size_t)q->b.n * sb), "cudaMalloc(interact b)");
  CU(g.d_dxlen.reserve((size_t)(q->a.n + q->b.n) * sizeof(int)), "cudaMalloc(interact len)");
  CU(cudaMemcpyAsync(g.d_dxa.p, q->a.seq, (size_t)q->a.n * sa, cudaMemcpyHostToDevice, st), "H2D interact a");
  CU(cudaMemcpyAsync(g.d_dxb.p, q->b.seq, (size_t)q->b.n * sb, cudaMemcpyHostToDevice, st), "H2D interact b");
  int *dlen = (int *)g.d_dxlen.p;
  CU(cudaMemcpyAsync(dlen, q->a.len, q->a.n * sizeof(int), cudaMemcpyHostToDevice, st), "H2D interact len a");
  CU(cudaMemcpyAsync(dlen + q->a.n, q->b.len, q->b.n * sizeof(int), cudaMemcpyHostToDevice, st), "H2D interact len b");
  d.seq_a = (const char *)g.d_dxa.p; d.seq_b = (const char *)g.d_dxb.p;
  d.stride_a = sa; d.stride_b = sb;
  d.len_a = dlen; d.len_b = dlen + q->a.n;
  d.nb = q->b.n;
  d.amax = std::max(1, max_len(q->a));
  d.bmax = std::max(1, max_len(q->b));
  d.pairs = nullptr;
  if (q->pairs) {
    CU(g.d_dxpairs.reserve((size_t)P * 2 * sizeof(int)), "cudaMalloc(interact pairs)");
    CU(cudaMemcpyAsync(g.d_dxpairs.p, q->pairs, (size_t)P * 2 * sizeof(int), cudaMemcpyHostToDevice, st), "H2D interact pairs");
    d.pairs = (const int *)g.d_dxpairs.p;
  }
  // launches of consecutive pairs whose (pair, k1) slots and structures fit the per-launch budgets
  long long cap = std::min<long long>(1 << 16, kInteractSlots / d.amax);
  if (ss_out) cap = std::min<long long>(cap, (long long)(kInteractSsBytes / ss_stride));
  cap = std::max<long long>(cap, 1);
  const long long np_max = std::min(cap, P);
  CU(g.d_ixslot.reserve((size_t)np_max * d.amax * sizeof(BfInteractSlot)), "cudaMalloc(interact slots)");
  CU(g.d_ixres.reserve((size_t)np_max * (4 * sizeof(double) + sizeof(long long) + 5 * sizeof(int))), "cudaMalloc(interact results)");
  if (ss_out) CU(g.d_dxss.reserve((size_t)np_max * ss_stride), "cudaMalloc(interact structures)");
  BfInteractOut out;
  out.e = (double *)g.d_ixres.p;
  out.ed = out.e + np_max;
  out.rank = (long long *)(out.ed + 2 * np_max);
  out.h = (int *)(out.rank + np_max);
  out.site = out.h + np_max;
  for (long long p0 = 0; p0 < P; p0 += cap) {
    const int np = (int)std::min(cap, P - p0);
    d.p0 = p0; d.np = np;
    d.ia0 = q->pairs ? 0 : (int)(p0 / d.nb);
    d.ib0 = q->pairs ? 0 : (int)(p0 % d.nb);
    CU(bf_launch_interact(g.dP, d, (BfInteractSlot *)g.d_ixslot.p, out, ss_out ? (char *)g.d_dxss.p : nullptr, ss_stride,
                          g.w.d_counters + 4, g.sm_count, st),
       "launch bf_k_interact");
    g.launches += ss_out ? 3 : 2;
    CU(cudaMemcpyAsync(e + p0, out.e, (size_t)np * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H interact energies");
    if (h_dcal) CU(cudaMemcpyAsync(h_dcal + p0, out.h, (size_t)np * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H interact H");
    if (ed) CU(cudaMemcpyAsync(ed + 2 * p0, out.ed, (size_t)np * 2 * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H interact ED");
    if (site) CU(cudaMemcpyAsync(site + 4 * p0, out.site, (size_t)np * 4 * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H interact sites");
    if (ss_out)
      CU(cudaMemcpyAsync(ss_out + (size_t)p0 * ss_stride, g.d_dxss.p, (size_t)np * ss_stride, cudaMemcpyDeviceToHost, st), "D2H interact structures");
  }
  CU(cudaStreamSynchronize(st), "bf_interact");
  return BF_OK;
}

namespace {
// pair table of dot-bracket db (n chars) into pt[0 .. n+1]; false when it is not a balanced '.', '(', ')' string with j - i >= 4
bool findpath_parse(const char *db, int n, short *pt, std::vector<int> &stk) {
  stk.clear();
  for (int i = 0; i <= n + 1; i++) pt[i] = 0;
  for (int i = 1; i <= n; i++) {
    const char c = db[i - 1];
    if (c == '(') stk.push_back(i);
    else if (c == ')') {
      if (stk.empty()) return false;
      const int o = stk.back();
      stk.pop_back();
      if (i - o < 4) return false;
      pt[o] = (short)i; pt[i] = (short)o;
    } else if (c != '.') return false;
  }
  return stk.empty();
}
}  // namespace

int bf_findpath(const bf_findpath_t *q, int32_t *saddle_dcal, int32_t *n_moves, int32_t *moves, int32_t *path_e) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!q || !saddle_dcal || q->n < 0 || q->stride < 1) return fail(BF_ERR_ARG, "bf_findpath: bad argument");
  if (q->stride > BF_FINDPATH_MAX_LEN) return fail(BF_ERR_ARG, "bf_findpath: stride above 2000");
  if (q->width < 1 || q->width > BF_FINDPATH_MAX_WIDTH) return fail(BF_ERR_ARG, "bf_findpath: width outside 1 .. 1024");
  const int n = q->n, S = q->stride;
  if (n && (!q->seq || !q->len || !q->s1 || !q->s2)) return fail(BF_ERR_ARG, "bf_findpath: null sequence or structure buffer");
  // pair tables, move lists (pairs of s1 only, ascending i, then pairs of s2 only) and their counts
  std::vector<short> pt((size_t)n * 2 * (S + 2));
  std::vector<int> mv((size_t)n * S, 0), nd((size_t)n * 2), stk;
  int nmax = 1, kmax = 0;
  for (int r = 0; r < n; r++) {
    const int len = q->len[r];
    if (len < 0 || len > S) return fail(BF_ERR_ARG, "bf_findpath: length outside 0 .. stride");
    for (int i = 0; i < len; i++)
      if (!bf_base_code(q->seq[(size_t)r * S + i])) return fail(BF_ERR_ARG, "bf_findpath: sequence character other than ACGUT");
    short *p1 = &pt[(size_t)r * 2 * (S + 2)], *p2 = p1 + S + 2;
    if (!findpath_parse(q->s1 + (size_t)r * S, len, p1, stk) || !findpath_parse(q->s2 + (size_t)r * S, len, p2, stk))
      return fail(BF_ERR_ARG, "bf_findpath: structure not balanced, a character other than '.()', or a pair with j - i < 4");
    int *m = &mv[(size_t)r * S], k = 0;
    for (int i = 1; i <= len; i++) if (p1[i] > i && p2[i] != p1[i]) m[k++] = i << 16 | p1[i];
    nd[2 * r] = k;
    for (int i = 1; i <= len; i++) if (p2[i] > i && p1[i] != p2[i]) m[k++] = i << 16 | p2[i];
    nd[2 * r + 1] = k - nd[2 * r];
    nmax = std::max(nmax, len);
    kmax = std::max(kmax, k);
    if (n_moves) n_moves[r] = k;
  }
  if (n == 0) return BF_OK;
  cudaStream_t st = g.stream;
  const int W = q->width, R = bf_findpath_runs(W), kw = std::max(1, (kmax + 63) / 64);
  // per-instance pair tables are interleaved (s1, s2); the kernel reads them through two pointers with a stride of two tables
  std::vector<short> pt1((size_t)n * (S + 2)), pt2((size_t)n * (S + 2));
  for (int r = 0; r < n; r++) {
    memcpy(&pt1[(size_t)r * (S + 2)], &pt[(size_t)r * 2 * (S + 2)], (S + 2) * sizeof(short));
    memcpy(&pt2[(size_t)r * (S + 2)], &pt[(size_t)r * 2 * (S + 2) + S + 2], (S + 2) * sizeof(short));
  }
  const size_t ptb = (size_t)n * (S + 2) * sizeof(short);
  CU(g.d_fpseq.reserve((size_t)n * S), "cudaMalloc(findpath seq)");
  CU(g.d_fplen.reserve((size_t)n * sizeof(int)), "cudaMalloc(findpath len)");
  CU(g.d_fppt.reserve(2 * ptb), "cudaMalloc(findpath pair tables)");
  CU(g.d_fpmv.reserve((size_t)n * S * sizeof(int)), "cudaMalloc(findpath moves)");
  CU(g.d_fpnd.reserve((size_t)n * 2 * sizeof(int)), "cudaMalloc(findpath counts)");
  CU(cudaMemcpyAsync(g.d_fpseq.p, q->seq, (size_t)n * S, cudaMemcpyHostToDevice, st), "H2D findpath seq");
  CU(cudaMemcpyAsync(g.d_fplen.p, q->len, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, st), "H2D findpath len");
  CU(cudaMemcpyAsync(g.d_fppt.p, pt1.data(), ptb, cudaMemcpyHostToDevice, st), "H2D findpath s1");
  CU(cudaMemcpyAsync((char *)g.d_fppt.p + ptb, pt2.data(), ptb, cudaMemcpyHostToDevice, st), "H2D findpath s2");
  CU(cudaMemcpyAsync(g.d_fpmv.p, mv.data(), (size_t)n * S * sizeof(int), cudaMemcpyHostToDevice, st), "H2D findpath move lists");
  CU(cudaMemcpyAsync(g.d_fpnd.p, nd.data(), (size_t)n * 2 * sizeof(int), cudaMemcpyHostToDevice, st), "H2D findpath counts");
  // within a memory budget: the grid's per-CTA workspaces (shaped by the whole call, so that the kernel's work does not depend on the
  // split) and the back-pointers of the instances of one launch
  const size_t budget = (size_t)std::max(1, bf_opt("BF_FINDPATH_MB", 1024)) << 20;
  const long long cap = bf_findpath_cap(W, kmax);
  const size_t ws_cta = bf_findpath_ws_bytes(W, nmax, kw, cap);
  const int grid_max = (int)std::max<long long>(1, std::min<long long>((long long)g.sm_count * bf_findpath_occupancy(), (long long)(budget / ws_cta)));
  const long long wsum = bf_findpath_width_sum(W);
  std::vector<long long> off((size_t)n + 1, 0);
  for (int r = 0; r < n; r++) off[r + 1] = off[r] + (long long)(nd[2 * r] + nd[2 * r + 1]) * wsum;
  // launches of consecutive instances whose back-pointers fit the budget (at least one instance each)
  std::vector<int> cut{0};
  for (int r = 1; r < n; r++)
    if ((size_t)(off[r + 1] - off[cut.back()]) * sizeof(int2) > budget) cut.push_back(r);
  cut.push_back(n);
  long long bp_max = 0;
  int n_max = 0;
  for (size_t c = 0; c + 1 < cut.size(); c++) {
    bp_max = std::max(bp_max, off[cut[c + 1]] - off[cut[c]]);
    n_max = std::max(n_max, cut[c + 1] - cut[c]);
  }
  CU(g.d_fpoff.reserve((size_t)n * sizeof(long long)), "cudaMalloc(findpath offsets)");
  CU(g.d_fpws.reserve((size_t)grid_max * ws_cta), "cudaMalloc(findpath workspaces)");
  CU(g.d_fpbp.reserve((size_t)std::max<long long>(bp_max, 1) * sizeof(int2)), "cudaMalloc(findpath back-pointers)");
  CU(g.d_fprun.reserve((size_t)n_max * R * 2 * sizeof(int)), "cudaMalloc(findpath runs)");
  CU(g.d_fpout.reserve((size_t)n_max * (1 + 2 * S + S + 1) * sizeof(int)), "cudaMalloc(findpath results)");
  std::vector<long long> loff((size_t)n);
  for (size_t c = 0; c + 1 < cut.size(); c++)
    for (int r = cut[c]; r < cut[c + 1]; r++) loff[r] = off[r] - off[cut[c]];
  CU(cudaMemcpyAsync(g.d_fpoff.p, loff.data(), (size_t)n * sizeof(long long), cudaMemcpyHostToDevice, st), "H2D findpath offsets");
  int *o_sad = (int *)g.d_fpout.p, *o_mv = o_sad + n_max, *o_pe = o_mv + (size_t)n_max * 2 * S;
  for (size_t c = 0; c + 1 < cut.size(); c++) {
    const int r0 = cut[c], nl = cut[c + 1] - r0;
    BfFindpathDev d;
    d.n = nl; d.stride = S;
    d.seq = (const char *)g.d_fpseq.p + (size_t)r0 * S;
    d.len = (const int *)g.d_fplen.p + r0;
    d.pt1 = (const short *)g.d_fppt.p + (size_t)r0 * (S + 2);
    d.pt2 = (const short *)((const char *)g.d_fppt.p + ptb) + (size_t)r0 * (S + 2);
    d.mv = (const int *)g.d_fpmv.p + (size_t)r0 * S;
    d.nd = (const int *)g.d_fpnd.p + 2 * r0;
    d.width = W; d.nmax = nmax; d.kw = kw; d.cap = cap;
    d.bp = (int2 *)g.d_fpbp.p;
    d.bp_off = (const long long *)g.d_fpoff.p + r0;
    d.run_sad = (int *)g.d_fprun.p; d.run_e0 = d.run_sad + (size_t)n_max * R;
    const int grid = (int)std::min<long long>(grid_max, (long long)nl * R);
    if (moves) CU(cudaMemsetAsync(o_mv, 0, (size_t)nl * 2 * S * sizeof(int), st), "clear findpath moves");
    if (path_e) CU(cudaMemsetAsync(o_pe, 0, (size_t)nl * (S + 1) * sizeof(int), st), "clear findpath energies");
    CU(bf_launch_findpath(g.dP, d, (unsigned char *)g.d_fpws.p, grid, g.w.d_counters + 5, o_sad, moves ? o_mv : nullptr, path_e ? o_pe : nullptr, st),
       "launch bf_k_findpath");
    g.launches += 2;
    CU(cudaMemcpyAsync(saddle_dcal + r0, o_sad, (size_t)nl * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H findpath saddles");
    if (moves) CU(cudaMemcpyAsync(moves + (size_t)r0 * 2 * S, o_mv, (size_t)nl * 2 * S * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H findpath moves");
    if (path_e) CU(cudaMemcpyAsync(path_e + (size_t)r0 * (S + 1), o_pe, (size_t)nl * (S + 1) * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H findpath energies");
  }
  CU(cudaStreamSynchronize(st), "bf_findpath");
  return BF_OK;
}

int bf_kinfold(const bf_kinfold_t *q, int32_t *status, double *t_end, int64_t *steps, int32_t *e_end, char *ss_end, int32_t *e_snap,
               char *ss_snap) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!q || !status || q->n < 0 || q->n_traj < 1 || q->stride < 1) return fail(BF_ERR_ARG, "bf_kinfold: bad argument");
  if (q->stride > BF_KINFOLD_MAX_LEN) return fail(BF_ERR_ARG, "bf_kinfold: stride above 2000");
  if (q->rule < 0 || q->rule > 2) return fail(BF_ERR_ARG, "bf_kinfold: rule outside 0 .. 2");
  if (q->max_steps < 1) return fail(BF_ERR_ARG, "bf_kinfold: max_steps below 1");
  if (q->n_snap < 0) return fail(BF_ERR_ARG, "bf_kinfold: n_snap below 0");
  const bool timed = q->rule != 2;
  if (timed && !(std::isfinite(q->t_max) && q->t_max > 0)) return fail(BF_ERR_ARG, "bf_kinfold: t_max not finite and positive");
  if (timed && q->n_snap > 0) {
    if (!q->t_snap) return fail(BF_ERR_ARG, "bf_kinfold: null snapshot times");
    for (int s = 0; s < q->n_snap; s++)
      if (!(q->t_snap[s] >= 0 && q->t_snap[s] <= q->t_max) || (s && q->t_snap[s] < q->t_snap[s - 1]))
        return fail(BF_ERR_ARG, "bf_kinfold: snapshot times not ascending in [0, t_max]");
  }
  const int n = q->n, S = q->stride, T = q->n_traj, ns = q->n_snap;
  if (n && (!q->seq || !q->len)) return fail(BF_ERR_ARG, "bf_kinfold: null sequence buffer");
  // start and stop pair tables; every pair canonical.  gmax: the most groups of 32 valid moves any step can have (every move is a
  // canonical pair with j - i >= 4)
  std::vector<short> pt((size_t)n * 2 * (S + 2), 0);
  std::vector<int> stk;
  std::vector<uint8_t> code(S + 2);
  int nmax = 1;
  long long npmax = 1;
  for (int r = 0; r < n; r++) {
    const int len = q->len[r];
    const char *seq = q->seq + (size_t)r * S;
    if (len < 0 || len > S) return fail(BF_ERR_ARG, "bf_kinfold: length outside 0 .. stride");
    for (int i = 1; i <= len; i++)
      if (!(code[i] = (uint8_t)bf_base_code(seq[i - 1]))) return fail(BF_ERR_ARG, "bf_kinfold: sequence character other than ACGUT");
    for (int w = 0; w < 2; w++) {
      const char *db = w ? q->stop : q->start;
      if (!db) continue;
      short *p = &pt[((size_t)r * 2 + w) * (S + 2)];
      if (!findpath_parse(db + (size_t)r * S, len, p, stk))
        return fail(BF_ERR_ARG, "bf_kinfold: structure not balanced, a character other than '.()', or a pair with j - i < 4");
      for (int i = 1; i <= len; i++)
        if (p[i] > i && !bf_ptype_bases(code[i], code[p[i]])) return fail(BF_ERR_ARG, "bf_kinfold: a non-canonical pair");
    }
    // canonical partners j >= i + 4 of every i, from counts of each base at and after i + 4
    long long np = 0, cnt[5] = {0, 0, 0, 0, 0};
    for (int i = len - 4; i >= 1; i--) {
      cnt[code[i + 4]]++;
      for (int b = 1; b <= 4; b++) np += bf_ptype_bases(code[i], b) ? cnt[b] : 0;
    }
    nmax = std::max(nmax, len);
    npmax = std::max(npmax, np);
  }
  if (n == 0) return BF_OK;
  cudaStream_t st = g.stream;
  std::vector<short> pts((size_t)n * 2 * (S + 2));   // all start tables, then all stop tables
  for (int r = 0; r < n; r++)
    for (int w = 0; w < 2; w++)
      memcpy(&pts[((size_t)w * n + r) * (S + 2)], &pt[((size_t)r * 2 + w) * (S + 2)], (S + 2) * sizeof(short));
  std::vector<double> rate(65536);
  const double kT = g.hP->kT;
  for (int x = 0; x < 65536; x++) {
    const double de = (double)(x - 32768);
    rate[x] = q->rule == 0 ? std::exp(-de * 10.0 / (2.0 * kT)) : std::min(1.0, std::exp(-de * 10.0 / kT));
  }
  const size_t ptb = (size_t)n * (S + 2) * sizeof(short);
  CU(g.d_kfseq.reserve((size_t)n * S), "cudaMalloc(kinfold seq)");
  CU(g.d_kflen.reserve((size_t)n * sizeof(int)), "cudaMalloc(kinfold len)");
  CU(g.d_kfpt.reserve(2 * ptb), "cudaMalloc(kinfold pair tables)");
  CU(g.d_kfrate.reserve(65536 * sizeof(double)), "cudaMalloc(kinfold rates)");
  CU(g.d_kfsnap.reserve((size_t)std::max(ns, 1) * sizeof(double)), "cudaMalloc(kinfold snapshot times)");
  CU(cudaMemcpyAsync(g.d_kfseq.p, q->seq, (size_t)n * S, cudaMemcpyHostToDevice, st), "H2D kinfold seq");
  CU(cudaMemcpyAsync(g.d_kflen.p, q->len, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, st), "H2D kinfold len");
  CU(cudaMemcpyAsync(g.d_kfpt.p, pts.data(), 2 * ptb, cudaMemcpyHostToDevice, st), "H2D kinfold pair tables");
  CU(cudaMemcpyAsync(g.d_kfrate.p, rate.data(), 65536 * sizeof(double), cudaMemcpyHostToDevice, st), "H2D kinfold rates");
  if (timed && ns) CU(cudaMemcpyAsync(g.d_kfsnap.p, q->t_snap, (size_t)ns * sizeof(double), cudaMemcpyHostToDevice, st), "H2D kinfold snapshot times");
  // half the budget for the grid's workspaces, half for the outputs of one launch
  const size_t budget = (size_t)std::max(1, bf_opt("BF_KINFOLD_MB", 1024)) << 20;
  const int gmax = timed ? (int)((npmax + 31) / 32) : 1;
  const size_t ws_cta = bf_kinfold_ws_bytes(gmax, nmax);
  const int occ = bf_kinfold_occupancy(nmax);
  const int grid_max = (int)std::max<long long>(1, std::min<long long>((long long)g.sm_count * occ, (long long)(budget / 2 / ws_cta)));
  const size_t per_u = 2 * sizeof(double) + 2 * sizeof(int) + (S + 1) + (size_t)ns * (sizeof(int) + S + 1);
  const long long units = (long long)n * T;
  const long long nl_max = std::min<long long>(units, std::max<long long>(1, (long long)(budget / 2 / per_u)));
  CU(g.d_kfws.reserve((size_t)grid_max * ws_cta), "cudaMalloc(kinfold workspaces)");
  CU(g.d_kfout.reserve((size_t)nl_max * per_u + 1024), "cudaMalloc(kinfold results)");
  char *ob = (char *)g.d_kfout.p;
  double *o_t = (double *)ob;
  long long *o_steps = (long long *)(o_t + nl_max);
  int *o_status = (int *)(o_steps + nl_max), *o_e = o_status + nl_max, *o_esnap = o_e + nl_max;
  char *o_ss = (char *)(o_esnap + (size_t)nl_max * ns), *o_sssnap = o_ss + (size_t)nl_max * (S + 1);
  for (long long u0 = 0; u0 < units; u0 += nl_max) {
    const int nl = (int)std::min<long long>(nl_max, units - u0);
    BfKinfoldDev d;
    d.stride = S; d.T = T;
    d.seq = (const char *)g.d_kfseq.p;
    d.len = (const int *)g.d_kflen.p;
    d.start = (const short *)g.d_kfpt.p;
    d.stop = q->stop ? (const short *)((const char *)g.d_kfpt.p + ptb) : nullptr;
    d.rate = (const double *)g.d_kfrate.p;
    d.rule = q->rule; d.t_max = q->t_max; d.seed = q->seed; d.max_steps = q->max_steps;
    d.n_snap = ns; d.t_snap = (const double *)g.d_kfsnap.p;
    d.u0 = u0; d.nu = nl; d.nmax = nmax; d.gmax = gmax;
    d.status = o_status; d.t_end = o_t; d.steps = o_steps; d.e_end = o_e; d.ss_end = o_ss; d.e_snap = o_esnap; d.ss_snap = o_sssnap;
    const int grid = (int)std::min<long long>(grid_max, (nl + 7) / 8);
    CU(bf_launch_kinfold(g.dP, d, (unsigned char *)g.d_kfws.p, grid, g.w.d_counters + 6, st), "launch bf_k_kinfold");
    g.launches++;
    CU(cudaMemcpyAsync(status + u0, o_status, (size_t)nl * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H kinfold status");
    if (t_end) CU(cudaMemcpyAsync(t_end + u0, o_t, (size_t)nl * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H kinfold times");
    if (steps) CU(cudaMemcpyAsync(steps + u0, o_steps, (size_t)nl * sizeof(long long), cudaMemcpyDeviceToHost, st), "D2H kinfold steps");
    if (e_end) CU(cudaMemcpyAsync(e_end + u0, o_e, (size_t)nl * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H kinfold energies");
    if (ss_end) CU(cudaMemcpyAsync(ss_end + u0 * (S + 1), o_ss, (size_t)nl * (S + 1), cudaMemcpyDeviceToHost, st), "D2H kinfold structures");
    if (e_snap && ns)
      CU(cudaMemcpyAsync(e_snap + u0 * ns, o_esnap, (size_t)nl * ns * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H kinfold snapshot energies");
    if (ss_snap && ns)
      CU(cudaMemcpyAsync(ss_snap + u0 * ns * (S + 1), o_sssnap, (size_t)nl * ns * (S + 1), cudaMemcpyDeviceToHost, st),
         "D2H kinfold snapshot structures");
  }
  CU(cudaStreamSynchronize(st), "bf_kinfold");
  return BF_OK;
}

int bf_subopt_zuker(const char *seq, int32_t len, const uint8_t *nopair, int32_t max_out, char *ss_out, int32_t *e_out, int32_t *n_out,
                    int32_t *truncated) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!seq || len <= 0 || !ss_out || !e_out || !n_out || max_out <= 0) return fail(BF_ERR_ARG, "bf_subopt_zuker: bad argument");
  if (g.force_generic || bf_fill_mfe_mode(len) == 0) return fail(BF_ERR_UNAVAILABLE, "bf_subopt_zuker: length outside the fill path");
  // E_pair of this one sequence; its MFE fill leaves the c / fML tables in the engine's table buffers
  int32_t l32 = len;
  bf_batch_t b;
  memset(&b, 0, sizeof(b));
  b.B = 1; b.stride = len; b.seq = seq; b.len = &l32; b.nopair = nopair;
  std::vector<int> ep((size_t)len * len);
  int rc = bf_pair_mfe(&b, ep.data());
  if (rc) return rc;
  const size_t slot = bf_tri_slot(len);
  std::vector<int> c(slot), fm(slot);
  CU(cudaMemcpy(c.data(), g.w.tri_c.p, slot * sizeof(int), cudaMemcpyDeviceToHost), "D2H c table");
  CU(cudaMemcpy(fm.data(), g.w.tri_f.p, slot * sizeof(int), cudaMemcpyDeviceToHost), "D2H fML table");
  std::vector<uint8_t> S(len + 2, 0), SP(len + 2, 0);
  for (int k = 1; k <= len; k++) {
    S[k] = (uint8_t)bf_base_code(seq[k - 1]);
    SP[k] = (nopair && nopair[k - 1]) ? 0 : S[k];
  }
  std::vector<std::pair<int, std::string>> out;
  bool trunc = false;
  if (bf_zuker_host(g.hP, len, S.data(), SP.data(), c.data(), fm.data(), ep.data(), max_out, &out, &trunc) < 0)
    return fail(BF_ERR_CUDA, "bf_subopt_zuker: E_pair disagrees with the MFE fill's tables");
  for (size_t k = 0; k < out.size(); k++) {
    e_out[k] = out[k].first;
    memcpy(ss_out + k * (size_t)(len + 1), out[k].second.c_str(), (size_t)len + 1);
  }
  *n_out = (int32_t)out.size();
  if (truncated) *truncated = trunc ? 1 : 0;
  return BF_OK;
}

int bf_subopt(const char *seq, int32_t len, const uint8_t *nopair, int32_t delta_dcal, int32_t max_out, char *ss_out, int32_t *e_out,
              int32_t *n_out, int32_t *truncated) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!seq || len <= 0 || !ss_out || !e_out || !n_out || max_out <= 0 || delta_dcal < 0) return fail(BF_ERR_ARG, "bf_subopt: bad argument");
  if (g.force_generic || bf_fill_mfe_mode(len) == 0) return fail(BF_ERR_UNAVAILABLE, "bf_subopt: length outside the fill path");
  // the MFE fill of this one sequence leaves its c / fML tables in the engine's table buffers
  int32_t l32 = len, mfe = 0;
  bf_batch_t b;
  memset(&b, 0, sizeof(b));
  b.B = 1; b.stride = len; b.seq = seq; b.len = &l32; b.nopair = nopair; b.want = BF_WANT_MFE;
  bf_result_t r;
  memset(&r, 0, sizeof(r));
  r.mfe_dcal = &mfe;
  int rc = bf_score_batch(&b, &r);
  if (rc) return rc;
  const size_t slot = bf_tri_slot(len);
  std::vector<int> c(slot), fm(slot);
  CU(cudaMemcpy(c.data(), g.w.tri_c.p, slot * sizeof(int), cudaMemcpyDeviceToHost), "D2H c table");
  CU(cudaMemcpy(fm.data(), g.w.tri_f.p, slot * sizeof(int), cudaMemcpyDeviceToHost), "D2H fML table");
  std::vector<uint8_t> S(len + 2, 0), SP(len + 2, 0);
  for (int k = 1; k <= len; k++) {
    S[k] = (uint8_t)bf_base_code(seq[k - 1]);
    SP[k] = (nopair && nopair[k - 1]) ? 0 : S[k];
  }
  std::vector<std::pair<int, std::string>> out;
  int mfe_host = 0;
  bool trunc = false;
  bf_wuchty_host(g.hP, len, S.data(), SP.data(), c.data(), fm.data(), delta_dcal, max_out, &out, &mfe_host, &trunc);
  if (mfe_host != mfe) return fail(BF_ERR_CUDA, "bf_subopt: host exterior pass disagrees with the device MFE");
  for (size_t k = 0; k < out.size(); k++) {
    e_out[k] = out[k].first;
    memcpy(ss_out + k * (size_t)(len + 1), out[k].second.c_str(), (size_t)len + 1);
  }
  *n_out = (int32_t)out.size();
  if (truncated) *truncated = trunc ? 1 : 0;
  return BF_OK;
}

int bf_last_kernel_ms(double out[3]) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  for (int k = 0; k < 3; k++) {
    out[k] = -1.0;
    if (!g.w.ran[k]) continue;
    CU(cudaEventSynchronize(g.w.ev[2 * k + 1]), "cudaEventSynchronize");
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, g.w.ev[2 * k], g.w.ev[2 * k + 1]), "cudaEventElapsedTime");
    out[k] = ms;
  }
  return BF_OK;
}

int bf_set_option(const char *key, int value) {
  // key "cl" -> BF_CL, "cl_c" -> BF_CL_C, ...: one of kOptions.  A negative value removes the variable (back to the default rule).
  if (!key || !*key) return fail(BF_ERR_ARG, "null option key");
  std::string name = "BF_";
  for (const char *p = key; *p; p++) {
    const char ch = *p;
    if (!((ch >= 'a' && ch <= 'z') || (ch >= 'A' && ch <= 'Z') || (ch >= '0' && ch <= '9') || ch == '_')) return fail(BF_ERR_ARG, std::string("bad option key: ") + key);
    name += (char)((ch >= 'a' && ch <= 'z') ? ch - 'a' + 'A' : ch);
  }
  if (std::find(std::begin(kOptions), std::end(kOptions), name) == std::end(kOptions)) return fail(BF_ERR_ARG, std::string("unknown option: ") + key);
  if (value < 0) unsetenv(name.c_str());
  else setenv(name.c_str(), std::to_string(value).c_str(), 1);
  return BF_OK;
}

int bf_debug_copy_table(int which, int32_t n_seq, void *host, size_t host_bytes, size_t *slot_entries) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (which < 0 || which > 2) return fail(BF_ERR_ARG, "which must be 0 (c), 1 (fML) or 2 (qb)");
  const size_t slot = bf_tri_slot(g.last_stride);
  if (slot_entries) *slot_entries = slot;
  if (!host) return BF_OK;
  DevBuf &t = which == 0 ? g.w.tri_c : which == 1 ? g.w.tri_f : g.w.tri_qb;
  const size_t bytes = (size_t)n_seq * slot * (which == 2 ? sizeof(double) : sizeof(int));
  if (bytes > host_bytes || bytes > t.cap) return fail(BF_ERR_ARG, "table copy larger than the host buffer or the table");
  CU(cudaDeviceSynchronize(), "cudaDeviceSynchronize");
  CU(cudaMemcpy(host, t.p, bytes, cudaMemcpyDeviceToHost), "D2H table");
  return BF_OK;
}

int64_t bf_kernel_launches(void) { return g.launches; }
int bf_sm_count(void) { return g.sm_count; }

// =====================================================================================================
//                      device-resident Replica-Exchange Monte-Carlo design loop
// =====================================================================================================
}  // extern "C"

namespace {
struct DesignLoop {
  Workspace w;
  cudaStream_t st = nullptr;
  BfDesignDev D;
  BfDesignCfg C;
  int B = 0, gstep = 0, re_attempt = 0;
  uint32_t want = 0;
  bool two = false;   // some job has two strands: the loop folds with the two-strand kernels
  bool pks = false;   // pseudoknot overlay: three constrained refolds after the MFE fold of every sub-step
  bool overlap = true;  // BF_DESIGN_OVERLAP=0: always fold MFE, then PF
  // avoid designs (oligo 3): the self-dimer fold runs on a stream of its own beside the single-strand fills.  It needs its own
  // workspace: run_device takes the work counters and ws_pf from the workspace it is given
  Workspace wd;
  cudaStream_t st_dimer = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  std::vector<void *> allocs;
  std::vector<uint8_t> active;
  uint8_t *d_active = nullptr;
  int *d_rowmap = nullptr;
  template <typename T>
  cudaError_t alloc(T **p, size_t n) {
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) { allocs.push_back(q); e = cudaMemset(q, 0, std::max<size_t>(n, 1) * sizeof(T)); }
    *p = (T *)q;
    return e;
  }
  void destroy() {
    if (st) cudaStreamSynchronize(st);
    if (st_dimer) cudaStreamSynchronize(st_dimer);
    for (void *q : allocs) cudaFree(q);
    allocs.clear();
    w.destroy();
    wd.destroy();
    if (ev_fork) cudaEventDestroy(ev_fork);
    if (ev_join) cudaEventDestroy(ev_join);
    if (st) cudaStreamDestroy(st);
    if (st_dimer) cudaStreamDestroy(st_dimer);
    st = st_dimer = nullptr;
    ev_fork = ev_join = nullptr;
  }
};

int design_rows(DesignLoop *h) {
  // batch rows = the replicas of the active jobs, job-major
  std::vector<int> rows;
  for (int j = 0; j < h->D.J; j++)
    if (h->active[j])
      for (int r = 0; r < h->D.R; r++) rows.push_back(j * h->D.R + r);
  h->B = (int)rows.size();
  if (h->B) CU(cudaMemcpyAsync(h->d_rowmap, rows.data(), rows.size() * sizeof(int), cudaMemcpyHostToDevice, h->st), "H2D row map");
  CU(cudaMemcpyAsync(h->d_active, h->active.data(), h->active.size(), cudaMemcpyHostToDevice, h->st), "H2D active jobs");
  CU(cudaStreamSynchronize(h->st), "design row map");   // `rows` is a temporary
  CU(bf_launch_design_gather(h->D, h->B, h->st), "launch bf_k_design_gather");
  g.launches++;
  return BF_OK;
}

// one scoring pass over the rows: the same pipeline bf_score_batch_device runs (MFE fill + backtrack, PF fill + exterior, eval)
int design_score(DesignLoop *h, bool init = false) {
  if (h->C.oligo == 3) {
    // avoid: two-strand partition function of the self-dimers (bf_k_design_propose wrote them), forked after propose.  PF only and
    // no scale override: ViennaRNA's default scale, as the host's fc.pf_dimer() of seq&seq.  Joined before the accept kernel.
    bf_batch_t bd;
    std::memset(&bd, 0, sizeof bd);
    bd.B = h->B; bd.stride = 2 * h->D.stride; bd.seq = h->D.dimer_seq; bd.len = h->D.dimer_len; bd.cut = h->D.dimer_cut; bd.want = BF_WANT_PF;
    bf_result_t rd;
    std::memset(&rd, 0, sizeof rd);
    rd.pf = h->D.o_dimer_pf;
    CU(cudaEventRecord(h->ev_fork, h->st), "fork self-dimer fold");
    CU(cudaStreamWaitEvent(h->st_dimer, h->ev_fork, 0), "fork self-dimer fold");
    const int rc = run_device(h->wd, &bd, &rd, true, h->st_dimer, nullptr, false);
    if (rc) return rc;
    CU(cudaEventRecord(h->ev_join, h->st_dimer), "join self-dimer fold");
  }
  bf_batch_t b;
  std::memset(&b, 0, sizeof b);
  b.B = h->B; b.stride = h->D.stride; b.seq = h->D.mut_seq; b.len = h->D.row_len; b.targets = h->D.row_tgt; b.n_targets = h->D.T; b.want = h->want;
  b.cut = h->two ? h->D.row_cut : nullptr;
  bf_result_t r;
  std::memset(&r, 0, sizeof r);
  r.mfe_dcal = h->D.o_mfe; r.mfe_ss = h->D.o_ss; r.pf = h->D.o_pf; r.eval_dcal = h->D.o_eval; r.defect = h->D.o_defect;
  // small batches: partition function beside the MFE fill, scaled by the parent sequence's MFE (kept per replica).  Single strands
  // up to 8 x the SM count (measured: pays at every size tried, 0.76 -> 0.42 ms per sub-step at 64 x 104 nt, 15.5 -> 14.4 ms at
  // 296 x 400 nt), two strands up to half the SM count
  const bool beside = !init && h->overlap && h->B * 2 <= g.sm_count * (h->two ? 1 : 16) && !(h->want & BF_WANT_DEFECT);
  int rc = run_device(h->w, &b, &r, h->two, h->st, beside ? h->D.row_scale : nullptr, false);
  if (rc) return rc;
  if (h->C.subopt) {
    // negative design: (best, second best) energies of the rows that fold into their target (rare rows; the others are skipped)
    CU(bf_launch_design_nd_flag(h->D, h->B, h->st), "launch bf_k_design_nd_flag");
    BfBatchDev db;
    db.B = h->B; db.stride = h->D.stride; db.seq = h->D.mut_seq; db.len = h->D.row_len; db.cut = h->two ? h->D.row_cut : nullptr; db.nopair = nullptr;
    const int wstride = h->D.stride + 2, grid = std::min(h->B, g.sm_count);
    CU(h->w.ws_mfe.reserve((size_t)grid * bf_twobest_slot(wstride) * sizeof(int2)), "cudaMalloc(second-best workspace)");
    CU(bf_launch_twobest(g.dP, db, (int2 *)h->w.ws_mfe.p, wstride, grid, h->w.d_counters + 3, h->D.o_e1, h->D.o_e2, h->st, h->D.nd_flag, h->two), "launch bf_k_mfe2");
    g.launches += 2;
  }
  if (h->pks) {
    // pseudoknot overlay (sequence_utils.py:1166-1228): forbid what is paired, fold again, paint the new pairs with the next bracket
    // family; three rounds.  A round that finds no pair leaves the overlay and the mask as they are, so the rounds the reference
    // skips are no-ops here; all rows go through all rounds.
    bf_batch_t b2 = b;
    b2.want = BF_WANT_MFE | BF_WANT_SS; b2.nopair = h->D.pk_nopair; b2.targets = nullptr; b2.n_targets = 0;
    bf_result_t r2;
    std::memset(&r2, 0, sizeof r2);
    r2.mfe_dcal = h->D.o_mfe2; r2.mfe_ss = h->D.o_ss2;
    for (int round = 0; round < 3; round++) {
      CU(bf_launch_design_pk_mask(h->D, h->B, h->st), "launch bf_k_design_pk_mask");
      rc = run_device(h->w, &b2, &r2, false, h->st, nullptr, false);
      if (rc) return rc;
      CU(bf_launch_design_pk_paint(h->D, h->B, round, h->st), "launch bf_k_design_pk_paint");
      g.launches += 2;
    }
  }
  if (h->C.oligo == 3) CU(cudaStreamWaitEvent(h->st, h->ev_join, 0), "join self-dimer fold");
  return BF_OK;
}
}  // namespace

extern "C" {

int bf_design_create(const bf_design_t *c, void **handle) {
  if (!g.inited) return fail(BF_ERR_NOT_INIT, "bf_init has not been called");
  if (!g.have_params) return fail(BF_ERR_NOT_INIT, "no energy parameters loaded");
  if (!c || !handle) return fail(BF_ERR_ARG, "null argument");
  if (c->n_jobs <= 0 || c->replicas <= 0 || c->stride <= 0 || c->stride > 2000) return fail(BF_ERR_ARG, "bf_design_create: bad shape (stride must be in 1..2000)");
  for (int k = 0; k < c->n_terms && k < 8; k++)
    if (c->term[k] < 0 || c->term[k] > kTermEdef) return fail(BF_ERR_ARG, "bf_design_create: unknown scoring term");
  if (!c->target || !c->len || !c->allowed || !c->init_seq || !c->temps || !c->tm_prob) return fail(BF_ERR_ARG, "bf_design_create: null buffer");
  if (c->n_terms <= 0 || c->n_terms > 8 || c->re_attempt <= 0) return fail(BF_ERR_ARG, "bf_design_create: bad scoring terms / re_attempt");
  const int J = c->n_jobs, R = c->replicas, S = c->stride;
  const size_t G = (size_t)J * R;
  // host-side preparation: partner tables and the lists of mutable positions
  std::vector<short> tpt((size_t)J * S, -1);
  std::vector<unsigned short> avail((size_t)J * S, 0);
  std::vector<int> n_avail(J, 0), len_a(J, 0);
  bool two = false;
  for (int j = 0; j < J; j++) {
    const int n = c->len[j];
    if (n <= 0 || n > S) return fail(BF_ERR_ARG, "bf_design_create: length outside (0, stride]");
    if (c->len_a) {
      if (c->len_a[j] < 0 || c->len_a[j] >= n) return fail(BF_ERR_ARG, "bf_design_create: strand A length outside [0, len)");
      len_a[j] = c->len_a[j];
      two = two || len_a[j] > 0;
    }
    // one stack per bracket family; the families beyond ( ) only with the pseudoknot overlay
    std::vector<int> stk[4];
    for (int i = 0; i < n; i++) {
      const char ch = c->target[(size_t)j * S + i];
      const char *po = strchr("([<{", ch), *pc = strchr(")]>}", ch);
      if (ch && po) {
        if (po - "([<{" > 0 && !c->pks) return fail(BF_ERR_ARG, "bf_design_create: targets may contain only . ( ) (pseudoknot brackets need pks = 1)");
        stk[po - "([<{"].push_back(i);
      } else if (ch && pc) {
        std::vector<int> &sk = stk[pc - ")]>}"];
        if (sk.empty()) return fail(BF_ERR_ARG, "bf_design_create: unbalanced target");
        tpt[(size_t)j * S + i] = (short)sk.back(); tpt[(size_t)j * S + sk.back()] = (short)i; sk.pop_back();
      } else if (ch != '.') return fail(BF_ERR_ARG, "bf_design_create: targets may contain only . ( ) and, with pks = 1, [ ] < > { }");
      const uint8_t a = c->allowed[(size_t)j * S + i];
      if (a == 0 || a > 15) return fail(BF_ERR_ARG, "bf_design_create: allowed-letter mask outside 1..15");
      if (__builtin_popcount(a) > 1) avail[(size_t)j * S + n_avail[j]++] = (unsigned short)i;
    }
    for (auto &sk : stk)
      if (!sk.empty()) return fail(BF_ERR_ARG, "bf_design_create: unbalanced target");
  }
  if (c->pks && two) return fail(BF_ERR_ARG, "bf_design_create: the pseudoknot overlay needs single-strand jobs");
  if (c->oligo == 3 && two) return fail(BF_ERR_ARG, "bf_design_create: avoid designs (oligo = 3) need single-strand jobs");
  if (c->subopt && c->pks) return fail(BF_ERR_ARG, "bf_design_create: negative design (subopt) does not combine with the pseudoknot overlay");
  if (!two && (bf_fill_mfe_mode(S) == 0 || bf_fill_pf_mode(S) == 0)) return fail(BF_ERR_UNAVAILABLE, "bf_design_create: stride outside the fill path");
  // optional scenario terms: alternative structures, motifs
  const int max_alt = c->alt_targets ? c->max_alt : 0;
  if (max_alt < 0 || max_alt > 16 || (max_alt > 0 && !c->n_alt)) return fail(BF_ERR_ARG, "bf_design_create: alternative structures: max_alt outside 0..16 or n_alt missing");
  for (int j = 0; j < J && max_alt > 0; j++) {
    if (c->n_alt[j] < 0 || c->n_alt[j] > max_alt) return fail(BF_ERR_ARG, "bf_design_create: n_alt outside 0..max_alt");
    for (int a = 0; a < c->n_alt[j]; a++) {
      int depth = 0;
      for (int i = 0; i < c->len[j]; i++) {
        const char ch = c->alt_targets[((size_t)j * max_alt + a) * S + i];
        if (ch == '(') depth++;
        else if (ch == ')') { if (--depth < 0) break; }
        else if (ch != '.') return fail(BF_ERR_ARG, "bf_design_create: alternative structures may contain only . ( )");
      }
      if (depth != 0) return fail(BF_ERR_ARG, "bf_design_create: unbalanced alternative structure");
    }
  }
  if (c->move_partner)
    for (int j = 0; j < J; j++)
      for (int i = 0; i < c->len[j]; i++)
        if (c->move_partner[(size_t)j * S + i] < -1 || c->move_partner[(size_t)j * S + i] >= c->len[j]) return fail(BF_ERR_ARG, "bf_design_create: move_partner outside the sequence");
  if ((c->snake_id != nullptr) != (c->snake_letter != nullptr)) return fail(BF_ERR_ARG, "bf_design_create: snake_id and snake_letter go together");
  if (c->n_motifs < 0 || c->n_motifs > 8 || (c->n_motifs > 0 && (!c->motif_mask || !c->motif_len || !c->motif_bonus))) return fail(BF_ERR_ARG, "bf_design_create: at most 8 motifs, with masks, lengths and bonuses");
  for (int m = 0; m < c->n_motifs; m++)
    if (c->motif_len[m] < 1 || c->motif_len[m] > 32) return fail(BF_ERR_ARG, "bf_design_create: motif length outside 1..32");
  DesignLoop *h = new DesignLoop;
  h->two = two;
  h->pks = c->pks != 0;
  h->overlap = bf_opt("BF_DESIGN_OVERLAP", 1) != 0;
  std::memset(&h->D, 0, sizeof h->D);
  std::memset(&h->C, 0, sizeof h->C);
  auto bail = [&](cudaError_t e, const char *what) { h->destroy(); delete h; return cuda_fail(e, what); };
#define DCU(call, what) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return bail(e_, what); } while (0)
  DCU(cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking), "cudaStreamCreate(design)");
  DCU(h->w.create(), "create design workspace");
  BfDesignDev &D = h->D;
  D.J = J; D.R = R; D.stride = S;
  char *tgt; short *d_tpt; uint8_t *allowed, *d_same; int *len, *d_len_a; unsigned short *d_avail; int *d_navail; double *temps, *tm_prob;
  DCU(h->alloc(&tgt, (size_t)J * S), "cudaMalloc(design)"); DCU(h->alloc(&d_tpt, (size_t)J * S), "cudaMalloc(design)");
  DCU(h->alloc(&allowed, (size_t)J * S), "cudaMalloc(design)"); DCU(h->alloc(&len, J), "cudaMalloc(design)"); DCU(h->alloc(&d_len_a, J), "cudaMalloc(design)"); DCU(h->alloc(&d_same, J), "cudaMalloc(design)");
  DCU(h->alloc(&d_avail, (size_t)J * S), "cudaMalloc(design)"); DCU(h->alloc(&d_navail, J), "cudaMalloc(design)");
  DCU(h->alloc(&temps, R), "cudaMalloc(design)"); DCU(h->alloc(&tm_prob, R), "cudaMalloc(design)");
  DCU(h->alloc(&D.job_rng, J), "cudaMalloc(design)");
  DCU(h->alloc(&D.best_seq, (size_t)J * S), "cudaMalloc(design)"); DCU(h->alloc(&D.best_ss, (size_t)J * (S + 1)), "cudaMalloc(design)");
  DCU(h->alloc(&D.best_rec, (size_t)J * kDesignRec), "cudaMalloc(design)");
  DCU(h->alloc(&D.solved_step, J), "cudaMalloc(design)"); DCU(h->alloc(&D.n_solved, J), "cudaMalloc(design)");
  DCU(h->alloc(&D.re_counts, (size_t)J * 3), "cudaMalloc(design)");
  DCU(h->alloc(&D.cur_seq, G * S), "cudaMalloc(design)"); DCU(h->alloc(&D.cur_ss, G * (S + 1)), "cudaMalloc(design)");
  DCU(h->alloc(&D.rec, G * kDesignRec), "cudaMalloc(design)"); DCU(h->alloc(&D.shelf, G), "cudaMalloc(design)");
  DCU(h->alloc(&D.rng, G), "cudaMalloc(design)"); DCU(h->alloc(&D.counts, G * 3), "cudaMalloc(design)");
  DCU(h->alloc(&h->d_rowmap, G), "cudaMalloc(design)"); DCU(h->alloc(&h->d_active, J), "cudaMalloc(design)");
  DCU(h->alloc(&D.mut_seq, G * S), "cudaMalloc(design)"); DCU(h->alloc(&D.row_len, G), "cudaMalloc(design)"); DCU(h->alloc(&D.row_cut, G), "cudaMalloc(design)");
  DCU(h->alloc(&D.row_scale, G), "cudaMalloc(design)"); DCU(h->alloc(&D.cur_mfe, G), "cudaMalloc(design)");
  if (c->move_partner) {
    short *d_mpt;
    DCU(h->alloc(&d_mpt, (size_t)J * S), "cudaMalloc(design)");
    DCU(cudaMemcpy(d_mpt, c->move_partner, (size_t)J * S * sizeof(short), cudaMemcpyHostToDevice), "H2D design");
    D.mpt = d_mpt;
  }
  if (c->snake_id && c->snake_letter) {
    signed char *d_sid; char *d_sl;
    DCU(h->alloc(&d_sid, (size_t)J * S), "cudaMalloc(design)"); DCU(h->alloc(&d_sl, (size_t)J * S * 4), "cudaMalloc(design)");
    DCU(cudaMemcpy(d_sid, c->snake_id, (size_t)J * S, cudaMemcpyHostToDevice), "H2D design");
    DCU(cudaMemcpy(d_sl, c->snake_letter, (size_t)J * S * 4, cudaMemcpyHostToDevice), "H2D design");
    D.snake_id = d_sid; D.snake_letter = d_sl;
  }
  D.max_alt = max_alt; D.T = 1 + max_alt;
  if (max_alt > 0) {
    char *d_alt; int *d_nalt;
    DCU(h->alloc(&d_alt, (size_t)J * max_alt * S), "cudaMalloc(design)"); DCU(h->alloc(&d_nalt, J), "cudaMalloc(design)");
    DCU(cudaMemcpy(d_alt, c->alt_targets, (size_t)J * max_alt * S, cudaMemcpyHostToDevice), "H2D design");
    DCU(cudaMemcpy(d_nalt, c->n_alt, J * sizeof(int), cudaMemcpyHostToDevice), "H2D design");
    D.alt = d_alt; D.n_alt = d_nalt;
  }
  DCU(h->alloc(&D.row_tgt, G * D.T * S), "cudaMalloc(design)"); DCU(h->alloc(&D.o_mfe, G), "cudaMalloc(design)");
  DCU(h->alloc(&D.o_ss, G * (S + 1)), "cudaMalloc(design)"); DCU(h->alloc(&D.o_pf, G * 5), "cudaMalloc(design)");
  DCU(h->alloc(&D.o_eval, G * D.T), "cudaMalloc(design)");
  if (c->subopt) { DCU(h->alloc(&D.nd_flag, G), "cudaMalloc(design)"); DCU(h->alloc(&D.o_e1, G), "cudaMalloc(design)"); DCU(h->alloc(&D.o_e2, G), "cudaMalloc(design)"); }
  if (h->pks) { DCU(h->alloc(&D.pk_nopair, G * S), "cudaMalloc(design)"); DCU(h->alloc(&D.o_mfe2, G), "cudaMalloc(design)"); DCU(h->alloc(&D.o_ss2, G * (S + 1)), "cudaMalloc(design)"); }
  if (c->oligo == 3) {   // self-dimer rows (stride 2 S <= 4000, bf_score_batch's limit), their PF columns, a second workspace and stream
    DCU(h->alloc(&D.dimer_seq, G * 2 * S), "cudaMalloc(design)"); DCU(h->alloc(&D.dimer_len, G), "cudaMalloc(design)"); DCU(h->alloc(&D.dimer_cut, G), "cudaMalloc(design)");
    DCU(h->alloc(&D.o_dimer_pf, G * 5), "cudaMalloc(design)");
    DCU(h->wd.create(), "create self-dimer workspace");
    DCU(cudaStreamCreateWithFlags(&h->st_dimer, cudaStreamNonBlocking), "cudaStreamCreate(self-dimer)");
    DCU(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming), "cudaEventCreate(self-dimer)");
    DCU(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming), "cudaEventCreate(self-dimer)");
  }
  h->want = BF_WANT_MFE | BF_WANT_SS | BF_WANT_PF | BF_WANT_EVAL;
  BfDesignCfg &C = h->C;
  C.n_terms = c->n_terms;
  for (int k = 0; k < c->n_terms; k++) {
    if (c->term[k] < 0 || c->term[k] > kTermEdef) return bail(cudaErrorInvalidValue, "bf_design_create: unknown scoring term");
    C.term[k] = c->term[k]; C.weight[k] = c->weight[k];
    if (c->term[k] == kTermEdef) h->want |= BF_WANT_DEFECT;
  }
  if (h->want & BF_WANT_DEFECT) DCU(h->alloc(&D.o_defect, G), "cudaMalloc(design)");
  C.metropolis_L = c->metropolis_L; C.point_mutations = c->point_mutations; C.acgu = c->acgu;
  for (int k = 0; k < 4; k++) C.nt_weight[k] = c->nt_weight[k];
  C.oligo = c->oligo;
  C.subopt = c->subopt != 0;
  C.n_motifs = c->n_motifs;
  for (int m = 0; m < c->n_motifs; m++) {
    C.motif_len[m] = c->motif_len[m]; C.motif_bonus[m] = c->motif_bonus[m];
    for (int k = 0; k < 32; k++) C.motif_mask[m][k] = k < c->motif_len[m] ? c->motif_mask[(size_t)m * 32 + k] : 0;
  }
  if (two && (h->want & BF_WANT_DEFECT)) { h->destroy(); delete h; return fail(BF_ERR_ARG, "bf_design_create: the Edef term needs single-strand jobs"); }
  h->re_attempt = c->re_attempt;
  D.tgt = tgt; D.tpt = d_tpt; D.allowed = allowed; D.len = len; D.len_a = d_len_a; D.same_halves = d_same; D.avail = d_avail; D.n_avail = d_navail; D.temps = temps; D.tm_prob = tm_prob;
  D.rowmap = h->d_rowmap;
  // uploads
  std::vector<unsigned long long> rng(G), jrng(J);
  unsigned long long sd = c->seed * 0x9E3779B97F4A7C15ull + 0x2545F4914F6CDD1Dull;
  auto next = [&sd]() { sd += 0x9E3779B97F4A7C15ull; unsigned long long z = sd; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; return z ^ (z >> 31); };
  for (auto &x : rng) x = next();
  for (auto &x : jrng) x = next();
  std::vector<int> shelf(G);
  for (size_t k = 0; k < G; k++) shelf[k] = (int)(k % R);   // replica r starts on shelf r (sequence_utils.py:880-884)
  std::vector<double> best((size_t)J * kDesignRec, 1e300);
  std::vector<int> sstep(J, -1);
  DCU(cudaMemcpy(tgt, c->target, (size_t)J * S, cudaMemcpyHostToDevice), "H2D design"); DCU(cudaMemcpy(d_tpt, tpt.data(), tpt.size() * sizeof(short), cudaMemcpyHostToDevice), "H2D design");
  DCU(cudaMemcpy(allowed, c->allowed, (size_t)J * S, cudaMemcpyHostToDevice), "H2D design"); DCU(cudaMemcpy(len, c->len, J * sizeof(int), cudaMemcpyHostToDevice), "H2D design"); DCU(cudaMemcpy(d_len_a, len_a.data(), J * sizeof(int), cudaMemcpyHostToDevice), "H2D design");
  {
    std::vector<uint8_t> same(J, 0);
    for (int j = 0; j < J; j++) {
      const int a = len_a[j], n = c->len[j];
      same[j] = a > 0 && n == 2 * a && std::memcmp(c->target + (size_t)j * S, c->target + (size_t)j * S + a, a) == 0;
    }
    DCU(cudaMemcpy(d_same, same.data(), J, cudaMemcpyHostToDevice), "H2D design");
  }
  DCU(cudaMemcpy(d_avail, avail.data(), avail.size() * sizeof(unsigned short), cudaMemcpyHostToDevice), "H2D design");
  DCU(cudaMemcpy(d_navail, n_avail.data(), J * sizeof(int), cudaMemcpyHostToDevice), "H2D design");
  DCU(cudaMemcpy(temps, c->temps, R * sizeof(double), cudaMemcpyHostToDevice), "H2D design"); DCU(cudaMemcpy(tm_prob, c->tm_prob, R * sizeof(double), cudaMemcpyHostToDevice), "H2D design");
  DCU(cudaMemcpy(D.rng, rng.data(), G * sizeof(unsigned long long), cudaMemcpyHostToDevice), "H2D design");
  DCU(cudaMemcpy(D.job_rng, jrng.data(), J * sizeof(unsigned long long), cudaMemcpyHostToDevice), "H2D design");
  DCU(cudaMemcpy(D.shelf, shelf.data(), G * sizeof(int), cudaMemcpyHostToDevice), "H2D design");
  DCU(cudaMemcpy(D.best_rec, best.data(), best.size() * sizeof(double), cudaMemcpyHostToDevice), "H2D design");
  DCU(cudaMemcpy(D.solved_step, sstep.data(), J * sizeof(int), cudaMemcpyHostToDevice), "H2D design");
  DCU(cudaMemcpy(D.cur_seq, c->init_seq, G * S, cudaMemcpyHostToDevice), "H2D design");
#undef DCU
  h->active.assign(J, 1);
  int rc = design_rows(h);
  // score the start sequences (sequence_utils.py:862-888) and record them as step 0
  if (!rc) rc = bf_launch_design_propose(h->D, h->C, h->B, true, h->st) == cudaSuccess ? BF_OK : fail(BF_ERR_CUDA, "launch bf_k_design_propose");
  if (!rc) rc = design_score(h, true);
  if (!rc) rc = bf_launch_design_accept(h->D, h->C, h->B, true, 0, h->st) == cudaSuccess ? BF_OK : fail(BF_ERR_CUDA, "launch bf_k_design_accept");
  if (!rc) rc = bf_launch_design_exchange(h->D, h->C, h->d_active, 0, h->st) == cudaSuccess ? BF_OK : fail(BF_ERR_CUDA, "launch bf_k_design_exchange");
  if (!rc && cudaStreamSynchronize(h->st) != cudaSuccess) rc = fail(BF_ERR_CUDA, std::string("design loop start: ") + cudaGetErrorString(cudaGetLastError()));
  if (rc) { h->destroy(); delete h; return rc; }
  g.launches += 3;
  *handle = h;
  return BF_OK;
}

int bf_design_run(void *handle, int32_t global_steps) {
  DesignLoop *h = (DesignLoop *)handle;
  if (!h || global_steps < 0) return fail(BF_ERR_ARG, "bf_design_run: bad argument");
  for (int s = 0; s < global_steps; s++) {
    h->gstep++;
    for (int k = 0; k < h->re_attempt && h->B > 0; k++) {
      CU(bf_launch_design_propose(h->D, h->C, h->B, false, h->st), "launch bf_k_design_propose");
      int rc = design_score(h);
      if (rc) return rc;
      CU(bf_launch_design_accept(h->D, h->C, h->B, false, h->gstep, h->st), "launch bf_k_design_accept");
      g.launches += 2;
    }
    CU(bf_launch_design_exchange(h->D, h->C, h->d_active, h->gstep, h->st), "launch bf_k_design_exchange");
    g.launches++;
  }
  return BF_OK;
}

int bf_design_busy(void *handle, int32_t *busy) {
  DesignLoop *h = (DesignLoop *)handle;
  if (!h || !busy) return fail(BF_ERR_ARG, "bf_design_busy: null argument");
  const cudaError_t e = cudaStreamQuery(h->st);
  if (e != cudaSuccess && e != cudaErrorNotReady) return cuda_fail(e, "bf_design_busy");
  *busy = e == cudaErrorNotReady ? 1 : 0;
  return BF_OK;
}

int bf_design_sync(void *handle) {
  DesignLoop *h = (DesignLoop *)handle;
  if (!h) return fail(BF_ERR_ARG, "bf_design_sync: null handle");
  CU(cudaStreamSynchronize(h->st), "bf_design_sync");
  return BF_OK;
}

int bf_design_set_active(void *handle, const uint8_t *active_jobs) {
  DesignLoop *h = (DesignLoop *)handle;
  if (!h || !active_jobs) return fail(BF_ERR_ARG, "bf_design_set_active: null argument");
  CU(cudaStreamSynchronize(h->st), "bf_design_set_active");
  for (int j = 0; j < h->D.J; j++) h->active[j] = active_jobs[j] ? 1 : 0;
  return design_rows(h);
}

int bf_design_read_swaps(void *handle, uint32_t *re_counts) {
  DesignLoop *h = (DesignLoop *)handle;
  if (!h || !re_counts) return fail(BF_ERR_ARG, "bf_design_read_swaps: null argument");
  CU(cudaStreamSynchronize(h->st), "bf_design_read_swaps");
  CU(cudaMemcpy(re_counts, h->D.re_counts, (size_t)h->D.J * 3 * sizeof(unsigned), cudaMemcpyDeviceToHost), "D2H re_counts");
  return BF_OK;
}

int bf_design_read_jobs(void *handle, char *best_seq, char *best_ss, double *best_rec, int32_t *solved_step, uint32_t *n_solved) {
  DesignLoop *h = (DesignLoop *)handle;
  if (!h) return fail(BF_ERR_ARG, "bf_design_read_jobs: null handle");
  CU(cudaStreamSynchronize(h->st), "bf_design_read_jobs");
  const size_t J = h->D.J, S = h->D.stride;
  if (best_seq) CU(cudaMemcpy(best_seq, h->D.best_seq, J * S, cudaMemcpyDeviceToHost), "D2H best_seq");
  if (best_ss) CU(cudaMemcpy(best_ss, h->D.best_ss, J * (S + 1), cudaMemcpyDeviceToHost), "D2H best_ss");
  if (best_rec) CU(cudaMemcpy(best_rec, h->D.best_rec, J * kDesignRec * sizeof(double), cudaMemcpyDeviceToHost), "D2H best_rec");
  if (solved_step) CU(cudaMemcpy(solved_step, h->D.solved_step, J * sizeof(int), cudaMemcpyDeviceToHost), "D2H solved_step");
  if (n_solved) CU(cudaMemcpy(n_solved, h->D.n_solved, J * sizeof(unsigned), cudaMemcpyDeviceToHost), "D2H n_solved");
  return BF_OK;
}

int bf_design_read_replicas(void *handle, char *seq, char *ss, double *rec, int32_t *shelf, uint32_t *counts) {
  DesignLoop *h = (DesignLoop *)handle;
  if (!h) return fail(BF_ERR_ARG, "bf_design_read_replicas: null handle");
  CU(cudaStreamSynchronize(h->st), "bf_design_read_replicas");
  const size_t G = (size_t)h->D.J * h->D.R, S = h->D.stride;
  if (seq) CU(cudaMemcpy(seq, h->D.cur_seq, G * S, cudaMemcpyDeviceToHost), "D2H cur_seq");
  if (ss) CU(cudaMemcpy(ss, h->D.cur_ss, G * (S + 1), cudaMemcpyDeviceToHost), "D2H cur_ss");
  if (rec) CU(cudaMemcpy(rec, h->D.rec, G * kDesignRec * sizeof(double), cudaMemcpyDeviceToHost), "D2H rec");
  if (shelf) CU(cudaMemcpy(shelf, h->D.shelf, G * sizeof(int), cudaMemcpyDeviceToHost), "D2H shelf");
  if (counts) CU(cudaMemcpy(counts, h->D.counts, G * 3 * sizeof(unsigned), cudaMemcpyDeviceToHost), "D2H counts");
  return BF_OK;
}

int bf_design_propose_only(void *handle, char *mut_seq) {
  DesignLoop *h = (DesignLoop *)handle;
  if (!h || !mut_seq) return fail(BF_ERR_ARG, "bf_design_propose_only: null argument");
  CU(bf_launch_design_propose(h->D, h->C, h->B, false, h->st), "launch bf_k_design_propose");
  g.launches++;
  CU(cudaMemcpyAsync(mut_seq, h->D.mut_seq, (size_t)h->B * h->D.stride, cudaMemcpyDeviceToHost, h->st), "D2H mutants");
  CU(cudaStreamSynchronize(h->st), "bf_design_propose_only");
  return BF_OK;
}

int bf_design_destroy(void *handle) {
  DesignLoop *h = (DesignLoop *)handle;
  if (!h) return BF_OK;
  h->destroy();
  delete h;
  return BF_OK;
}

}  // extern "C"
