// bf_capi.cu -- engine state and the C-ABI declared in include/b200fold.h.
#include <cuda_runtime.h>

#include <algorithm>
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
                                       "BF_BLK_MIN", "BF_BLK_MIN_PF", "BF_FORCE_GENERIC", "BF_DESIGN_OVERLAP"};

int bf_opt(const char *name, int dflt) {
  const char *v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
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

// exterior recursions by one CTA per sequence instead of one warp per sequence: batches that leave SMs idle (BF_EXT_WIDE=0/1 overrides)
bool wide_ext(int B, int stride) {
  const int v = bf_opt("BF_EXT_WIDE", -1);
  if (v >= 0) return v != 0 && bf_ext_wide_ok(stride);
  return B <= 2 * g.sm_count && bf_ext_wide_ok(stride);
}

// all pointers are device pointers
// scale_override (device, B ints, dcal/mol): energies that set the partition function's per-nucleotide scale instead of this
// call's own MFE.  The result does not depend on the scale beyond rounding, and without that dependency the partition function
// runs on the workspace's second stream beside the MFE fill -- worth it when both grids fit the GPU together (small batches).
int run_device(Workspace &w, const bf_batch_t *b, const bf_result_t *r, bool two, cudaStream_t st, const int *scale_override = nullptr,
               bool timing = true) {
  if (b->B == 0) return BF_OK;
  BfBatchDev db;
  db.B = b->B; db.stride = b->stride; db.seq = b->seq; db.len = b->len; db.cut = b->cut; db.nopair = b->nopair;
  const int wstride = b->stride + 2;
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
  const bool fill_mfe = !two && !g.force_generic && bf_fill_mfe_mode(b->stride) != 0;
  const bool fill_pf = !two && !g.force_generic && bf_fill_pf_mode(b->stride) != 0;
  if (b->want & (BF_WANT_MFE | BF_WANT_SS)) {
    int *out_mfe = r->mfe_dcal;
    if (!out_mfe) { CU(w.d_mfe_scratch.reserve((size_t)b->B * sizeof(int)), "cudaMalloc(mfe scratch)"); out_mfe = (int *)w.d_mfe_scratch.p; }
    if (timing) cudaEventRecord(w.ev[0], st);
    if (fill_mfe) {
      const size_t slot = bf_tri_slot(b->stride) * sizeof(int);
      CU(w.tri_c.reserve((size_t)b->B * slot), "cudaMalloc(c table)");
      CU(w.tri_f.reserve((size_t)b->B * slot), "cudaMalloc(fML table)");
      int *f5 = nullptr;
      const size_t wsi = bf_mfe_ws_slot(b->stride, b->B) * sizeof(int);
      if (wsi) {
        int grid = 0;
        CU(bf_mfe_fill_grid(db, g.sm_count, &grid), "size bf_k_mfe_fill");
        CU(w.ws_ring.reserve((size_t)grid * wsi), "cudaMalloc(ring workspace)");
      }
      if (bf_mfe_fill_does_ext(b->stride, b->B)) {
        CU(w.f5buf.reserve((size_t)b->B * (b->stride + 4) * sizeof(int)), "cudaMalloc(f5)");
        f5 = (int *)w.f5buf.p;
      }
      CU(bf_launch_mfe_fill(g.dP, db, (int *)w.tri_c.p, (int *)w.tri_f.p, (int *)w.ws_ring.p, g.sm_count, w.d_counters + 0, st, f5),
         "launch bf_k_mfe_fill");
      if (!f5 && wide_ext(b->B, b->stride)) {   // few sequences: the exterior recursion by one CTA per sequence (bf_ext.cu)
        CU(w.f5buf.reserve((size_t)b->B * (b->stride + 4) * sizeof(int)), "cudaMalloc(f5)");
        f5 = (int *)w.f5buf.p;
        CU(bf_launch_f5_wide(g.dP, db, (const int *)w.tri_c.p, f5, st), "launch bf_k_f5_wide");
        g.launches++;
      }
      CU(bf_launch_trace(g.dP, db, (const int *)w.tri_c.p, (const int *)w.tri_f.p, out_mfe, (b->want & BF_WANT_SS) ? r->mfe_ss : nullptr,
                         b->stride + 1, st, f5), "launch bf_k_trace");
      g.launches += 2;
    } else {
      int occ = bf_occupancy_mfe(two, wstride);
      int grid = std::min(b->B, g.sm_count * occ);
      size_t slot = bf_mfe_slot_ints(wstride) * sizeof(int);
      // keep the workspace within a sane share of HBM
      while (grid > g.sm_count && (size_t)grid * slot > ((size_t)48 << 30)) grid -= g.sm_count;
      CU(w.ws_mfe.reserve((size_t)grid * slot), "cudaMalloc(mfe workspace)");
      CU(bf_launch_mfe(g.dP, db, two, (int *)w.ws_mfe.p, wstride, grid, w.d_counters + 0, out_mfe,
                       (b->want & BF_WANT_SS) ? r->mfe_ss : nullptr, b->stride + 1, st), "launch bf_k_mfe");
      g.launches++;
    }
    if (timing) cudaEventRecord(w.ev[1], st);
    w.ran[0] = timing;
    mfe_for_scale = out_mfe;
  }
  const bool want_out = (b->want & (BF_WANT_BPP | BF_WANT_DEFECT)) != 0;
  if (want_out && (two || !fill_pf))
    return fail(BF_ERR_UNAVAILABLE, "base-pair probabilities / ensemble defect: single-strand sequences within the fill path's length range only");
  if ((b->want & BF_WANT_PF) || want_out) {
    BfBatchDev dbp = db;
    dbp.nopair = nullptr;  // hard constraints are added after fc.pf() in the reference (sequence_utils.py:1181)
    // a constrained MFE is not a bound on the unconstrained ensemble: only use it for scaling when unconstrained
    const bool beside = scale_override && !want_out && !b->nopair;
    cudaStream_t sp = beside ? w.st2 : st;
    if (beside) CU(cudaStreamWaitEvent(sp, w.ev_fork, 0), "fork");
    const int *scale_src = beside ? scale_override : (b->nopair ? nullptr : mfe_for_scale);
    if (timing) cudaEventRecord(w.ev[2], sp);
    if (fill_pf) {
      const size_t slot = bf_tri_slot(b->stride) * sizeof(double);
      CU(w.tri_qb.reserve((size_t)b->B * slot), "cudaMalloc(qb table)");
      CU(w.d_lnscale.reserve((size_t)b->B * sizeof(double)), "cudaMalloc(lnscale)");
      int grid = 0;
      CU(bf_pf_fill_grid(dbp, g.sm_count, &grid), "size bf_k_pf_fill");
      const size_t ws = bf_pf_ws_slot(b->stride, b->B) * sizeof(double);
      if (ws) CU(w.ws_qm.reserve((size_t)grid * ws), "cudaMalloc(qm workspace)");
      double *qmseq = nullptr;
      if (want_out) {
        CU(w.qm_seq.reserve((size_t)b->B * 2 * slot), "cudaMalloc(per-sequence qm/qm1)");
        qmseq = (double *)w.qm_seq.p;
      }
      CU(bf_launch_pf_fill(g.dP, dbp, (double *)w.tri_qb.p, (double *)w.ws_qm.p, qmseq, scale_src, (double *)w.d_lnscale.p, g.sm_count,
                           w.d_counters + 1, sp, r->pf), "launch bf_k_pf_fill");
      g.launches++;
      if (!bf_pf_fill_does_ext(b->stride, b->B)) {
        if (wide_ext(b->B, b->stride))
          CU(bf_launch_q5_wide(g.dP, dbp, (const double *)w.tri_qb.p, (const double *)w.d_lnscale.p, r->pf, sp), "launch bf_k_q5_wide");
        else
          CU(bf_launch_pf_ext(g.dP, dbp, (const double *)w.tri_qb.p, (const double *)w.d_lnscale.p, r->pf, sp), "launch bf_k_pf_ext");
        g.launches++;
      }
      if (want_out) {
        int ogrid = 0;
        CU(bf_out_grid(dbp, g.sm_count, &ogrid), "size bf_k_pf_out");
        CU(w.ws_out.reserve((size_t)ogrid * bf_out_ws_slot(b->stride) * sizeof(double)), "cudaMalloc(outside workspace)");
        if (b->want & BF_WANT_BPP) CU(cudaMemsetAsync(r->bpp, 0, (size_t)b->B * b->stride * b->stride * sizeof(double), st), "clear bpp");
        CU(bf_launch_pf_out(g.dP, dbp, (const double *)w.tri_qb.p, qmseq, (double *)w.ws_out.p, (const double *)w.d_lnscale.p,
                            (b->want & BF_WANT_DEFECT) ? b->targets : nullptr, b->n_targets, b->stride,
                            (b->want & BF_WANT_DEFECT) ? r->defect : nullptr, (b->want & BF_WANT_BPP) ? r->bpp : nullptr, ogrid,
                            w.d_counters + 2, st), "launch bf_k_pf_out");
        g.launches++;
      }
    } else {
      int occ = bf_occupancy_pf(two, wstride);
      int grid = std::min(b->B, g.sm_count * occ);
      size_t slot = bf_pf_slot_doubles(wstride) * sizeof(double);
      while (grid > g.sm_count && (size_t)grid * slot > ((size_t)64 << 30)) grid -= g.sm_count;
      CU(w.ws_pf.reserve((size_t)grid * slot), "cudaMalloc(pf workspace)");
      CU(bf_launch_pf(g.dP, dbp, two, (double *)w.ws_pf.p, wstride, grid, w.d_counters + 1, scale_src, r->pf, sp), "launch bf_k_pf");
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
  bf_fill_set_sms(g.sm_count);
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
  for (DevBuf *b : {&g.d_defect, &g.d_bpp, &g.d_seq, &g.d_len, &g.d_cut, &g.d_nopair, &g.d_targets, &g.d_mfe, &g.d_ss, &g.d_pf, &g.d_eval, &g.d_in, &g.d_out, &g.d_zero}) b->release();
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
