// One ADVI step (and one batch upload) as a single C-ABI call each: the whole launch sequence is
// issued from native code so the host language pays one FFI crossing per step instead of one per
// kernel.  Same sequence as the individual entry points; see include/spmf_b200.h.
//
// Replaces, per minibatch, bayesianquilts' minibatch_fit_surrogate_posterior body [EXT L3/L4]
// around PoissonFactorization.unormalized_log_prob (poisson.py:575-621).
#include <cuda_runtime.h>

#include "../../include/spmf_b200.h"

#define STEP_TRY(call)            \
  do {                            \
    int rc__ = (call);            \
    if (rc__ != SPMF_OK) return rc__; \
  } while (0)
#define CUDA_TRY(call)                         \
  do {                                         \
    cudaError_t e__ = (call);                  \
    if (e__ != cudaSuccess) return (int)e__;   \
  } while (0)

extern "C" {

int spmf_advi_step(const spmf_step_args* a) {
  if (!a) return SPMF_ERR_BAD_ARG;
  cudaStream_t caller = (cudaStream_t)a->caller_stream;
  cudaStream_t hot = a->hot_stream ? (cudaStream_t)a->hot_stream : caller;
  cudaStream_t side = a->side_stream ? (cudaStream_t)a->side_stream : hot;
  const bool multi = (hot != caller) || (side != hot);
  if (multi && (!a->ev_fork || !a->ev_join || !a->ev_done)) return SPMF_ERR_BAD_ARG;
  const int D = a->D, K = a->K, S = a->S;

  // per-step scalars to the device first (graph replay updates this one node's argument)
  if (a->step_state && !a->state_preset)
    STEP_TRY(spmf_step_state_set(a->step_state, a->rng_step, a->adam_t, a->adam_lr, a->adam_beta1, a->adam_beta2,
                                 a->adam_eps, a->clip_value, caller));
  if (multi) {
    CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_fork, caller));
    if (hot != caller) CUDA_TRY(cudaStreamWaitEvent(hot, (cudaEvent_t)a->ev_fork, 0));
    if (side != caller) CUDA_TRY(cudaStreamWaitEvent(side, (cudaEvent_t)a->ev_fork, 0));
  }
  // ---- Gamma draws + implicit gradients: only the backward needs them (side stream)
  if (a->fresh_noise)
    STEP_TRY(spmf_gamma_draw_grad_dev(a->params, a->noise, a->dgda, D, K, S, a->seed, a->rng_step, a->step_state, side));
  else
    STEP_TRY(spmf_gamma_grad(a->params, a->noise, D, K, S, a->dgda, side));
  // ---- hot path
  const bool hybrid = a->hot_cols > 0;
  if (hybrid && (!a->rank || !a->rowmid || !a->xhot || !a->ApT3 || !a->dzrT3 || !a->EVt)) return SPMF_ERR_BAD_ARG;
  if (a->fresh_noise)
    STEP_TRY(spmf_fill_noise_dev(a->noise, a->params, D, K, S, a->seed, a->rng_step, SPMF_NOISE_NORMAL, a->step_state,
                                 hot));
  // data-independent half of the backward: needs the noise only -> side stream, under the data term
  const bool split_bwd = a->scr_dpre && (side == hot || a->ev_noise);
  if (split_bwd) {
    if (side != hot) {
      CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_noise, hot));
      CUDA_TRY(cudaStreamWaitEvent(side, (cudaEvent_t)a->ev_noise, 0));
    }
    STEP_TRY(spmf_backward_pre_m(a->params, a->noise, a->dgda, a->eta, D, K, S, (float)a->nrows, a->u_tau_scale,
                                 a->s_tau_scale, a->decay, a->w_entropy, a->w_prior, a->world_size, a->grads,
                                 a->scr_f, a->scr_dpre, a->model, side));
  }
  // Adam on the tensors without a data term: their gradients are final now, nothing later in the step reads
  // their parameters (the data half of the backward touches v, w, u, s only) -> off the critical path
  const long long n_block = a->comm_off + a->comm_slack;
  const bool tail_early = a->adam_tail_early && a->adam_lr > 0.f;
  if (tail_early) {
    if (!split_bwd || !a->step_state || n_block <= 0 || n_block > a->n_params) return SPMF_ERR_BAD_ARG;
    if (a->n_params > n_block)
      STEP_TRY(spmf_adam_step_dev(a->params + n_block, a->grads + n_block, a->adam_m + n_block, a->adam_v + n_block,
                                  a->n_params - n_block, a->adam_lr, a->adam_beta1, a->adam_beta2, a->adam_eps,
                                  a->adam_t, a->clip_value, 1.0f, a->step_state, side));
  }
  if (side != hot) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_join, side));
  // (hybrid step with auxiliary streams: the fp64 operand sums are first read by spmf_rows_finish, so
  // they leave the critical path and run next to the encode GEMM)
  const bool pre_fork = hybrid && a->aux_stream1 && a->ev_aux_fork && a->ev_aux_join1;
  STEP_TRY(spmf_draw_operands_ranked_m(a->params, a->noise, a->eta, hybrid ? a->rank : nullptr, D, K, S, a->Ap,
                                       a->EV, a->PH, pre_fork ? nullptr : a->vsum, pre_fork ? nullptr : a->phisum,
                                       a->scr_d, a->model, hot));
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV, REC = KP * SV;
  if (a->ev_rows0) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_rows0, hot));
  const bool dense_link = a->link != SPMF_LINK_POISSON;
  if (dense_link) {
    // links without a closed-form sum(rate) (log_transform / Bernoulli): the whole data term runs in the
    // dense CUDA-core kernels of spmf_dense.cu; tables stay in feature order
    if (hybrid || !a->gs || !a->xdense) return SPMF_ERR_BAD_ARG;
    const float* xd = a->xdense_in ? a->xdense_in : a->xdense;
    if (!a->xdense_in) STEP_TRY(spmf_dense_scatter(a->rowptr, a->cols, a->vals, a->nrows, D, a->xdense, hot));
    STEP_TRY(spmf_dense_encode(xd, a->eta, a->rowsum, a->inv_xi, a->scale_rows, a->nrows, D, K, S, a->link, a->Ap,
                               a->z, hot));
    STEP_TRY(spmf_dense_rows(xd, a->rowsum, a->lgam, a->inv_xi, a->scale_rows, a->nrows, D, K, S, a->link,
                             SPMF_DENSE_OPTIMISTIC, 0, a->EV, a->PH, a->z, a->dzr, a->rowacc, a->gs, hot));
    // non-finite entries met: count them / find the smallest finite log-likelihood, then redo the row pass
    // with the reference's replacement (both launches return at once otherwise)
    STEP_TRY(spmf_dense_rows(xd, a->rowsum, a->lgam, a->inv_xi, a->scale_rows, a->nrows, D, K, S, a->link,
                             SPMF_DENSE_STATS, 1, a->EV, a->PH, a->z, a->dzr, a->rowacc, a->gs, hot));
    STEP_TRY(spmf_dense_rows(xd, a->rowsum, a->lgam, a->inv_xi, a->scale_rows, a->nrows, D, K, S, a->link,
                             SPMF_DENSE_GUARDED, 1, a->EV, a->PH, a->z, a->dzr, a->rowacc, a->gs, hot));
    if (a->ev_rows1) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_rows1, hot));
    STEP_TRY(spmf_batch_sums(a->z, a->rowacc, a->nrows, K, S, a->zcolsum, a->datasums, a->scr_d, hot));
    if (a->ev_cols0) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_cols0, hot));
    STEP_TRY(spmf_zero_col_grads(a->GAp, a->GEV, a->Gph, D, K, S, hot));
    STEP_TRY(spmf_dense_cols(xd, a->eta, a->nrows, D, K, S, a->link, 1, a->z, a->dzr, a->EV, a->PH, a->GAp, a->GEV,
                             a->Gph, a->gs, hot));
    if (a->ev_cols1) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_cols1, hot));
  } else {
  if (!hybrid) {
    STEP_TRY(spmf_csr_rows(a->rowptr, a->cols, a->vals, a->rowsum, a->lgam, a->inv_xi, a->scale_rows, a->nrows,
                           D, K, S, a->Ap, a->EV, a->PH, a->vsum, a->z, a->dzr, a->rowacc, 0, a->gs, hot));
  } else {
    // encode product of the hot block on the tensor cores: z = X_hot . A'[0:H]  (un-scaled)
    const int H = a->hot_cols;
    const int Hp = (H + 63) / 64 * 64;
    // the EV / phi tile blocks and the zeroing of the column-gradient tables do not depend on the
    // GEMM: run them next to it on an auxiliary stream when one is available
    if (pre_fork) {
      cudaStream_t s1 = (cudaStream_t)a->aux_stream1;
      CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_aux_fork, hot));
      CUDA_TRY(cudaStreamWaitEvent(s1, (cudaEvent_t)a->ev_aux_fork, 0));
      STEP_TRY(spmf_hot_ev_tiles(a->EV, a->PH, D, H, K, S, a->EVt, s1));
      STEP_TRY(spmf_zero_col_grads(a->GAp, a->GEV, a->Gph, D, K, S, s1));
      STEP_TRY(spmf_operand_sums(a->EV, a->PH, D, K, S, a->vsum, a->phisum, a->scr_d, s1));
      CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_aux_join1, s1));
    }
    STEP_TRY(spmf_split3_transpose(a->Ap, REC, (long long)D * REC, H, Hp, REC, a->ApT3, a->t3_qstride, NQ, hot));
    CUDA_TRY(cudaMemsetAsync(a->z, 0, (size_t)NQ * a->nrows * REC * sizeof(float), hot));
    STEP_TRY(spmf_umma_gemm3(a->xhot, 0, a->nrows, a->ApT3, a->t3_qstride, a->z, REC, (long long)a->nrows * REC,
                             REC, Hp, NQ, a->gemm_splits, hot));
    if (pre_fork) CUDA_TRY(cudaStreamWaitEvent(hot, (cudaEvent_t)a->ev_aux_join1, 0));
    // per-nonzero terms of the hot block in the fused tcgen05 tile kernel; the gather kernel keeps
    // the uncovered entries only
    if (!pre_fork) {
      STEP_TRY(spmf_hot_ev_tiles(a->EV, a->PH, D, H, K, S, a->EVt, hot));
      STEP_TRY(spmf_zero_col_grads(a->GAp, a->GEV, a->Gph, D, K, S, hot));
    }
    STEP_TRY(spmf_csr_rows_cold(a->rowptr, a->cols, a->vals, a->rowmid, a->rowsum, a->inv_xi, a->scale_rows,
                                a->nrows, D, K, S, a->Ap, a->EV, a->PH, a->z, a->dzr, a->rowacc, a->gs, hot));
    if (a->ev_tile0) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_tile0, hot));
    STEP_TRY(spmf_hot_tile(a->xhot, a->EVt, a->z, a->nrows, D, H, K, S, a->dzr, a->rowacc, a->GEV, a->Gph, a->gs,
                           hot));
    if (a->ev_tile1) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_tile1, hot));
    STEP_TRY(spmf_rows_finish(a->rowsum, a->lgam, a->inv_xi, a->scale_rows, a->nrows, K, S, a->vsum, a->z, a->dzr,
                              a->rowacc, a->gs, hot));
  }
  // exact guard of poisson.py:606-616: if a row pass met a non-finite log-likelihood, the data term of
  // this step is re-evaluated densely with the reference's replacement semantics (conditional launch:
  // returns at once otherwise); dzr / rowacc are rewritten BEFORE the column side reads them
  const bool guard = a->gs && a->xdense;
  if (guard && a->dense_raw)
    STEP_TRY(spmf_guard_rows_fix_dense(a->dense_raw, a->dense_raw_dtype, hybrid ? a->rank : nullptr, a->rowsum, a->lgam,
                                       a->inv_xi, a->scale_rows, a->nrows, D, K, S, a->EV, a->PH, a->z, a->dzr,
                                       a->rowacc, a->xdense, a->gs, hot));
  else if (guard)
    STEP_TRY(spmf_guard_rows_fix(a->rowptr, a->cols, a->vals, a->rowsum, a->lgam, a->inv_xi, a->scale_rows, a->nrows,
                                 D, K, S, a->EV, a->PH, a->z, a->dzr, a->rowacc, a->xdense, a->gs, hot));
  if (a->ev_rows1) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_rows1, hot));
  // column sums of z and the batch totals: only the backward reads them -> next to the column side
  const bool cols_fork = hybrid && a->aux_stream1 && a->aux_stream2 && a->ev_aux_fork && a->ev_aux_join1 && a->ev_aux_join2;
  if (!cols_fork)
    STEP_TRY(spmf_batch_sums(a->z, a->rowacc, a->nrows, K, S, a->zcolsum, a->datasums, a->scr_d, hot));
  if (a->ev_cols0) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_cols0, hot));
  if (!hybrid) {
    STEP_TRY(spmf_csc_cols(a->colptr, a->crows, a->cvals, a->nnz, a->nrows, D, K, S, a->z, a->dzr, a->EV, a->PH,
                           a->GAp, a->GEV, a->Gph, 0, hot));
  } else {
    // two independent accumulations into the column-gradient tables (zeroed before the tile kernel,
    // which has added GEV / Gphi of the covered entries):
    //   GA'[0:H] += X_hot^T . dzr                     -- tcgen05 GEMM, aux stream 1
    //   cold CSC (the uncovered entries): GEV, Gphi, GA'  -- gather kernel, aux stream 2
    const int H = a->hot_cols;
    const int Bp = (a->nrows + 127) / 128 * 128;     // whole 128-row tiles of the count block
    const bool fork = cols_fork;
    cudaStream_t s1 = fork ? (cudaStream_t)a->aux_stream1 : hot;
    cudaStream_t s2 = fork ? (cudaStream_t)a->aux_stream2 : hot;
    if (fork) {
      CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_aux_fork, hot));
      CUDA_TRY(cudaStreamWaitEvent(s1, (cudaEvent_t)a->ev_aux_fork, 0));
      CUDA_TRY(cudaStreamWaitEvent(s2, (cudaEvent_t)a->ev_aux_fork, 0));
    }
    if (fork) STEP_TRY(spmf_batch_sums(a->z, a->rowacc, a->nrows, K, S, a->zcolsum, a->datasums, a->scr_d, s1));
    if (a->ev_gemm0) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_gemm0, s1));
    STEP_TRY(spmf_split3_transpose(a->dzr, REC, (long long)a->nrows * REC, a->nrows, Bp, REC, a->dzrT3,
                                   a->t3_qstride, NQ, s1));
    // X_hot^T is never built: the GEMM reads the X tiles as an MN-major operand
    STEP_TRY(spmf_umma_gemm3_at(a->xhot, (H + 63) / 64 * 64, a->nrows, H, a->dzrT3, a->t3_qstride, a->GAp, REC,
                                (long long)D * REC, REC, NQ, a->gemm_splits, s1));
    if (a->ev_gemm1) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_gemm1, s1));
    STEP_TRY(spmf_csc_cols_accum(a->colptr, a->crows, a->cvals, a->nnz, a->nrows, D, K, S, a->z, a->dzr, a->EV,
                                 a->PH, a->GAp, a->GEV, a->Gph, s2));
    if (fork) {
      CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_aux_join1, s1));
      CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_aux_join2, s2));
      CUDA_TRY(cudaStreamWaitEvent(hot, (cudaEvent_t)a->ev_aux_join1, 0));
      CUDA_TRY(cudaStreamWaitEvent(hot, (cudaEvent_t)a->ev_aux_join2, 0));
    }
  }
  if (guard)        // ... and GEV / Gphi after it (GA' was computed from the fixed dzr)
    STEP_TRY(spmf_guard_cols_fix(a->nrows, D, K, S, a->EV, a->PH, a->z, a->GEV, a->Gph, a->xdense, a->gs, hot));
  if (a->ev_cols1) CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_cols1, hot));
  }   // sparse / tensor-core data term
  if (side != hot) CUDA_TRY(cudaStreamWaitEvent(hot, (cudaEvent_t)a->ev_join, 0));
  if (split_bwd)
    STEP_TRY(spmf_backward_post_m(a->params, a->noise, a->eta, hybrid ? a->rank : nullptr, D, K, S, a->GAp, a->GEV,
                                  a->Gph, a->zcolsum, a->datasums, a->phisum, (float)a->nrows, a->u_tau_scale,
                                  a->s_tau_scale, a->decay, a->w_entropy, a->w_prior, a->world_size, a->grads,
                                  a->parts, a->scr_f, a->scr_dpre, a->gs, a->model, hot));
  else
    STEP_TRY(spmf_backward_params_ranked_m(a->params, a->noise, a->dgda, a->eta, hybrid ? a->rank : nullptr, D, K, S,
                                           a->GAp, a->GEV, a->Gph, a->zcolsum, a->datasums, a->phisum,
                                           (float)a->nrows, a->u_tau_scale, a->s_tau_scale, a->decay, a->w_entropy,
                                           a->w_prior, a->world_size, a->grads, a->parts, a->scr_f, a->scr_d, a->gs,
                                           a->model, hot));
  if (a->adam_lr > 0.f && a->world_size > 1) {
    // the exchange must come between the backward and the Adam step of the data-touched block: only the
    // early tail step may run inside this call
    if (!tail_early) return SPMF_ERR_BAD_ARG;
  } else if (a->adam_lr > 0.f) {
    // the scalar slack inside the gradient block is host-side bookkeeping, not a parameter gradient
    CUDA_TRY(cudaMemsetAsync(a->grads + a->comm_off, 0, (size_t)a->comm_slack * sizeof(float), hot));
    STEP_TRY(spmf_adam_step_dev(a->params, a->grads, a->adam_m, a->adam_v, tail_early ? a->comm_off : a->n_params,
                                a->adam_lr, a->adam_beta1, a->adam_beta2, a->adam_eps, a->adam_t, a->clip_value, 1.0f,
                                a->step_state, hot));
  }
  if (hot != caller) {
    CUDA_TRY(cudaEventRecord((cudaEvent_t)a->ev_done, hot));
    CUDA_TRY(cudaStreamWaitEvent(caller, (cudaEvent_t)a->ev_done, 0));
  }
  return SPMF_OK;
}

// ---- graph replay ------------------------------------------------------------------------------------
// The captured graph holds every kernel / memset / cross-stream dependency of one step EXCEPT the kernel
// that writes the per-step scalars: that one is launched eagerly right before each replay, so the
// executable graph itself is never modified (updating a kernel node's arguments before every launch
// made the replay re-upload the graph and was slower than the eager multi-stream launch).
struct StepGraph {
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  void* state_dst = nullptr;
};

int spmf_step_graph_create(const spmf_step_args* a_in, void** handle) {
  if (!a_in || !handle || !a_in->step_state) return SPMF_ERR_BAD_ARG;
  // the legacy default stream (0) cannot be captured: record the sequence with the hot stream as its
  // origin instead (the replay may still be launched into any stream, the default one included)
  spmf_step_args copy = *a_in;
  copy.state_preset = 1;
  if (!copy.caller_stream) {
    if (!copy.hot_stream) return SPMF_ERR_UNSUPPORTED;
    copy.caller_stream = copy.hot_stream;
  }
  const spmf_step_args* a = &copy;
  if (a->ev_rows0 || a->ev_rows1 || a->ev_cols0 || a->ev_cols1 || a->ev_gemm0 || a->ev_gemm1 || a->ev_tile0 ||
      a->ev_tile1)
    return SPMF_ERR_BAD_ARG;                      // timing events are recorded outside graphs only
  cudaStream_t caller = (cudaStream_t)a->caller_stream;
  StepGraph* g = new StepGraph();
  cudaError_t e = cudaStreamBeginCapture(caller, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) { delete g; return (int)e; }
  const int rc = spmf_advi_step(a);
  e = cudaStreamEndCapture(caller, &g->graph);
  if (rc != SPMF_OK || e != cudaSuccess || !g->graph) {
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
    cudaGetLastError();
    return rc != SPMF_OK ? rc : (e != cudaSuccess ? (int)e : SPMF_ERR_UNSUPPORTED);
  }
  g->state_dst = a->step_state;
  e = cudaGraphInstantiate(&g->exec, g->graph, 0);
  if (e != cudaSuccess) {
    cudaGraphDestroy(g->graph);
    delete g;
    cudaGetLastError();
    return (int)e;
  }
  *handle = g;
  return SPMF_OK;
}

int spmf_step_graph_launch(void* handle, unsigned int rng_step, int adam_t, float lr, float beta1, float beta2,
                           float eps, float clip_value, void* stream) {
  StepGraph* g = (StepGraph*)handle;
  if (!g || !g->exec) return SPMF_ERR_BAD_ARG;
  STEP_TRY(spmf_step_state_set(g->state_dst, rng_step, adam_t, lr, beta1, beta2, eps, clip_value, stream));
  CUDA_TRY(cudaGraphLaunch(g->exec, (cudaStream_t)stream));
  return SPMF_OK;
}

int spmf_step_graph_destroy(void* handle) {
  StepGraph* g = (StepGraph*)handle;
  if (!g) return SPMF_OK;
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->graph) cudaGraphDestroy(g->graph);
  delete g;
  return SPMF_OK;
}

int spmf_prepare_batch(const unsigned short* cols16, const unsigned short* vals16, const long long* rowptr,
                       int* cols, float* vals, int nrows, long long nnz, int D, float* rowsum, float* lgam,
                       int* colptr, int* crows, float* cvals, int* scratch, void* stream) {
  if (cols16 || vals16) STEP_TRY(spmf_csr_unpack16(cols16, vals16, nnz, cols, vals, stream));
  STEP_TRY(spmf_csr_row_consts(rowptr, vals, nrows, rowsum, lgam, stream));
  return spmf_csr_to_csc(rowptr, cols, vals, nrows, D, colptr, crows, cvals, scratch, stream);
}

}  // extern "C"
