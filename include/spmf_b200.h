/* spmf_b200 -- C ABI of the B200-native ADVI step for sparse Poisson matrix factorisation.
 *
 * Drop-in boundary for ONE path of mederrata/spmf: the ELBO + gradient step of
 * `PoissonFactorization` (reference: mederrata_spmf/poisson.py, class at :25-717, energy at
 * :575-621, likelihood at :156-184, encoder at :623-701) and the slices of its un-vendored
 * training stack (bayesianquilts / TFP: surrogate sampling, log q, GradientTape backward, Adam)
 * that the step needs.  The reference is pure Python with no FFI; these are the entry points a
 * reference-side binding (ctypes, see INTEGRATION.md) would bind for that path.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its name ends in `_host`; the caller owns all memory;
 *  - no allocation, no global state, asynchronous on `stream` (a cudaStream_t passed as void*);
 *  - return 0 on success, a negative SPMF_ERR_* for bad arguments / unsupported configurations,
 *    or a positive cudaError_t if a launch failed;
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails;
 *  - `gs` (where present, may be NULL) = device guard state (see "dense evaluation" below): the row passes
 *    raise its flag when they meet a non-finite log-likelihood, the backward / loss-part kernels read it.
 *
 * Device layouts (KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S/SV; draw s = q*SV + sv):
 *   params / grads / adam moments : flat fp32, tensor offsets from spmf_layout()
 *                                   (order: v,w,u,s | u_eta,u_tau,s_eta,s_tau,u_eta_a,u_tau_a,s_eta_a,s_tau_a;
 *                                    each as (loc|conc_raw , scale_raw); v stored transposed as (D,K))
 *   noise                         : flat fp32 [var][s][elem]; N(0,1) for v,w,u,s, Gamma(alpha,1) otherwise
 *   Ap, EV, GAp, GEVnz            : [NQ][D][REC]      A' = a_d u_dk / eta_d,  EV = eta_d v_kd; REC = SV*KP floats,
 *                                                      element (sv,k) at spmf_rec_pos(KP,SV,sv,k)
 *   PH, Gphinz                    : [NQ][D][SV]       phi_d = eta_d b_d w_d
 *   z, dzr                        : [NQ][B][REC]      z_bk and r_b * dL/dz_bk (same record layout)
 *   rowacc                        : [NQ][B][4][SV]    per-row (sum x log lam - lgamma, z.vsum, |z|^2, #non-finite)
 */
#ifndef SPMF_B200_H
#define SPMF_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define SPMF_OK 0
#define SPMF_ERR_BAD_ARG (-1)
#define SPMF_ERR_UNSUPPORTED (-2)
#define SPMF_ERR_PEER_TIMEOUT (-3)   /* a peer rank never reached the step's exchange (spmf_p2p_status) */
#define SPMF_MAX_K 512        /* latent dimensions of the gather and dense paths */
#define SPMF_MAX_TILE_K 128   /* latent dimensions of the tensor-core (tcgen05) hybrid path */
#define SPMF_NUM_TENSORS 24
#define SPMF_NUM_VARS 12
#define SPMF_NUM_PARTS 16

/* ---- layout helpers (host only, no device work) ---- */
int spmf_kpad(int K);       /* latent dim padded to a power of two */
int spmf_draw_vec(int S);   /* draws processed per vector lane: 4, 2 or 1 (the rule for K <= 128) */
/* draws per gather record for latent dim K: the largest SV in {4,2,1} that divides S with
 * spmf_kpad(K)*SV <= 512 floats.  Equals spmf_draw_vec(S) for K <= 128; every layout below uses it. */
int spmf_draw_vec_k(int K, int S);
/* position of (draw sv, latent k) inside one SV*KP-float gather record (k-vector-major, see
 * csrc/spmf_record.cuh); negative on bad arguments. */
int spmf_rec_pos(int KP, int SV, int sv, int k);
/* tensor_offsets[25], noise_offsets[13] in floats.  Replaces the variable bookkeeping of
 * create_distributions (poisson.py:403-573: surrogate_vars / var_list). */
int spmf_layout(int D, int K, int S, long long* tensor_offsets_host, long long* noise_offsets_host);
long long spmf_backward_scratch_floats(int D, int K, int S);
long long spmf_backward_scratch_doubles(int D, int K, int S);

/* ---- surrogate sampling [EXT L3: surrogate_distribution.sample(S)], poisson.py:403-573 ---- */
#define SPMF_NOISE_NORMAL 1 /* N(0,1) base draws of v, w, u, s */
#define SPMF_NOISE_GAMMA 2  /* Gamma(alpha,1) draws of the 8 InverseGamma-based variables */
int spmf_fill_noise(float* noise, const float* params, int D, int K, int S,
                    unsigned long long seed, unsigned int step, int which, void* stream);
int spmf_sample(const float* params, const float* noise, int D, int K, int S, float* samples,
                void* stream);
/* encoding_matrix / intercept_matrix / decoding_matrix for every draw (poisson.py:652-701),
 * plus vsum[NQ][SV][KP] = sum_d EV and phisum[NQ][SV] = sum_d PH for the closed-form -sum(rate). */
int spmf_draw_operands(const float* params, const float* noise, const float* eta, int D, int K, int S,
                       float* Ap, float* EV, float* PH, double* vsum, double* phisum,
                       double* scratch, void* stream);

/* ---- data term, sparse counts (poisson.py:156-184 log_likelihood_components, :597-618 z prior +
 *      reduce, :623-650 encode) and its backward ---- */
/* per-row constants of a CSR shard: rowsum[r] = sum_d x, lgam[r] = sum_d lgamma(x+1) */
int spmf_csr_row_consts(const long long* rowptr, const float* vals, long long nrows, float* rowsum,
                        float* lgam, void* stream);
/* row pass: z = r_b * x.A' ; lambda at nonzeros ; dz ; per-row scalars.  r_b = rowsum*inv_xi if
 * scale_rows else 1.  `rowptr` points at the first row of the batch; offsets index cols/vals. */
int spmf_csr_rows(const long long* rowptr, const int* cols, const float* vals, const float* rowsum,
                  const float* lgam, float inv_xi, int scale_rows, int nrows, int D, int K, int S,
                  const float* Ap, const float* EV, const float* PH, const double* vsum, float* z,
                  float* dzr, float* rowacc, int variant, void* gs, void* stream);
/* encode only (inference): z[NQ][B][SV][KP] */
int spmf_csr_encode(const long long* rowptr, const int* cols, const float* vals, const float* rowsum,
                    float inv_xi, int scale_rows, int nrows, int D, int K, int S, const float* Ap,
                    float* z, void* stream);
/* column pass over the CSC copy of the same batch (rows are batch-local): accumulates into
 * GAp, GEVnz, Gphinz, which this call zeroes first. */
int spmf_csc_cols(const int* colptr, const int* rows, const float* vals, int nnz, int nrows, int D,
                  int K, int S, const float* z, const float* dzr, const float* EV, const float* PH,
                  float* GAp, float* GEVnz, float* Gphinz, int variant, void* stream);
/* sums over the rows of the batch: zcolsum[NQ][SV][KP], datasums[NQ][4][SV] */
int spmf_batch_sums(const float* z, const float* rowacc, int nrows, int K, int S, double* zcolsum,
                    double* datasums, double* scratch, void* stream);

/* Optimiser step arguments [EXT L4: tf.optimizers.Adam + clip in bayesianquilts' loop] of the fused
 * multi-GPU tail (spmf_unpack_adam). */
typedef struct spmf_adam_args {
  float lr, beta1, beta2, eps, clip_value, grad_scale;
  int step;          /* 1-based optimiser step (bias correction) */
  int reserved;
  float *params, *m, *v;
} spmf_adam_args;

/* ---- backward to the 24 variational tensors + loss parts [EXT L3/L4 GradientTape] ----
 * parts[S][16]: 12 prior terms in the reference's var_list order (poisson.py:572), log q, 'z', 'x'
 * (the dict of unormalized_log_prob_parts, poisson.py:582-621), [15] = per-draw loss. */
/* dgda[var][s][elem] (noise layout, Gamma variables only) = d g / d alpha of every Gamma draw:
 * the implicit-reparameterisation gradient tf.random.gamma supplies in the reference stack [EXT]. */
int spmf_gamma_grad(const float* params, const float* noise, int D, int K, int S, float* dgda,
                    void* stream);
/* Gamma draws (same Philox stream as spmf_fill_noise) and their implicit gradients in one pass */
int spmf_gamma_draw_grad(const float* params, float* noise, float* dgda, int D, int K, int S,
                         unsigned long long seed, unsigned int step, void* stream);
int spmf_backward_params(const float* params, const float* noise, const float* dgda, const float* eta,
                         int D, int K, int S, const float* GAp, const float* GEVnz, const float* Gphinz,
                         const double* zcolsum, const double* datasums, const double* phisum,
                         float batch_rows, float u_tau_scale, float s_tau_scale, float decay,
                         float w_entropy, float w_prior, int world_size, float* grads, double* parts,
                         float* scratch_f, double* scratch_d, void* gs, void* stream);

/* The same backward in two halves: `pre` = everything that does not depend on the data term (prior +
 * entropy gradients of all 24 tensors, the loss parts) -- it can run on a side stream while the data
 * term is being evaluated; `post` = the data half (u, v, w, s) + parts.  pre then post ==
 * spmf_backward_params_ranked (the gradient is linear in the upstream data terms).  scr_d must not be
 * shared with the reductions of the data term if the two run concurrently. */
int spmf_backward_pre(const float* params, const float* noise, const float* dgda, const float* eta, int D, int K,
                      int S, float batch_rows, float u_tau_scale, float s_tau_scale, float decay, float w_entropy,
                      float w_prior, int world_size, float* grads, float* scr_f, double* scr_d, void* stream);
int spmf_backward_post(const float* params, const float* noise, const float* eta, const int* rank, int D, int K,
                       int S, const float* GAp, const float* GEVnz, const float* Gphinz, const double* zcolsum,
                       const double* datasums, const double* phisum, float batch_rows, float u_tau_scale,
                       float s_tau_scale, float decay, float w_entropy, float w_prior, int world_size,
                       float* grads, double* parts, float* scr_f, const double* scr_d, void* gs, void* stream);

/* ---- optimiser [EXT L4: Adam + clip in bayesianquilts' batched_minimize] ---- */
int spmf_adam_step(float* params, const float* grads, float* m, float* v, long long n, float lr,
                   float beta1, float beta2, float eps, int step, float clip_value, float grad_scale,
                   void* stream);
int spmf_sumsq(const float* g, long long n, float* tmp, double* out, double* scratch, void* stream);
/* multi-GPU: after the all-reduce of the gradient block, fold the summed ('z','x') (hi,lo) float pairs
 * in the block's scalar slack back into parts[S][16], recompute the per-draw loss ([15]), write the
 * mean loss, zero the slack.  S <= 64. */
int spmf_unpack_parts(float* comm_slack, int slack_floats, int S, float w_entropy, float w_prior, double* parts,
                      double* loss_out, void* stream);
/* the same plus Adam over grads[0, n_data) (the whole flat buffer), one launch: the multi-GPU tail */
int spmf_unpack_adam(float* comm_slack, int slack_floats, int S, float w_entropy, float w_prior, double* parts,
                     double* loss_out, const float* grads, long long n_data, const spmf_adam_args* adam,
                     void* stream);
int spmf_colsum(const float* in, long long n, int c, int q, double* out, double* scratch, void* stream);
/* the same over fp64 input: out[q][c] = sum over rows of in[q][n][c] in a fixed order; scratch: 64*q*c doubles */
int spmf_colsum_f64(const double* in, long long n, int c, int q, double* out, double* scratch, void* stream);

/* ---- multi-GPU tail over NVLink peer memory (net-new, SURVEY.md 8e; replaces ncclAllReduce -> spmf_unpack_adam) ----
 * One process per GPU.  Gradient, parameter and flag buffers come from spmf_p2p_alloc (cudaMalloc, zeroed) and
 * are mapped into the peers with CUDA IPC: spmf_p2p_export fills a 64-byte handle, the host exchanges the
 * handles once, spmf_p2p_open maps a peer's buffer (peer access enabled lazily).
 * spmf_p2p_reduce_adam -- ONE kernel per step and rank: wait for every rank's gradients; for this rank's 1/world
 * slice of the block [0, comm_off) add the world partial gradients in rank order (16-byte peer loads), apply Adam
 * (moments live on the owner only) and store the new values into every rank's parameter buffer; Adam on the
 * replicated tensors [n_block, n_params) locally; fold the ('z','x') (hi,lo) pairs of all ranks into parts /
 * loss_out (as spmf_unpack_parts); leave when every peer's stores have landed, then zero the local slack.
 * `epoch` must increase by one per call (same value on every rank).  Waits are bounded (~10 s): a missing peer
 * sets a status word (spmf_p2p_status -> SPMF_ERR_PEER_TIMEOUT) instead of hanging the device. */
#define SPMF_P2P_MAX_WORLD 8
#define SPMF_P2P_HANDLE_BYTES 64
typedef struct spmf_p2p_args {
  int world, rank, S, slack;           /* slack = floats of bookkeeping at the end of the reduced block */
  unsigned int epoch;
  int skip_tail;                       /* 1: the replicated tensors were already stepped (adam_tail_early) */
  long long n_params, n_block, comm_off;   /* n_block = comm_off + slack */
  double w_entropy, w_prior;
  float* grads[SPMF_P2P_MAX_WORLD];    /* [q] = rank q's gradient buffer as mapped in THIS process */
  float* params[SPMF_P2P_MAX_WORLD];
  void* flags[SPMF_P2P_MAX_WORLD];     /* spmf_p2p_flag_bytes() each, zeroed once before the first call */
  double* parts;                       /* [S][16] local */
  double* loss_out;
  const spmf_adam_args* adam;          /* params = params[rank]; lr = 0: reduce + parts only */
} spmf_p2p_args;
int spmf_p2p_alloc(long long bytes, void** ptr);
int spmf_p2p_free(void* ptr);
int spmf_p2p_export(void* ptr, unsigned char* handle64);
int spmf_p2p_open(const unsigned char* handle64, void** ptr);
int spmf_p2p_close(void* ptr);
long long spmf_p2p_flag_bytes(void);
int spmf_p2p_status(const void* flags, void* stream);
int spmf_p2p_reduce_adam(const spmf_p2p_args* args, void* stream);
/* Host-only: the floats [*lo, *hi) of the reduced block [0, comm_off) whose sum, Adam update and moments belong
 * to `rank` in spmf_p2p_reduce_adam (comm_off a multiple of 4, 1 <= world <= SPMF_P2P_MAX_WORLD).  The ranges of
 * ranks 0..world-1 follow each other and cover the block once; a rank may own an empty range.  With the
 * peer-memory exchange, adam_m / adam_v of a rank are current only inside its own range: a checkpoint gathers
 * them by it. */
int spmf_p2p_owned_range(long long comm_off, int world, int rank, long long* lo, long long* hi);

/* ---- data formats either side of the path ---- */
/* compute_scales (poisson.py:113-154): colsum[D] (double) and colnnz[D] (float, as the reference
 * accumulates the non-zero counter in fp32) over a CSR shard; accumulates (caller zeroes). */
int spmf_csr_colstats(const int* cols, const float* vals, long long nnz, int D, double* colsum,
                      float* colnnz, void* stream);
/* CSR batch -> CSC batch (colptr[D+1], rows batch-local).  scratch: spmf_csc_scratch_ints(D) ints. */
long long spmf_csc_scratch_ints(int D);
int spmf_csr_to_csc(const long long* rowptr, const int* cols, const float* vals, int nrows, int D,
                    int* colptr, int* rows_out, float* vals_out, int* scratch, void* stream);
/* compact transfer format of a CSR batch: uint16 column ids (D <= 65536) and / or uint16 counts,
 * widened on the device (either source may be NULL = that array was sent at full width). */
int spmf_csr_unpack16(const unsigned short* cols16, const unsigned short* vals16, long long nnz,
                      int* cols, float* vals, void* stream);
/* 2-byte transfer format: rowptr (zero-based, nrows+1) indexes two byte streams -- gaps8[j] = col_j - col_{j-1} - 1
 * within the row (col_{-1} = -1; wider gaps are bridged on the host by zero-valued entries) and vals8[j] = count,
 * 255 = "see the overflow list" (ovf_idx[i] = entry, ovf_val[i] = its count).  Expanded to int32 / fp32 here. */
int spmf_csr_unpack8(const long long* rowptr, const unsigned char* gaps8, const unsigned char* vals8, int nrows,
                     const int* ovf_idx, const float* ovf_val, int n_ovf, int* cols, float* vals, void* stream);
/* dense (B,D) fp32 counts -> CSR (rowptr[B+1] int64, cols, vals); two calls: count then fill. */
int spmf_dense_count(const float* x, int nrows, int D, long long* rowptr, void* stream);
int spmf_dense_fill(const float* x, int nrows, int D, const long long* rowptr, int* cols, float* vals,
                    void* stream);

/* ---- hybrid path: tcgen05 tensor-core GEMMs on the dense hot-column block + gathers elsewhere ----
 * The two products of the step that touch the counts only (encode x.A', poisson.py:640-643, and its
 * transpose GA' = x^T.dzr in the backward) run on the 5th-gen tensor cores for the H most
 * populated columns; so do the per-nonzero terms (rate, x/rate) of that block (spmf_hot_tile below),
 * while the gather kernels handle the remaining entries.
 * Column order: `rank[d]` = table row of feature d (descending column population), so the hot block
 * is rows [0,H) of every operand table.  All *_ranked entry points take rank == NULL as identity. */
/* 0: gather kernels, 2: tile-hybrid (GEMMs + fused tile kernel; KP in {8,16,32} with REC = KP*SV in
 * {32,64,128}, or KP in {64,128}).  Always 0 for K > SPMF_MAX_TILE_K: the tensor-core entry points of
 * the tile-hybrid step (spmf_hot_ev_tiles, spmf_hot_tile, spmf_csr_rows_cold, spmf_rows_finish,
 * spmf_csc_cols_accum) reject such K with SPMF_ERR_BAD_ARG. */
int spmf_hybrid_supported(int K, int S);
int spmf_draw_operands_ranked(const float* params, const float* noise, const float* eta, const int* rank,
                              int D, int K, int S, float* Ap, float* EV, float* PH, double* vsum,
                              double* phisum, double* scratch, void* stream);
/* the reduction half of spmf_draw_operands(_ranked) on its own (pass vsum = phisum = NULL there):
 * vsum[NQ][REC] = sum_d EV, phisum[NQ][SV] = sum_d PH in fp64 */
int spmf_operand_sums(const float* EV, const float* PH, int D, int K, int S, double* vsum, double* phisum,
                      double* scratch, void* stream);
int spmf_backward_params_ranked(const float* params, const float* noise, const float* dgda, const float* eta,
                                const int* rank, int D, int K, int S, const float* GAp, const float* GEVnz,
                                const float* Gphinz, const double* zcolsum, const double* datasums,
                                const double* phisum, float batch_rows, float u_tau_scale, float s_tau_scale,
                                float decay, float w_entropy, float w_prior, int world_size, float* grads,
                                double* parts, float* scr_f, double* scr_d, void* gs, void* stream);
/* Operands of the tcgen05 GEMM live in global memory "UMMA-tiled": tile by tile in the byte order the
 * tensor core reads from shared memory (K-major, no swizzle), so that a pipeline stage is two
 * contiguous TMA bulk copies.  A (bf16 counts): tiles [row/128][k/64] of 128 x 64; B3 (three bf16
 * terms of an fp32 operand): tiles [k/64][term] of N x 64.  Sizes / element offsets: */
long long spmf_umma_tiled_a_elems(long long M, long long Kd);          /* bf16 elements, M and Kd padded */
long long spmf_umma_tiled_b_elems(int N, long long Kd);
long long spmf_umma_tiled_a_index(long long row, long long k, long long Kd);
int spmf_umma_tile_a(const void* src_bf16, long long ld, int M, int Kd, void* dst, void* stream); /* row-major -> tiled */
/* CSR batch (original column ids) -> ranked + partitioned CSR (zero-based rowptr_out[nrows+1]; per row
 * the entries covered by the tensor-core products first, stored with a NEGATIVE value as their flag,
 * the others from rowmid[row] on) and the dense hot block as UMMA-tiled bf16: xhot = X[nrows][Hp]
 * (Hp = ceil64(H); every element of the 128-row-padded block is written here; size from
 * spmf_umma_tiled_a_elems).  Covered = rank < H and the count is exactly representable in bf16.
 * rowsum / lgam (both or neither): also emit the per-row constants of spmf_csr_row_consts in the same
 * pass. */
int spmf_hot_split(const long long* rowptr, const int* cols, const float* vals, int nrows, long long nnz,
                   const int* rank, int H, long long* rowptr_out, int* cols_out, float* vals_out, int* rowmid,
                   void* xhot, float* rowsum, float* lgam, void* stream);
/* the same, reading the 2-byte transfer format directly (spmf_csr_unpack8 fused in: column-gap bytes, count
 * bytes, sorted overflow list; entry indices relative to rowptr[0]) */
int spmf_hot_split_u8(const long long* rowptr, const unsigned char* gaps8, const unsigned char* vals8,
                      const int* ovf_idx, const float* ovf_val, int novf, int nrows, const int* rank, int H,
                      long long* rowptr_out, int* cols_out, float* vals_out, int* rowmid, void* xhot, float* rowsum,
                      float* lgam, void* stream);
/* the same, reading the compact upload format directly (spmf_csr_unpack16 fused in): exactly one of
 * cols / cols16 and one of vals / vals16 is non-NULL */
int spmf_hot_split_packed(const long long* rowptr, const int* cols, const unsigned short* cols16, const float* vals,
                          const unsigned short* vals16, int nrows, long long nnz, const int* rank, int H,
                          long long* rowptr_out, int* cols_out, float* vals_out, int* rowmid, void* xhot,
                          float* rowsum, float* lgam, void* stream);
/* Direct dense ingest: a dense [nrows][D] batch of counts in FEATURE order (dtype SPMF_DENSE_*) -> the hybrid
 * form without a CSR round trip: xhot = the UMMA-tiled bf16 block of the H hot columns (rank order), the row
 * constants, and the UNCOVERED nonzeros only (cold column, or a count not exact in bf16) as a ranked CSR with
 * rowmid = 0 -- what the tile-hybrid step reads.  cols_out / vals_out must hold the batch's nonzero count. */
#define SPMF_DENSE_U8 1
#define SPMF_DENSE_U16 2
#define SPMF_DENSE_F32 4
int spmf_dense_hot_split(const void* x, int dtype, int nrows, int D, const int* rank, int H, long long* rowptr_out,
                         int* cols_out, float* vals_out, int* rowmid, void* xhot, float* rowsum, float* lgam,
                         void* stream);
/* fp32 src[NQ][R][C] (row stride lds) -> UMMA-tiled B3 operand dst[NQ] with k = source row (i.e. the
 * transpose), hi+mid+lo = src to 24 bits; k in [R, Rpad) is written as zeros.  C % 32 == 0, Rpad % 64 == 0. */
int spmf_split3_transpose(const float* src, long long lds, long long src_qstride, int R, int Rpad, int C,
                          void* dst3, long long dst_qstride, int NQ, void* stream);
/* C[q][M][N] (fp32, row stride ldc, accumulated with atomics) += A[q] (UMMA-tiled, M x Kd)
 * * (B3[q] hi+mid+lo)^T (UMMA-tiled, N x Kd) on tcgen05; N in {32,64,128,256,512}, Kd % 64 == 0,
 * `splits` = split-K factor (<= 0: automatic). */
int spmf_umma_gemm3(const void* A, long long a_qstride, int M, const void* B3, long long b_qstride, float* C,
                    long long ldc, long long c_qstride, int N, int Kd, int NQ, int splits, void* stream);
/* C[q][M][N] += X^T . (B3[q] hi+mid+lo)^T with X = the UMMA-tiled counts X[x_rows][x_kd] read as an
 * MN-major operand (M = its columns, first M of them; K = its rows): GA' = X_hot^T . dzr without a
 * transposed copy of the counts.  B3 is UMMA-tiled over k = rows of X, padded to a multiple of 128. */
int spmf_umma_gemm3_at(const void* X, int x_kd, int x_rows, int M, const void* B3, long long b_qstride, float* C,
                       long long ldc, long long c_qstride, int N, int NQ, int splits, void* stream);
/* bring-up probe: one CTA, raw shared-memory operand images, explicit descriptor fields (major-ness,
 * leading / stride byte offsets, byte step per k=16 MMA); dumps the 128-lane x N-column fp32
 * accumulator block to out[128][N].  Pins the UMMA conventions the kernels rely on (tests only). */
int spmf_umma_probe(const void* a_img, int a_bytes, const void* b_img, int b_bytes, int M, int N, int a_mn,
                    int b_mn, int lbo_a, int sbo_a, int step_a, int lbo_b, int sbo_b, int step_b, int nk,
                    float* out, void* stream);
/* ---- tile-hybrid step: the per-nonzero terms of the hot block on the tensor cores as well ----
 * spmf_hot_tile fuses, per 128-row x 64-column tile and draw: rate = z.EV + phi (tcgen05.mma into
 * tensor memory), x log rate and w = x/rate on the CUDA cores, then dz += w.EV and GEV = w^T.z,
 * Gphi = w^T.1 as two more MMAs -- the (S,B,D) rate tensor of poisson.py:174-184 never exists.
 * Order: spmf_hot_ev_tiles (per step) ; spmf_csr_rows_cold (z final, raw cold partials) ;
 * spmf_hot_tile (adds the hot block into dzacc / rowacc, atomics into GEVnz / Gphinz, which must be
 * zeroed before) ; spmf_rows_finish (dzr = r (dz - vsum - z), per-row scalars). */
long long spmf_hot_tile_scratch_bytes(int H, int K, int S);   /* size of the EVt workspace */
int spmf_hot_ev_tiles(const float* EV, const float* PH, int D, int H, int K, int S, void* EVt, void* stream);
int spmf_csr_rows_cold(const long long* rowptr, const int* cols, const float* vals, const int* rowmid,
                       const float* rowsum, float inv_xi, int scale_rows, int nrows, int D, int K, int S,
                       const float* Ap, const float* EV, const float* PH, float* z, float* dzacc, float* rowacc,
                       void* gs, void* stream);
int spmf_hot_tile(const void* xhot, const void* EVt, const float* z, int nrows, int D, int H, int K, int S,
                  float* dzacc, float* rowacc, float* GEVnz, float* Gphinz, void* gs, void* stream);
int spmf_rows_finish(const float* rowsum, const float* lgam, float inv_xi, int scale_rows, int nrows, int K, int S,
                     const double* vsum, const float* z, float* dzr, float* rowacc, void* gs, void* stream);
/* column side of the tile-hybrid step, in pieces that callers overlap on several streams: zero the three
 * column-gradient tables; accumulate (atomics) the CSC copy of the uncovered entries into them (full
 * column pass; GA' of the covered entries comes from spmf_umma_gemm3_at).  nnz_bound >= the copy's count
 * (the count itself is colptr[D], device side). */
int spmf_zero_col_grads(float* GAp, float* GEVnz, float* Gphinz, int D, int K, int S, void* stream);
int spmf_csc_cols_accum(const int* colptr, const int* rows, const float* vals, int nnz_bound, int nrows, int D,
                        int K, int S, const float* z, const float* dzr, const float* EV, const float* PH,
                        float* GAp, float* GEVnz, float* Gphinz, void* stream);
/* CSC copy of ONE part of a partitioned CSR (spmf_hot_split): part 0 = the first rowmid[r] entries of
 * every row, part 1 = the rest; values are stored as |x|.  rowmid == NULL: whole rows. */
int spmf_csr_to_csc_part(const long long* rowptr, const int* rowmid, int part, const int* cols, const float* vals,
                         int nrows, int D, int* colptr, int* rows_out, float* vals_out, int* scratch,
                         void* stream);

/* ---- per-step scalars on the device (CUDA-graph replay of a step) ----
 * A captured step freezes its kernel arguments, so what changes per step (Philox step, Adam step / rates)
 * is read from a small device struct (spmf_step_state_bytes()) by the `_dev` variants below; a NULL state
 * means "use the arguments".  spmf_step_state_set is the kernel that writes it. */
int spmf_step_state_bytes(void);
int spmf_step_state_set(void* step_state, unsigned int rng_step, int adam_t, float lr, float beta1, float beta2,
                        float eps, float clip_value, void* stream);
const void* spmf_step_state_kernel_ptr(void);
int spmf_step_state_value(unsigned int rng_step, int adam_t, float lr, float beta1, float beta2, float eps,
                          float clip_value, void* out36);
int spmf_fill_noise_dev(float* noise, const float* params, int D, int K, int S, unsigned long long seed,
                        unsigned int step, int which, const void* step_state, void* stream);
int spmf_gamma_draw_grad_dev(const float* params, float* noise, float* dgda, int D, int K, int S,
                             unsigned long long seed, unsigned int step, const void* step_state, void* stream);
int spmf_adam_step_dev(float* params, const float* grads, float* m, float* v, long long n, float lr, float beta1,
                       float beta2, float eps, int step, float clip_value, float grad_scale,
                       const void* step_state, void* stream);

/* ---- one call per step / per uploaded batch ----
 * spmf_advi_step issues the whole sequence above (noise, Gamma gradients, operands, row pass, sums,
 * column pass, backward, optional Adam) from native code.  Streams: `caller_stream` is the stream
 * the caller orders its work on; if `hot_stream` / `side_stream` are given (with the three events)
 * the data-term path runs on `hot_stream`, the Gamma work on `side_stream`, fork/join by events,
 * and `caller_stream` waits for the result.  The ev_rows/ev_cols events, if non-NULL, bracket the
 * two hot kernels (bench instrumentation).  adam_lr <= 0 skips the optimiser (multi-GPU: all-reduce
 * the gradient block first, then call spmf_adam_step). */
typedef struct spmf_step_args {
  /* model */
  int D, K, S, world_size;
  float u_tau_scale, s_tau_scale, decay, w_entropy, w_prior;
  float inv_xi;
  int scale_rows;
  /* noise */
  int fresh_noise;
  unsigned int rng_step;
  unsigned long long seed;
  /* flat buffers */
  float *params, *grads, *adam_m, *adam_v, *noise, *dgda;
  const float* eta;
  long long n_params, comm_off, comm_slack;
  /* workspace */
  float *Ap, *EV, *PH, *GAp, *GEV, *Gph, *z, *dzr, *rowacc, *scr_f;
  double *vsum, *phisum, *zcolsum, *datasums, *parts, *scr_d;
  /* batch */
  const long long* rowptr;
  const int* cols;
  const float* vals;
  const float *rowsum, *lgam;
  const int *colptr, *crows;
  const float* cvals;
  int nrows, nnz;
  /* optimiser: adam_lr > 0 (world_size == 1 only) ends the step with spmf_adam_step; with several ranks
   * the caller all-reduces the gradient block first and then calls spmf_unpack_adam */
  float adam_lr, adam_beta1, adam_beta2, adam_eps, clip_value;
  int adam_t;
  /* streams / events (cudaStream_t / cudaEvent_t) */
  void *caller_stream, *hot_stream, *side_stream;
  void *ev_fork, *ev_join, *ev_done;
  void *ev_rows0, *ev_rows1, *ev_cols0, *ev_cols1;
  /* hybrid path (hot_cols > 0): rowptr/cols/vals above are the ranked, partitioned CSR of spmf_hot_split
   * (rowptr zero-based) and colptr/crows/cvals the CSC of its uncovered entries; rank maps feature -> table row */
  const int* rank;
  int hot_cols, gemm_splits;
  long long t3_qstride;            /* elements between draw groups in ApT3 / dzrT3 */
  const int* rowmid;
  const void* xhot;                /* UMMA-tiled bf16 hot block (spmf_hot_split) */
  void *ApT3, *dzrT3;              /* UMMA-tiled bf16 B3 workspaces, [NQ] x spmf_umma_tiled_b_elems */
  void *ev_gemm0, *ev_gemm1;       /* optional events around the tensor-core launches of the column side */
  /* optional: two more streams (+ three events) on which the GA' GEMM and the cold column pass run
   * concurrently; NULL = everything in order on the hot stream */
  void *aux_stream1, *aux_stream2;
  void *ev_aux_fork, *ev_aux_join1, *ev_aux_join2;
  /* the per-nonzero terms of the hot block run in the fused tcgen05 tile kernel (spmf_hot_tile);
   * EVt = its workspace of spmf_hot_tile_scratch_bytes (required when hot_cols > 0) */
  void* EVt;
  void *ev_tile0, *ev_tile1;       /* optional events around spmf_hot_tile (bench instrumentation) */
  /* split backward: with scr_dpre (a second double scratch of spmf_backward_scratch_doubles) and
   * ev_noise given, the data-independent half of the backward runs on the side stream under the data
   * term; otherwise the one-pass backward runs after it */
  double* scr_dpre;
  void* ev_noise;
  /* link function and exact guard: link = SPMF_LINK_*; gs = device guard state (spmf_guard_state_bytes());
   * xdense = scratch of nrows*D floats (touched only when the guard fires, or every step by the dense
   * links); xdense_in = optional dense fp32 [nrows][D] batch in feature order (dense links: used
   * instead of scattering the CSR).  gs == NULL or xdense == NULL: non-finite entries are dropped and
   * counted, not replaced.  `eta` above is [2][D] (decoder scale | encoder divisor). */
  int link;
  void* gs;
  float* xdense;
  const float* xdense_in;
  /* optional device step state (spmf_step_state_bytes()): when given, the step starts by writing
   * (rng_step, adam_t, adam_*) into it and the noise / Adam kernels read it -- required for graph replay */
  void* step_state;
  int model;          /* SPMF_MODEL_* */
  int state_preset;   /* != 0: step_state was already written on the stream (graph replay); leave 0 otherwise */
  /* batch ingested dense (spmf_dense_hot_split): rowptr / cols / vals hold the uncovered entries only, the raw
   * upload (feature order) is what the guard densifies from */
  const void* dense_raw;
  int dense_raw_dtype;
  /* 1: Adam on the tensors that never see a data term ([comm_off + comm_slack, n_params): their gradient is
   * final after the data-independent half of the backward) runs on the side stream under the data term; the
   * closing Adam then covers [0, comm_off) only.  Needs the split backward (scr_dpre) and adam_lr > 0.  With
   * world_size > 1 this is the only Adam the step applies -- the block [0, comm_off) belongs to the exchange
   * (spmf_p2p_reduce_adam with skip_tail = 1, or all-reduce + spmf_unpack_adam over n_data = comm_off + slack). */
  int adam_tail_early;
} spmf_step_args;
int spmf_advi_step(const spmf_step_args* args);
/* Replay of a whole step as ONE CUDA graph launch (all streams, events and kernels of spmf_advi_step):
 * create captures the sequence for one argument block (pointers, sizes and flags are frozen; args->step_state
 * must be set; kernel-timing events must be NULL), launch updates the per-step scalars and replays it
 * on `stream`.  The handle is owned by the caller.  Typical use: one graph per resident batch. */
int spmf_step_graph_create(const spmf_step_args* args, void** handle);
int spmf_step_graph_launch(void* handle, unsigned int rng_step, int adam_t, float lr, float beta1, float beta2,
                           float eps, float clip_value, void* stream);
int spmf_step_graph_destroy(void* handle);
/* widen a compact batch (either 16-bit source may be NULL), build its row constants and CSC copy */
int spmf_prepare_batch(const unsigned short* cols16, const unsigned short* vals16, const long long* rowptr,
                       int* cols, float* vals, int nrows, long long nnz, int D, float* rowsum, float* lgam,
                       int* colptr, int* crows, float* cvals, int* scratch, void* stream);

/* ---- model variants ----
 * SPMF_MODEL_BERNOULLI = BernoulliFactorization (bernoulli.py:31-649): v and w use an Identity bijector and
 * Normal(0, 0.1) / Normal(0, 1) priors (bernoulli.py:186-215) instead of Softplus + HalfNormal; everything
 * else (horseshoe+ hierarchy on u and s, surrogate families, var_list order) is shared.  The `_m`
 * variants take the model id; the plain entry points are the Poisson model. */
#define SPMF_MODEL_POISSON 0
#define SPMF_MODEL_BERNOULLI 1
int spmf_sample_m(const float* params, const float* noise, int D, int K, int S, float* samples, int model,
                  void* stream);
int spmf_draw_operands_ranked_m(const float* params, const float* noise, const float* eta, const int* rank,
                                int D, int K, int S, float* Ap, float* EV, float* PH, double* vsum,
                                double* phisum, double* scratch, int model, void* stream);
int spmf_backward_params_ranked_m(const float* params, const float* noise, const float* dgda, const float* eta,
                                  const int* rank, int D, int K, int S, const float* GAp, const float* GEVnz,
                                  const float* Gphinz, const double* zcolsum, const double* datasums,
                                  const double* phisum, float batch_rows, float u_tau_scale, float s_tau_scale,
                                  float decay, float w_entropy, float w_prior, int world_size, float* grads,
                                  double* parts, float* scr_f, double* scr_d, void* gs, int model, void* stream);
int spmf_backward_pre_m(const float* params, const float* noise, const float* dgda, const float* eta, int D, int K,
                        int S, float batch_rows, float u_tau_scale, float s_tau_scale, float decay, float w_entropy,
                        float w_prior, int world_size, float* grads, float* scr_f, double* scr_d, int model,
                        void* stream);
int spmf_backward_post_m(const float* params, const float* noise, const float* eta, const int* rank, int D, int K,
                         int S, const float* GAp, const float* GEVnz, const float* Gphinz, const double* zcolsum,
                         const double* datasums, const double* phisum, float batch_rows, float u_tau_scale,
                         float s_tau_scale, float decay, float w_entropy, float w_prior, int world_size,
                         float* grads, double* parts, float* scr_f, const double* scr_d, void* gs, int model,
                         void* stream);

/* ---- dense evaluation of the data term (csrc/spmf_dense.cu): link functions without a closed-form
 *      sum(rate) and the exact non-finite guard of poisson.py:606-616 ----
 * Links: linear Poisson (poisson.py:43,54,177-183), log_transform Poisson (poisson.py:41-42, 52-53),
 * Bernoulli-logit (bernoulli.py:148) with either decoder.  xd = the batch as dense fp32 [nrows][D] in
 * TABLE order (column = table row of the feature).  eta_enc[D] (table order) = the encoder divisor of
 * the log link (log(x/eta + 1)); the linear encoder's 1/eta is folded into A'.
 * The dense row pass finishes in place: dzr = r (dz - z), rowacc = (sum_d ll, 0, |z|^2, #non-finite);
 * no closed-form terms remain downstream (spmf_backward_* / parts are told through the guard state).
 * Guard state (spmf_guard_state_bytes() bytes on the device): flag bit 0 = a non-finite entry was met
 * this step, bit 1 = dense-only link; nbad; (min finite log-likelihood, its entry).  Reset before every
 * evaluation of the data term (spmf_guard_reset; the training step's last kernel does it for the next step). */
#define SPMF_LINK_POISSON 0
#define SPMF_LINK_POISSON_LOG 1
#define SPMF_LINK_BERNOULLI 2
#define SPMF_LINK_BERNOULLI_LOG 3
#define SPMF_DENSE_OPTIMISTIC 0 /* value + gradient, non-finite entries dropped and flagged */
#define SPMF_DENSE_STATS 1      /* count non-finite entries, find the smallest finite log-likelihood */
#define SPMF_DENSE_GUARDED 2    /* value + gradient with the reference's replacement (needs the statistics) */
int spmf_guard_state_bytes(void);
int spmf_guard_reset(void* gs, int flag, void* stream);
/* host-side decode of a copied-back guard state */
int spmf_guard_decode(const void* gs_host, int* flag, int* nbad, float* min_ll);
/* xd[nrows][D] = 0, then |vals| scattered at (row, cols[j]); cols must already be table rows */
int spmf_dense_scatter(const long long* rowptr, const int* cols, const float* vals, int nrows, int D, float* xd,
                       void* stream);
/* z = r_b sum_d enc(x_bd) A'_d  (poisson.py:623-650 with either encoder) */
int spmf_dense_encode(const float* xd, const float* eta_enc, const float* rowsum, float inv_xi, int scale_rows,
                      int nrows, int D, int K, int S, int link, const float* Ap, float* z, void* stream);
/* conditional != 0: the launch returns at once unless flag bit 0 is set */
int spmf_dense_rows(const float* xd, const float* rowsum, const float* lgam, float inv_xi, int scale_rows, int nrows,
                    int D, int K, int S, int link, int mode, int conditional, const float* EV, const float* PH,
                    const float* z, float* dzr, float* rowacc, void* gs, void* stream);
/* accumulates (atomics) GEV, Gphi and -- with_ga -- GA' = enc(x)^T . dzr into tables zeroed by the caller */
int spmf_dense_cols(const float* xd, const float* eta_enc, int nrows, int D, int K, int S, int link, int with_ga,
                    const float* z, const float* dzr, const float* EV, const float* PH, float* GAp, float* GEV,
                    float* Gph, const void* gs, void* stream);
/* The exact guard of the linear link as two conditional cooperative launches around the column side of
 * the sparse / tensor-core step (both return at once unless flag bit 0 is set): rows fix = densify the
 * batch into xd (scratch of nrows*D floats) -> statistics -> guarded dense row pass (overwrites dzr,
 * rowacc); columns fix = zero GEV / Gphi -> guarded dense column pass.  GA' needs no fix: the column
 * side computes it from the fixed dzr. */
int spmf_guard_rows_fix(const long long* rowptr, const int* cols, const float* vals, const float* rowsum,
                        const float* lgam, float inv_xi, int scale_rows, int nrows, int D, int K, int S,
                        const float* EV, const float* PH, const float* z, float* dzr, float* rowacc, float* xd,
                        void* gs, void* stream);
/* the same for a batch that was ingested dense (spmf_dense_hot_split): the batch is densified from the raw
 * dense upload (feature order, permuted by rank) instead of from a CSR */
int spmf_guard_rows_fix_dense(const void* raw, int raw_dtype, const int* rank, const float* rowsum, const float* lgam,
                              float inv_xi, int scale_rows, int nrows, int D, int K, int S, const float* EV,
                              const float* PH, const float* z, float* dzr, float* rowacc, float* xd, void* gs,
                              void* stream);
int spmf_guard_cols_fix(int nrows, int D, int K, int S, const float* EV, const float* PH, const float* z,
                        float* GEV, float* Gph, const float* xd, void* gs, void* stream);

/* ---- posterior predictive check (csrc/spmf_ppc.cu) ----
 * One pass over every (draw, row, feature) entry of a batch: the rate of the entry as the data term forms it
 * (any link; xd, z, EV, PH as for spmf_dense_rows, z from spmf_csr_encode / spmf_dense_encode), a replicate
 * x_rep ~ Poisson(rate) or Bernoulli(sigmoid(rate)) drawn from the Philox stream keyed by (seed, draw s,
 * global row = row_offset + local row, feature d) -- independent of the batch split, the launch geometry and the
 * training streams -- and its statistics:
 *   row_total[S][nrows] (sum_d x_rep), row_nnz[S][nrows], row_disc[S][nrows][2] = (D(x_rep), D(x)) in fp64
 *   summed in feature order, D = sum_d (y - rate)^2 / rate (Poisson) or (y - p)^2 / (p (1 - p)) (Bernoulli);
 *   disc_sum[S][2] = the sums of row_disc over the rows (fixed order; scratch: 128*S doubles);
 *   accumulated (zeroed by the caller): col_total / col_sumsq [S][D] (uint64), col_nnz [S][D] (uint32) by
 *   integer atomics, draw_max[S] (largest replicate) and draw_invalid[S] (entries whose Poisson rate is negative,
 *   not finite or above 2^24, or whose logit is not finite: replicate 0, left out of both discrepancies);
 *   out[S][nrows][D] (int32, may be NULL) = the replicates themselves.
 * Every output is bit-identical from run to run.  1 <= S <= SPMF_PPC_MAX_S, row_offset + nrows <= SPMF_PPC_MAX_ROW. */
#define SPMF_PPC_MAX_S 65535
#define SPMF_PPC_MAX_ROW (1LL << 48)
int spmf_ppc_rows(const float* xd, int nrows, int D, int K, int S, int link, const float* EV, const float* PH,
                  const float* z, unsigned long long seed, long long row_offset, long long* row_total, int* row_nnz,
                  double* row_disc, unsigned long long* col_total, unsigned long long* col_sumsq,
                  unsigned int* col_nnz, unsigned int* draw_max, unsigned long long* draw_invalid, int* out,
                  double* disc_sum, double* scratch, void* stream);
/* observed statistics of a CSR batch (column ids = features): row_total[nrows], row_nnz[nrows] written;
 * col_total[D], col_sumsq[D] (fp64, exact for integer counts) and col_nnz[D] accumulated (caller zeroes) */
int spmf_ppc_observed(const long long* rowptr, const int* cols, const float* vals, int nrows, int D,
                      double* row_total, int* row_nnz, double* col_total, double* col_sumsq, unsigned int* col_nnz,
                      void* stream);

/* ---- PSIS leave-one-out (csrc/spmf_loo.cu) ----
 * ll: row-major [nrows][ld] fp64 (ld >= S), ll[b][s] = log p(x_b | theta_s).  Per row b:
 * elpd[b] = PSIS-LOO log predictive density, lppd[b] = log mean_s exp(ll[b][s]), khat[b] = Pareto k-hat.
 * 1 <= S <= SPMF_LOO_MAX_S (8192).  Deterministic: bit-identical from run to run, and independent of nrows.
 *
 * The algorithm is ArviZ's _psislw / _gpdfit with r_eff = 1 (the surrogate draws are independent); all in fp64:
 *  1. r_s = -ll_s - max_s(-ll_s).  M = ceil(min(0.2 S, 3 sqrt(S))), capped at S - 1.  cutoff = max(r_(S-M),
 *     log(DBL_MIN)), r_(S-M) the (M+1)-th largest value; the tail is the n values strictly above the cutoff.
 *  2. n <= 4: khat = +inf, no smoothing.  Otherwise the generalised Pareto fit (Zhang & Stephens 2009, Vehtari's
 *     prior) to y = exp(tail) - exp(cutoff), ascending: m = 30 + floor(sqrt(n)) grid points
 *     b_j = 1/y_n + (1 - sqrt(m/(j - 1/2))) / (3 y_floor(n/4 + 1/2)), k_j = mean_i log1p(-b_j y_i),
 *     L_j = n (log(-b_j/k_j) - k_j - 1), w_j = 1 / sum_i exp(L_i - L_j) (an exp that overflows gives w_j = 0);
 *     w_j < 10 DBL_EPSILON is dropped and the rest renormalised; b = sum_j w_j b_j, k = mean_i log1p(-b y_i),
 *     sigma = -k/b, khat = (n k + 5)/(n + 10).
 *  3. If khat and sigma > 0 are finite, the i-th smallest tail value becomes
 *     log(sigma expm1(-khat log1p(-(i - 1/2)/n)) / khat + exp(cutoff)) (-log1p(-p) when |khat| < DBL_EPSILON), and
 *     every log weight is clamped at 0, the largest raw one.  Otherwise khat = +inf and the raw weights stay.
 *  4. lw = r - logsumexp(r); elpd = logsumexp(lw + ll); lppd = logsumexp(ll) - log S.
 *  5. A row holding -inf (and no NaN / +inf): elpd = -inf (the estimate 1/mean(1/p) = 0), khat = +inf, lppd as in 4.
 *     A row holding NaN or +inf: NaN in all three outputs. */
#define SPMF_LOO_MAX_S 8192
int spmf_psis_loo(const double* ll, long long ld, int nrows, int S, double* elpd, double* lppd, float* khat,
                  void* stream);
/* The same, and lw[b][s] (row stride ldw >= S) = the normalised log weights of step 4, smoothed and truncated, in
 * draw order (sum_s exp(lw[b][s]) = 1); a tied draw of the tail takes the smoothed weight a stable sort of the
 * log-ratios gives it.  Rows of step 5 (elpd not finite) get lw = NaN.  elpd, lppd and khat are bit-identical to
 * spmf_psis_loo's. */
int spmf_psis_loo_lw(const double* ll, long long ld, int nrows, int S, double* elpd, double* lppd, float* khat,
                     double* lw, long long ldw, void* stream);

/* ---- LOO-PIT (csrc/spmf_pit.cu, CDFs and binning in csrc/spmf_pit.cuh) ----
 * The probability integral transform of every entry under its row's leave-one-out predictive, non-randomised
 * (Czado, Gneiting & Held 2009) for counts.
 * spmf_loo_pit_accum: one chunk of S <= SPMF_LOO_PIT_MAX_DRAWS draws; xd, z, EV, PH as for spmf_ppc_rows (any link,
 * K <= SPMF_MAX_K); lw = the chunk's first column of spmf_psis_loo_lw's weights (lw[b * ldw + s], s < S).  For
 * every entry (b, d), adds in fp64
 *   acc[b][d][0] += sum_s exp(lw[b][s]) F(x_bd - 1 | theta_s),   acc[b][d][1] += sum_s exp(lw[b][s]) F(x_bd | theta_s)
 * with F the Poisson CDF of the rate (links 0, 1) or the Bernoulli CDF of the logit (links 2, 3) that link_rate
 * forms, and adds to inv[b][d] the draws at which the entry is invalid: a Poisson rate that is negative, not
 * finite or above 2^24, a logit that is not finite, or an observed value that is not an integer of the support
 * (0 <= x <= 2^24, or x in {0, 1} for Bernoulli).  Invalid draws add nothing to acc.  Within the chunk the draws
 * are added in ascending s, into the value acc held before the call: calling the chunks in order sums every entry
 * in one fixed order, independent of nrows, the batch split and the launch geometry, so acc is bit-identical from
 * run to run.  rate_out[S][nrows][D] (fp32, may be NULL) = the rate (or logit) of every entry.
 * spmf_loo_pit_hist: for every entry with inv == 0 and finite acc (a row of NaN weights is left out), the PIT
 * distribution F(u) = 0 (u <= P-), (u - P-)/(P+ - P-) (P- < u < P+), 1 (u >= P+) with P-, P+ = acc clamped to
 * [0, 1]; bin j = 0..J-1 gets F((j+1)/J) - F(j/J), or, if P+ <= P-, unit mass in bin min(J - 1, floor(P+ J)).
 * Adds (the caller zeroes) col_hist[D][J], col_n[D] (valid entries) and col_pit_sum[D] (sum of (P- + P+)/2).
 * The sums over the rows run in a fixed order (blocks of 1024 rows, then the blocks in order; no atomics), so the
 * outputs are bit-identical from run to run.  1 <= J <= SPMF_LOO_PIT_MAX_BINS; scratch: spmf_loo_pit_hist_scratch
 * _doubles(nrows, D, J) doubles. */
#define SPMF_LOO_PIT_MAX_DRAWS 64
#define SPMF_LOO_PIT_MAX_BINS 1000
int spmf_loo_pit_accum(const float* xd, int nrows, int D, int K, int S, int link, const float* EV, const float* PH,
                       const float* z, const double* lw, long long ldw, double* acc, int* inv, float* rate_out,
                       void* stream);
long long spmf_loo_pit_hist_scratch_doubles(int nrows, int D, int J);
int spmf_loo_pit_hist(const double* acc, const int* inv, int nrows, int D, int J, double* col_hist,
                      long long* col_n, double* col_pit_sum, double* scratch, void* stream);

const char* spmf_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SPMF_B200_H */
