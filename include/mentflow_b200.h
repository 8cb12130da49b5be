/*
 * mentflow_b200 -- C ABI of the B200-native MENT-Flow hot path.
 *
 * The reference (austin-hoover/ment-flow) is pure Python/PyTorch and has no FFI layer of
 * its own; the functions below are what a reference-side binding (ctypes, see
 * INTEGRATION.md) calls in place of the reference Python functions cited on each entry
 * (paths relative to the reference's `mentflow/` package, per-file line numbers).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to fp32 / int32 / int64 data owned by the caller
 *     (PyTorch tensors in the shipped host layer); row-major, contiguous, 16-byte aligned;
 *   - `stream` is a cudaStream_t passed as void*; nothing here allocates, synchronises or
 *     keeps global mutable state, so calls are safe from autograd worker threads;
 *   - return value: 0 on success, a cudaError_t code (>0) for CUDA failures,
 *     negative MFB_E_* for argument errors; mfb_error_string() decodes both;
 *   - workspaces are caller-allocated; query the size with the matching *_workspace_bytes.
 *   - there is no CPU implementation behind any entry point.
 */
#ifndef MENTFLOW_B200_H
#define MENTFLOW_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MFB_ABI_VERSION 5

#define MFB_E_BADARG (-1)      /* null pointer / non-positive size / unsupported shape   */
#define MFB_E_UNSUPPORTED (-2) /* combination not compiled (e.g. D > 8, hidden != 64)    */
#define MFB_E_WORKSPACE (-3)   /* workspace too small                                    */

/* per-call `flags` of the entry points that have a tensor-core and a CUDA-core implementation of the same
 * result (A/B tests, parity cross-checks).  There is no process-wide switch: the library keeps no mutable state. */
#define MFB_FLAG_NO_TENSOR_CORES 1

int mfb_abi_version(void);
const char* mfb_error_string(int code);
/* number of SMs of the current device (grid sizing is done inside the library) */
int mfb_sm_count(void);

/* ------------------------------------------------------------------------------------
 * Screen geometry of one 1-D projection, 8 floats per projection (device array [K][8]):
 *   [0] c0        first bin centre            (diagnostics/diagnostics.py:111 `coords`)
 *   [1] spacing   centre spacing, accurate: (c[B-1]-c[0])/(B-1) evaluated in float64
 *   [2] sigma     absolute kernel width       (diagnostics/diagnostics.py:113-114)
 *   [3] delta     the reference's fp32 c[1]-c[0] used in the normalisation
 *                 (diagnostics/histogram.py:40); differs from [1] by up to 1e-5 relative
 *   [4..7]        reserved (0)
 * 2-D screens use two consecutive records (x axis, then y axis).
 * ------------------------------------------------------------------------------------ */
#define MFB_GEOM_STRIDE 8

/* ---- fused linear projection + Gaussian KDE, 1-D screens ------------------------------
 * Replaces, for all K (transform, Histogram1D) pairs at once:
 *   simulate/simulate.py:29-33        for transform ...: u = transform(x.clone())
 *   simulate/transform.py:67-68       u = x @ M.T            (only the measured row)
 *   diagnostics/diagnostics.py:116-127  project -> kde_histogram_1d
 *   diagnostics/histogram.py:37-39    K_nb = exp(-0.5((u-c_b)/sigma)^2), sum over n
 * x[n][d]; proj[K][d] (row `axis` of M_k, or M_k^T d_hat); out partial sums are reduced
 * deterministically into sums[K][B] = S_kb = sum_n K_nb (unnormalised; this is what ranks
 * all-reduce).  max_sigma_over_delta = largest sigma/delta of the K screens (host value; sets
 * the deposit window: bins further than ~8.9 sigma from a particle are skipped).
 *
 * Multipole kicks (CompositeTransform(linear.., MultipoleTransform, linear..) followed by
 * Histogram1D, simulate/transform.py:35-55,78-146; experiments/rec_2d/nonlinear/setup.py:24-44):
 * the projection, its backward and the exact histogram take optional rows mp[K][2 d + 4] =
 * [wa (d) | wb (d) | a | b | order | 0], and the projected coordinate becomes
 *   u = proj_k . x + a_k Re(z^m) + b_k Im(z^m),  z = wa_k . x + i wb_k . x,  m = order - 1.
 * mp NULL selects the linear kernels.  The host side folds the matrices, the kick strength /
 * (order-1)! and the reference's U[:,3] = X[:,1] + .. quirk into proj, a and b
 * (simulate.multipole_terms).
 *
 * mfb_project_kde1d_fwd deposits and merges in two launches.  profiles NULL: sums only (n = 0
 * gives zeros; n_total is ignored, meas and kl must be NULL).  profiles given: n >= 1,
 * n_total > 0, and the merge kernel also normalises (diagnostics/histogram.py:39-43:
 * p = (S/N) / (sum_b (S_b/N) * delta + 1e-10), N = n_total) and -- when meas[K][B] is given --
 * evaluates kl[k] = sum_b (xlogy(t,t) - t log(p + pad)) / B (core.py:89-117 with
 * loss.py:15-17); kl is NULL iff meas is NULL.  sums[K][B] is the unnormalised input of
 * mfb_kde1d_finish and of the backward.                                                   */
int64_t mfb_kde1d_workspace_bytes(int64_t n, int d, int k, int b);
int mfb_project_kde1d_fwd(const float* x, int64_t n, int d, const float* proj, const float* mp,
                          const float* geom, int k, int b, float max_sigma_over_delta, double n_total,
                          const float* meas, float pad, float* sums, float* profiles, float* kl,
                          void* workspace, int64_t workspace_bytes, void* stream);
/* The same tail from already merged (e.g. all-reduced across ranks) sums.                   */
int mfb_kde1d_finish(const float* sums, double n_total, const float* geom, int k, int b,
                     const float* meas, float pad, float* profiles, float* kl, void* stream);
/* gsums = d/dS of <gprof, profiles> + <gkl, kl>; gprof or gkl may be NULL (not both).       */
int mfb_kde1d_finish_bwd(const float* sums, double n_total, const float* geom, int k, int b,
                         const float* meas, float pad, const float* gprof, const float* gkl,
                         float* gsums, void* stream);
/* The same tail at N > 1 GPUs with the cross-rank sum INSIDE the kernel (SURVEY 8e; replaces the NCCL all-reduce of
 * S[K][B] + the entropy sums that sat between deposit and tail): every rank owns a peer-mapped block of
 * mfb_kde1d_p2p_block_floats(k, b, tail_doubles) floats, zero-initialised, whose addresses AS MAPPED IN THIS PROCESS
 * are passed in peer_blocks_host[world] (host array).  The kernel copies local_sums[K][B] (+ local_tail doubles)
 * into its own block, exchanges an epoch over NVLink, adds all ranks' rows in rank order (bit-identical on every
 * rank) and finishes like mfb_kde1d_finish; sums[K][B] receives the reduced sums, tail_out the reduced doubles.
 * state: 3 zero-initialised uint32 in local device memory (epoch, two arrival counters), advanced by the kernel
 * itself so that a captured graph replays correctly.  Every rank must launch it once per step; k*b even,
 * k <= 1024.                                                                                                 */
int64_t mfb_kde1d_p2p_block_floats(int k, int b, int tail_doubles);
int mfb_kde1d_finish_p2p(const uint64_t* peer_blocks_host, int rank, int world, uint32_t* state,
                         const float* local_sums, const double* local_tail, int tail_doubles, double n_total,
                         const float* geom, int k, int b, const float* meas, float pad, float* sums,
                         float* profiles, float* kl, double* tail_out, void* stream);
/* deposit + (merge of the deposit's partials, cross-rank sum, normalise, KL) in two launches: the sharded counterpart
 * of mfb_project_kde1d_fwd with profiles, linear maps only.                                                    */
int mfb_project_kde1d_loss_fwd_p2p(const float* x, int64_t n, int d, const float* proj, const float* geom, int k,
                                   int b, float max_sigma_over_delta, double n_total, const float* meas, float pad,
                                   const uint64_t* peer_blocks_host, int rank, int world, uint32_t* state,
                                   const double* local_tail, int tail_doubles, float* sums, float* profiles,
                                   float* kl, double* tail_out, void* workspace, int64_t workspace_bytes,
                                   void* stream);
/* dL/dx[n][d] (+)= sum_k du_k/dx * sum_b gsums[k][b] K_nb (-(u-c_b)/sigma^2), du_k/dx = proj_k
 * without mp; accumulate!=0 adds into gx instead of overwriting it.                       */
int mfb_project_kde1d_bwd(const float* x, int64_t n, int d, const float* proj, const float* mp,
                          const float* geom, int k, int b, float max_sigma_over_delta,
                          const float* gsums, float* gx, int accumulate, void* stream);

/* ---- fused projection + exact histogram, 1-D screens -----------------------------------
 * Replaces diagnostics/diagnostics.py:128-131 (torch.histogram(x_proj, edges)): bin i holds
 * edges[i] <= u < edges[i+1], last bin closed, everything else dropped.  edges[K][B+1];
 * counts[K][B] int64, ADDED to (zero them first; integer adds => bit-reproducible).  mp as
 * for the KDE (NULL: linear).                                                             */
int mfb_project_hist1d(const float* x, int64_t n, int d, const float* proj, const float* mp,
                       const float* edges, int k, int b, int64_t* counts, void* stream);

/* ---- 2-D screens ------------------------------------------------------------------------
 * diagnostics/diagnostics.py:179-191 -> histogram.py:89-101, 47-74: P = Kx^T Ky.
 * proj[K][2][d], geom[K][2][8]; sums[K][bx][by] unnormalised.  Deposits are accumulated in
 * fixed point (44 fractional bits; 64-bit integers globally) so the result is independent
 * of the atomics' order, the CTA decomposition and the rank count.
 * workspace = int64 accumulators [2][K][bx][by] (plane 0 in units of 2^-22, plane 1 in units
 * of 2^-44; this is what ranks all-reduce exactly).                                      */
#define MFB_KDE2D_FRAC_BITS 44
int64_t mfb_kde2d_workspace_bytes(int64_t n, int d, int k, int bx, int by);
/* Screens of up to 128 x 96 bins and batches of at least 4096 particles run as tcgen05 GEMMs over the
 * particle axis (the reference's own formulation, diagnostics/histogram.py:47-74: P = Kx^T Ky), dense
 * kernel rows in split bf16; otherwise (or with MFB_FLAG_NO_TENSOR_CORES in `flags`) windowed fixed-point
 * deposits.                                                                                          */
int mfb_project_kde2d_fwd(const float* x, int64_t n, int d, const float* proj, const float* geom,
                          int k, int bx, int by, float max_sigma_over_delta, float* sums,
                          void* workspace, int64_t workspace_bytes, int flags, void* stream);
/* 1 if mfb_project_kde2d_fwd with these arguments takes the tensor-core path (any bandwidth), 0 if it takes
 * the windowed fixed-point path (sigma / bin spacing up to 1.0734, like mfb_project_kde2d_bwd)        */
int mfb_kde2d_uses_tensor_cores(int64_t n, int d, int bx, int by, int flags);
/* P <- P / (sum(P) dx dy + 1e-10)  (histogram.py:70-73) and its backward                */
int mfb_kde2d_normalize(const float* sums, const float* geom, int k, int bx, int by,
                        float* profiles, void* stream);
int mfb_kde2d_normalize_bwd(const float* sums, const float* geom, int k, int bx, int by,
                            const float* gprof, float* gsums, void* stream);
int mfb_project_kde2d_bwd(const float* x, int64_t n, int d, const float* proj, const float* geom,
                          int k, int bx, int by, float max_sigma_over_delta, const float* gsums,
                          float* gx, int accumulate, void* stream);
/* diagnostics/diagnostics.py:192-201 (np.histogramdd): edges_x[K][bx+1], edges_y[K][by+1];
 * counts[K][bx][by] int64, added to                                                      */
int mfb_project_hist2d(const float* x, int64_t n, int d, const float* proj, const float* edges_x,
                       const float* edges_y, int k, int bx, int by, int64_t* counts, void* stream);

/* ---- neural spline flow (zuko 1.3.1 NSF as built by generate/build.py:36-46) ------------
 * One autoregressive layer per call, in each of three directions: forward, inverse and backward.
 * params: packed fp32 block of one layer (layout: mfb_nsf_layer_param_floats / nsf.cu), pre-masked.
 * order_host: HOST array of d ints, the layer's autoregressive order (the feature with order 0 has a
 * bias-only spline).  params and order_host are required in every direction.
 *
 * tc_image selects the implementation.  NULL: fp32 CUDA-core kernels, every shape.  Otherwise the
 * layer's operand image from mfb_nsf_tc_prepare (mfb_nsf_tc_image_bytes bytes, 16-byte aligned) and
 * the tcgen05 kernels: the conditioner's masked GEMMs run as tcgen05.mma tiles over fp16 (hi, lo)
 * splits of the fp32 operands with fp32 accumulators in TMEM, the spline is the epilogue.  They are
 * compiled for hidden_units = 64, hidden_layers = 3, bins = 20, d = 2..6 (mfb_nsf_tc_supported) and
 * need an order that is a permutation.  They bulk-copy tiles of the layer input v (forward and
 * backward), so there v must be 16-byte aligned as well.  With tc_image, another shape returns
 * MFB_E_UNSUPPORTED; an order that is not a permutation, an unaligned image or an unaligned v
 * returns MFB_E_BADARG.
 *
 * mfb_nsf_tc_prepare turns the packed parameters of n_layers layers (layer l at
 * params + l * layer_stride_floats; all-zero masked blocks are skipped) into n_layers operand images
 * of mfb_nsf_tc_image_bytes bytes each; orders_host = HOST array [n_layers][d].                  */
int64_t mfb_nsf_layer_param_floats(int d, int hidden_units, int hidden_layers, int bins);
int mfb_nsf_tc_supported(int d, int hidden_units, int hidden_layers, int bins);
int64_t mfb_nsf_tc_image_bytes(int d, int hidden_layers);
int mfb_nsf_tc_prepare(const float* params, int64_t layer_stride_floats, int n_layers, int d,
                       int hidden_units, int hidden_layers, int bins, const int32_t* orders_host,
                       void* images, void* stream);

/* Forward: y = RQS(MaskedMLP(v))(v), logq_out = logq_in - ladj.  Replaces generate/flows/zuko.py:24-29
 * (rsample_and_log_prob / transform.inv) layer by layer.  first_layer != 0: logq_in is ignored and
 * replaced by log N(v; 0, I).  logq_in/logq_out may be NULL (sample only).                       */
int mfb_nsf_layer_fwd(const float* v, int64_t n, int d, int hidden_units, int hidden_layers, int bins,
                      const float* params, const void* tc_image, const int32_t* order_host,
                      const float* logq_in, int first_layer, float* y, float* logq_out, void* stream);

/* Inverse (density direction): v = A^-1(y) and ladj_out = ladj_in + log|det dA/dv|(v).  Replaces
 * generate/flows/zuko.py:21-22,31-32,43-50 (log_prob / inverse / inverse_steps).  Call the layers in
 * REVERSE order; with last_layer != 0 (the flow's first layer) ladj_out receives
 * log q(x) = log N(v;0,I) - sum ladj instead.  ladj_in / ladj_out may be NULL.  The CUDA-core kernel
 * makes d conditioner sweeps per particle.  The tcgen05 kernel inverts the bias-only spline of the
 * feature first in the order, then gives every further feature one pass of the conditioner (first
 * layer, two hidden GEMMs, its own output tile) and the inverse spline in registers: S x 4 GEMM round
 * trips per 128-particle tile instead of d sweeps.                                               */
int mfb_nsf_layer_inv(const float* y, int64_t n, int d, int hidden_units, int hidden_layers, int bins,
                      const float* params, const void* tc_image, const int32_t* order_host,
                      const float* ladj_in, int last_layer, float* v, float* ladj_out, void* stream);

/* Backward (replaces torch autograd through the zuko graph).  Activations are recomputed from the
 * layer input v.  gy = dL/dy [n][d], glogq = dL/dlogq_out [n] (may be NULL); outputs gv = dL/dv
 * [n][d] and gparams = dL/dparams in the packed forward layout (added to when accumulate != 0).
 * params_om: the same masked weights in out-major layout
 * W1 [64][d] | Wl [64 out][64 in] x (L-1) | Wout [d*64 (59->64 padded rows)][64 in], no biases
 * (mfb_nsf_layer_param_om_floats floats).  dL/dlogq_in = glogq (pass-through).  With tc_image the
 * layer runs as three tcgen05 kernels (nsf_tc.cu kBwd, nsf_tc_bwd.cu); a training step passes the
 * images it built for its forward pass.                                                          */
int64_t mfb_nsf_layer_param_om_floats(int d, int hidden_units, int hidden_layers);
int64_t mfb_nsf_layer_bwd_workspace_bytes(int64_t n, int d, int hidden_layers);
int mfb_nsf_layer_bwd(const float* v, const float* gy, const float* glogq, int64_t n, int d, int hidden_units,
                      int hidden_layers, int bins, const float* params, const float* params_om,
                      const void* tc_image, const int32_t* order_host, int first_layer, float* gv,
                      float* gparams, int accumulate, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- parameter layouts --------------------------------------------------------------------
 * zuko keeps every MaskedLinear as weight [out][in] + a 0/1 mask applied on each call (zuko/nn.py, reached from
 * generate/build.py:36-46); the kernels take pre-masked, transposed blocks.  One launch converts the whole flow:
 * w_in [T][64][d], b_in [T][64], w_hid [T][L-1][64][64], b_hid [T][L-1][64], w_out [T][d*P][64], b_out [T][d*P]
 * (P = 3*bins-1) and masks of the weights' shapes -> packed [T][mfb_nsf_layer_param_floats] and, if not NULL,
 * packed_om [T][mfb_nsf_layer_param_om_floats].  mfb_nsf_unpack_grads is its backward: dL/dpacked -> dL/d(each
 * tensor), masked entries exactly 0.                                                              */
int mfb_nsf_pack_params(const float* w_in, const float* b_in, const float* w_hid, const float* b_hid,
                        const float* w_out, const float* b_out, const float* m_in, const float* m_hid,
                        const float* m_out, int transforms, int d, int hidden_units, int hidden_layers, int bins,
                        float* packed, float* packed_om, void* stream);
int mfb_nsf_unpack_grads(const float* gpacked, const float* m_in, const float* m_hid, const float* m_out,
                         int transforms, int d, int hidden_units, int hidden_layers, int bins, float* g_w_in,
                         float* g_b_in, float* g_w_hid, float* g_b_hid, float* g_w_out, float* g_b_out,
                         void* stream);

/* ---- Monte-Carlo entropy pieces (entropy.py:58-62, prior.py:25-26) ----------------------
 * out[0] = sum logq, out[1] = sum |x|^2, out[2+i] = sum x_i, out[2+d+i*d+j] = sum x_i x_j
 * (double precision, deterministic two-stage reduction; the x_i / x_i x_j block only when
 * with_cov != 0; logq may be NULL).  entropy.py:35-38 (torch.cov) uses the second block. */
int64_t mfb_moments_workspace_bytes(int64_t n, int d);
int mfb_moments(const float* x, const float* logq, int64_t n, int d, int with_cov, double* out,
                void* workspace, int64_t workspace_bytes, void* stream);
/* The scalar ends of MENTFlow.loss as one launch each (they sit on the critical path of every step):
 * h[0] = (float)(a * sums[0] + b * sums[1] - c) in double -- entropy.py:58-62 with a = 1/N,
 * b = 1/(2 s^2 N), c = log prior normalisation (prior.py:25-26);
 * out[0] = h[0] + mu * mean(d[0..k)), out[1] = mean(d[0..k)) -- core.py:111-113 (h may be NULL: 0).   */
int mfb_mc_entropy(const double* sums, double a, double b, double c, float* h, void* stream);
int mfb_loss_tail(const float* d, int k, const float* h, float mu, float* out, void* stream);
/* Multi-GPU plumbing of the entropy sums (SURVEY 8e: ONE packed all-reduce per forward step): n doubles
 * <-> 2n floats (hi[0..n), lo[0..n)), hi + lo = value to 2^-48, so that they can ride at the tail of the
 * float32 all-reduce of the profile sums; the two halves are summed over ranks separately.            */
int mfb_f64_split(const double* in, int n, float* out_hi_lo, void* stream);
int mfb_f64_join(const float* in_hi_lo, int n, double* out, void* stream);

/* ---- k-nearest-neighbour entropy (KNNEntropyEstimator) ----------------------------------------
 * x[n][d], 1 <= d <= 8, 1 <= k <= 16, k < n < 2^31.  r[i] = distance from x_i to its k-th nearest OTHER particle
 * (self excluded by index, so a duplicate is a neighbour at distance 0), idx[i] = that particle's index, neighbours
 * ordered by (r^2, j): ties go to the smaller index.  A particle without k others at a finite distance (NaN or inf
 * coordinates, r^2 overflowing) gets r[i] = inf, idx[i] = i.  logsum[0] = sum_i log(r_i + pad) in double.  All
 * pairs in fp32 direct differences; deterministic (no floating-point atomics).  d > 8 or k > 16: MFB_E_UNSUPPORTED. */
int64_t mfb_knn_workspace_bytes(int64_t n, int d, int k);
int mfb_knn_kth(const float* x, int64_t n, int d, int k, double pad, float* r, int32_t* idx, double* logsum,
                void* workspace, int64_t workspace_bytes, void* stream);
/* gx[n][d] = glogsum[0] * d logsum / dx with the neighbours held fixed:
 *   w_i (x_i - x_idx[i]) + sum over j with idx[j] = i, ascending j, of w_j (x_i - x_j),  w_j = 1 / (r_j (r_j + pad)),
 * 0 where r_j = 0.  sorted_idx[n] = idx stably sorted, perm[n] (int64) the positions it came from.            */
int mfb_knn_kth_bwd(const float* x, int64_t n, int d, const float* r, const int32_t* idx,
                    const int32_t* sorted_idx, const int64_t* perm, double pad, const double* glogsum,
                    float* gx, void* stream);
/* Row ranges, for particles sharded over ranks.  x[n][d] is the whole batch (every rank's particles in rank order);
 * a rank searches and differentiates only its rows [row0, row0 + nrows), 0 <= row0 <= row0 + nrows <= n.  The
 * results are bit for bit the rows of mfb_knn_kth / mfb_knn_kth_bwd on the whole batch, whatever the range.
 * Arguments are checked before any launch: a range outside [0, n], k >= n, n >= 2^31 or a NULL pointer return
 * MFB_E_BADARG, d > 8 or k > 16 MFB_E_UNSUPPORTED.  nrows = 0 launches nothing and returns 0 (the outputs r, idx
 * of mfb_knn_kth_rows, gx of mfb_knn_kth_bwd_rows and the workspace may then be NULL).
 *   mfb_knn_kth_rows: r[nrows], idx[nrows] of the queries row0 + q (idx indexes the whole batch; a query without k
 *     others at a finite distance gets r = inf and its own index row0 + q).  No log sum: it needs every rank's r.
 *     Workspace: mfb_knn_rows_workspace_bytes(n, nrows, d, k) (0 for nrows = 0 or bad arguments).
 *   mfb_knn_logsum: logsum[0] = sum_i log(r_i + pad) over r[n] of the whole batch (the concatenated r of the ranges),
 *     added in the same order as mfb_knn_kth adds it, so it equals mfb_knn_kth's logsum bit for bit.  Workspace:
 *     8 * ceil(n / 256) bytes.
 *   mfb_knn_kth_bwd_rows: gx[nrows][d] = rows row0 .. row0 + nrows - 1 of mfb_knn_kth_bwd's gx; r, idx, sorted_idx
 *     and perm are those of the whole batch.                                                                       */
int64_t mfb_knn_rows_workspace_bytes(int64_t n, int64_t nrows, int d, int k);
int mfb_knn_kth_rows(const float* x, int64_t n, int d, int k, int64_t row0, int64_t nrows, float* r, int32_t* idx,
                     void* workspace, int64_t workspace_bytes, void* stream);
int mfb_knn_logsum(const float* r, int64_t n, double pad, double* logsum, void* workspace, int64_t workspace_bytes,
                   void* stream);
int mfb_knn_kth_bwd_rows(const float* x, int64_t n, int d, const float* r, const int32_t* idx,
                         const int32_t* sorted_idx, const int64_t* perm, int64_t row0, int64_t nrows, double pad,
                         const double* glogsum, float* gx, void* stream);

/* ---- sliced Wasserstein distance (loss.py sliced_wasserstein_distance; POT's ot.sliced_wasserstein_distance) ------
 * x[n][d], 1 <= d <= 8, 1 <= n < 2^31; theta[nproj][d] the directions.  u_k = x theta_k, each an fp32 fused
 * multiply-add chain from zero in ascending coordinate order, sorted stably (ties keep the smaller index, -0 and +0
 * compare equal, every NaN sorts last) by an 8-bit LSD radix sort per direction.  The directions are processed in
 * chunks of as many as workspace_bytes holds, at least one: mfb_swd_workspace_bytes(n, c) is the size for chunks of
 * c directions (c <= 65535).  Results do not depend on the chunking, bit for bit.
 * sorted[nproj][n] = the sorted u_k, perm[nproj][n] (may be NULL) = the particle index of each entry.            */
int64_t mfb_swd_workspace_bytes(int64_t n, int nproj_chunk);
int mfb_swd_sort(const float* x, int64_t n, int d, const float* theta, int nproj, float* sorted, int32_t* perm,
                 void* workspace, int64_t workspace_bytes, void* stream);
/* wpp[k] (double) = W_p^p between the samples' projections u_k and the reference projections y_sorted[k][0..m)
 * (ascending, e.g. from mfb_swd_sort): sum over rank pairs (i, j) of len_ij |u_(i) - v_(j)|^p, len_ij the overlap
 * of [i/n, (i+1)/n) and [j/m, (j+1)/m) computed exactly in int64; p >= 1 finite.  grad_coef[nproj][n] (may be NULL)
 * receives dW_p^p(k)/du_{k,i} at each particle's own index, with the ranks held fixed.  Per-CTA double partials are
 * added in a fixed order: no floating-point atomics.                                                               */
int mfb_swd_wpp(const float* x, int64_t n, int d, const float* theta, int nproj, const float* y_sorted, int64_t m,
                double p, double* wpp, float* grad_coef, void* workspace, int64_t workspace_bytes, void* stream);
/* gx[n][d] = sum over k ascending of gwpp[k] theta_k grad_coef[k][n] (gwpp: nproj doubles on the device)      */
int mfb_swd_bwd(const float* grad_coef, int64_t n, int d, const float* theta, int nproj, const double* gwpp,
                float* gx, void* stream);

/* ---- tanh-MLP generator (generate/nn.py NNGenerator) -------------------------------------------------------------
 * x[n][dout] = W_out t_L + b_out, t_l = tanh(W_l t_{l-1} + b_l), t_0 = z[n][din]; hidden_layers = L tanh layers of
 * hidden_units.  Weights in nn.Linear layout: w_in[H][din], b_in[H], w_hid[L-1][H][H], b_hid[L-1][H] (both may be NULL
 * when L = 1), w_out[dout][H], b_out[dout].  fp32 on the CUDA cores, accurate tanh.  Compiled for 1 <= din, dout <= 8,
 * H = 64, 1 <= L <= 8 (mfb_nn_supported); another shape returns MFB_E_UNSUPPORTED, a NULL required pointer or n < 1
 * MFB_E_BADARG, both before any launch.                                                                             */
int mfb_nn_supported(int din, int dout, int hidden_units, int hidden_layers);
int mfb_nn_fwd(const float* z, int64_t n, int din, int dout, int hidden_units, int hidden_layers, const float* w_in,
               const float* b_in, const float* w_hid, const float* b_hid, const float* w_out, const float* b_out,
               float* x, void* stream);
/* Backward from z and gx = dL/dx: the forward is recomputed on chip.  gz[n][din] = dL/dz (may be NULL); the six
 * parameter gradients are written (not accumulated) in the weights' layouts.  Per-CTA partials in the workspace are
 * added in CTA order: no floating-point atomics, repeated calls are bitwise equal.  0 from the size query: shape not
 * supported.                                                                                                        */
int64_t mfb_nn_bwd_workspace_bytes(int64_t n, int din, int dout, int hidden_units, int hidden_layers);
int mfb_nn_bwd(const float* z, const float* gx, int64_t n, int din, int dout, int hidden_units, int hidden_layers,
               const float* w_in, const float* b_in, const float* w_hid, const float* b_hid, const float* w_out,
               const float* b_out, float* gz, float* gw_in, float* gb_in, float* gw_hid, float* gb_hid, float* gw_out,
               float* gb_out, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- classical MENT (ment.py, sample.py) --------------------------------------------------
 * rho(x) = exp(log prior(x)) * prod clamp(h(u(x)), 0, 1e10) over two families of Lagrange tables, evaluated in
 * double like scipy's RegularGridInterpolator and 0 outside the box of the bin centres (ment.py:36-52, 227-249);
 * either family may be empty (k = 0 / k2 = 0):
 *   1-D screens: h_k linear on tables[k][0..b) at the bin centres coords[k][0..b), u = proj[k] . x;
 *   2-D screens (LagrangeFunction over an N-D RegularGridInterpolator; experiments/config/rec_nd_2d_ment.yaml):
 *     h bilinear on tables2[k2][bx][by] at the bin-centre grids cx2[k2][bx] x cy2[k2][by], u = proj2[k2][2][d] . x
 *     (the two measured rows of each transfer matrix).
 * prior: log p(x) = prior_neg_half_inv_s2 * |x|^2 + prior_log_norm (Gaussian prior.py:25-26; a flat prior passes 0
 * and its log constant).
 *
 * Multipole kicks: every transfer map is linear or a chain linear* -> MultipoleTransform (order 3, 4 or 5, normal or
 * skew) -> linear* (simulate/transform.py:35-146; experiments/rec_2d/nonlinear).  The measured coordinate of a row is
 * then proj . x + a Re(z^m) + b Im(z^m), z = wa . x + i wb . x, m = order - 1, with mp[k][2 d + 4] = [wa (d) | wb (d) |
 * a | b | order | 0] for the 1-D screens and mp2[k2][2][2 d + 4] for the two rows of each 2-D screen (they share wa,
 * wb and the order).  A row of a linear map has order 0 and adds no kick.  The host folds matrices, kick
 * strength / (order-1)! and the reference's quirks into these terms (simulate.multipole_terms,
 * simulate.multipole_inverse_terms).
 * With mp, mp2 and (integrate) inv_mp all NULL every map is linear.  If any of them is given the kernels with kicks
 * run; mp is then required when k > 0, mp2 when k2 > 0 and inv_mp by the integration, otherwise MFB_E_BADARG.  */
/* rho at explicit points x[g][d]                                                          */
int mfb_ment_prob(const float* x, int64_t g, int d, const float* proj, const float* coords, const float* tables,
                  int k, int b, const float* mp, const float* proj2, const float* cx2, const float* cy2,
                  const float* tables2, int k2, int bx, int by, const float* mp2, float prior_neg_half_inv_s2,
                  float prior_log_norm, float* out, void* stream);
/* rho on the cell centres of a regular grid generated from the index ('ij' order, last axis fastest) instead of
 * res^D x D materialised points (sample.py:99-104 GridSampler).  shape / first_centre / step are HOST arrays of d
 * entries.                                                                                */
int mfb_ment_prob_grid(int d, const int32_t* shape_host, const float* first_centre_host, const float* step_host,
                       const float* proj, const float* coords, const float* tables, int k, int b, const float* mp,
                       const float* proj2, const float* cx2, const float* cy2, const float* tables2, int k2,
                       int bx, int by, const float* mp2, float prior_neg_half_inv_s2, float prior_log_norm,
                       float* out, void* stream);
/* integrate mode (ment.py:267-317): pred[i] = sum over the integration grid (n_int_axes = d - 1 or d - 2 HOST
 * arrays) of rho(x(u)), u = meas_coords[i] on meas_axis and the grid point on the other axes.  meas_axis2 >= 0
 * selects a 2-D screen: pred[nb_meas][nb_meas2], meas_coords2 on meas_axis2; meas_axis2 = -1 a 1-D one.
 * The screen is mapped back with the folded inverse of its transfer map,
 *   x = linv u + p Re(zi^m) + q Im(zi^m),  zi = r0 . u + i r2 . u,
 * inv_mp[4 d + 2] = [r0 (d) | r2 (d) | p (d) | q (d) | order | 0] (order 0, or inv_mp NULL: a linear map, x = linv u;
 * linv = M^-1).  d >= 2.                                                                  */
int mfb_ment_integrate(int d, const float* meas_coords, int nb_meas, int meas_axis, const float* meas_coords2,
                       int nb_meas2, int meas_axis2, int n_int_axes, const int32_t* int_shape_host,
                       const float* int_first_host, const float* int_step_host, const float* linv,
                       const float* inv_mp, const float* proj, const float* coords, const float* tables, int k,
                       int b, const float* mp, const float* proj2, const float* cx2, const float* cy2,
                       const float* tables2, int k2, int bx, int by, const float* mp2,
                       float prior_neg_half_inv_s2, float prior_log_norm, float* pred, void* stream);
/* sample.py:27-57: cdf of (rho + pad) over the cells in double, then `size` draws: cell by
 * inverse-CDF search with a Philox4x32-10 stream (seed, offset), uniform position inside the
 * cell (+ 0.5*U(-delta,delta) when jitter != 0).  workspace[0] (device double) = total mass. */
int64_t mfb_cdf_workspace_bytes(int64_t g);
int mfb_cdf_build(const float* rho, int64_t g, double pad, double* cdf, void* workspace,
                  int64_t workspace_bytes, void* stream);
int mfb_cdf_sample(const double* cdf, int64_t g, const void* workspace, int d,
                   const int32_t* shape_host, const float* first_edge_host, const float* cell_host,
                   int jitter, uint64_t seed, uint64_t offset, int64_t size, float* out, void* stream);
/* ment.py:360-367: pred[pred<thresh]=0; where meas!=0 and pred!=0: h *= 1 + lr*(meas/pred-1) */
int mfb_gs_update(float* table, const float* meas, const float* pred, int n, float lr, float thresh,
                  void* stream);

/* ---- base noise of the flow ---------------------------------------------------------------
 * generate/flows/zuko.py:15-16,24-26 (`flow.base.rsample`: zuko DiagNormal -> torch.randn).
 * out[numel] ~ N(0,1) from Philox4x32-10 with torch's CUDA element assignment: for the (seed,
 * offset) of torch's CUDA generator the result is bitwise the tensor torch.randn(numel,
 * device="cuda") returns, and mfb_randn_offset_increment(numel) is what torch adds to the offset.
 * _state form: state[0] = seed, state[1] = offset live in DEVICE memory; with advance != 0 the
 * offset is moved on after the draw (stream-ordered), so a captured graph draws fresh noise at
 * every replay.                                                                              */
int64_t mfb_randn_offset_increment(int64_t numel);
int mfb_randn_philox(float* out, int64_t numel, uint64_t seed, uint64_t offset, void* stream);
int mfb_randn_philox_state(float* out, int64_t numel, uint64_t* state, int advance, void* stream);

/* ---- diagnostics --------------------------------------------------------------------------
 * Self-test of the tcgen05/TMEM building blocks: d[128][n] = a[128][64] * b[n][64]^T through
 * fp16 (hi,lo)-split kind::f16 MMAs with TMEM accumulators (n = 64, 128 or 256).  *err != 0
 * if the MMA never completed.                                                              */
int mfb_selftest_umma(const float* a, const float* b, int n, float* d, int* err, void* stream);
/* the same GEMM with the A operand in tensor memory (tcgen05.st + tcgen05.mma with a TMEM A address), n <= 128 */
int mfb_selftest_umma_ts(const float* a, const float* b, int n, float* d, int* err, void* stream);
/* One K step (16) with 32-byte-row SWIZZLE_32B operand tiles: d[128][n] = a[128][16] * b[n][16]^T
 * (values rounded to fp16).  mode 0: both operands SWIZZLE_32B; mode 1: a sits in K step `kstep`
 * of a 64-wide SWIZZLE_128B tile (the layouts the flow kernel mixes).  n = 64 or 128.        */
int mfb_selftest_umma_sw32(const float* a, const float* b, int n, int mode, int kstep, float* d, int* err,
                           void* stream);
/* The 2-SM MMA of a CTA pair (cluster of 2, cta_group::2): d[256][64] = a[256][K] * b[64][K]^T (values rounded to
 * fp16), each CTA holding 128 rows of a and 32 rows of b.  mode 0: K = 16, SWIZZLE_32B tiles; mode 1: K = 64,
 * SWIZZLE_128B tiles.  err: 1 / 2 = the completion / request mbarrier timed out.                            */
int mfb_selftest_umma_pair(const float* a, const float* b, int mode, float* d, int* err, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MENTFLOW_B200_H */
