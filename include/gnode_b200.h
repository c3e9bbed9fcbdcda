/*
 * gnode_b200.h -- C ABI of the B200-native GN-ODE rollout library (libgnode_b200.so).
 *
 * The reference (sissykosm/GN-ODE-SIR) is pure Python and has no FFI; its boundary
 * for this path is the Python class interface ODEfunc / ODEBlock.  Every entry
 * point below names the reference code it replaces (paths relative to the reference
 * root).  The Python drop-in classes in gn-ode-sir_b200/ bind these symbols with
 * ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - all tensors are caller-allocated DEVICE memory, fp32, row-major, H == 64;
 *   - the library owns only graph/batch handles (device CSR + tiny descriptors);
 *   - every call takes the CUDA stream to enqueue on; no call synchronises the
 *     stream or the device (graph/batch creation use their own blocking copies);
 *   - return value 0 on success, negative on error; gnode_last_error() returns a
 *     thread-local description of the most recent failure;
 *   - there is NO CPU fallback: without a CUDA device every compute entry fails.
 *
 * Row space: a "batch" is a list of instances (one graph + one trial each).
 * Instance i owns the contiguous global rows [row0_i, row0_i + n_i); M = sum n_i.
 * This is the reference's block-diagonal batching
 *   ode_nn_ngraph_sim.py:68-71  (B copies of one graph, rows b*N + n)
 *   ode_nn_ngraphs.py:65-71     (ragged concatenation of different graphs).
 */
#ifndef GNODE_B200_H
#define GNODE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNODE_H 64              /* hidden width the kernels are specialised for */
#define GNODE_OK 0
#define GNODE_ERR_ARG (-1)
#define GNODE_ERR_CUDA (-2)
#define GNODE_ERR_UNSUPPORTED (-3)

typedef struct gnode_graph* gnode_graph_t;
typedef struct gnode_batch* gnode_batch_t;

/* Device pointers to the model parameters; names are the reference's state_dict
 * keys (ode_nn_ngraph_sim.py:47-48,123-131).  The two unused LayerNorms have no
 * arithmetic on the path and are not passed. */
typedef struct {
    const float* lin_w;   /* odefunc.linear.weight [H,H] (out,in)           */
    const float* lin_b;   /* odefunc.linear.bias   [H]                       */
    const float* s1_w;    /* linearS1.weight       [H,1] -> H contiguous     */
    const float* s1_b;    /* linearS1.bias         [H]                       */
    const float* l3_w;    /* linear3.weight        [4,H]                     */
    const float* l3_b;    /* linear3.bias          [4]                       */
    const float* s2_w;    /* linearS2.weight       [1,4] -> 4 contiguous     */
    const float* s2_b;    /* linearS2.bias         [1]                       */
} gnode_params_t;

/* Flat layout of the gradient vector written by gnode_rollout_backward
 * (same order as gnode_params_t). */
#define GNODE_GRAD_OFF_LIN_W 0
#define GNODE_GRAD_OFF_LIN_B (GNODE_H * GNODE_H)
#define GNODE_GRAD_OFF_S1_W (GNODE_GRAD_OFF_LIN_B + GNODE_H)
#define GNODE_GRAD_OFF_S1_B (GNODE_GRAD_OFF_S1_W + GNODE_H)
#define GNODE_GRAD_OFF_L3_W (GNODE_GRAD_OFF_S1_B + GNODE_H)
#define GNODE_GRAD_OFF_L3_B (GNODE_GRAD_OFF_L3_W + 4 * GNODE_H)
#define GNODE_GRAD_OFF_S2_W (GNODE_GRAD_OFF_L3_B + 4)
#define GNODE_GRAD_OFF_S2_B (GNODE_GRAD_OFF_S2_W + 4)
#define GNODE_GRAD_COUNT (GNODE_GRAD_OFF_S2_B + 1)

#define GNODE_GRAD_ADJOINT 0   /* torchdiffeq odeint_adjoint semantics (what the reference trains with) */
#define GNODE_GRAD_DISCRETE 1  /* exact back-propagation of the discrete Euler loop */

const char* gnode_last_error(void);
int gnode_version(void);
/* Kernel variant of the forward step: bit 0 = tcgen05 3xTF32 tensor-core transform (else fused FFMA),
 * bit 1 = MUFU ex2/rcp sigmoid (else expf + IEEE division). Default: env GNODE_VARIANT or the build default. */
int gnode_set_variant(int variant);
int gnode_get_variant(void);
/* Structure of the tensor-core step kernel (variants with bit 0 set): 5 = pipelined, S_k stream by TMA (default: one
 * 1024-thread CTA per SM running two 128-row tile pipelines that share the weight operand; the S_k tile arrives by TMA
 * tensor loads straight into the UMMA operand layout, the raw fp32 tile is the hi operand and S_k is read once; the
 * decoder's hidden layer comes out of the step's two GEMMs), 6 = 5 with a block barrier after the I' store, 7 = 5 with
 * 3xTF32 (the lo x lo term of the 4-term split product dropped: ~2 % faster, per-product error 2^-20 instead of 1.5 * 2^-21),
 * 3 = the same pipeline with LDG-fed operands (round 1; also what runs when no tensor map can be encoded), 0 = generic.
 * Default: env GNODE_STEP_KERNEL or 5. All produce the same trajectories within the parity tolerance.
 * These switches (variant, step kernel, R state, persistent) are PROCESS-WIDE settings read at every rollout call:
 * set them before launching work from several threads, not concurrently with it. */
int gnode_set_step_kernel(int kernel);
int gnode_get_step_kernel(void);
/* How inference rollouts (traj == NULL, default step kernel) carry the R block. 1 (default) = not at all: R feeds only
 * the decoder's linear3 (ode_nn_ngraph_sim.py:172-176) and dS + dI + dR = 0 (:75-77), i.e. S + I + R is conserved channel
 * by channel, so the decoder's pre-activations of R_k are W3 (S_0 + I_0 + R_0) - W3 S_k - W3 I_k: four floats per row
 * written once by the encoder launch, minus two terms the transform's GEMMs deliver anyway. The 64-float R plane is
 * neither read nor written and nothing of R is computed per step (512 B per node-step less traffic; probabilities agree
 * with the full-plane path to fp32 rounding, < 1e-6 on the goldens). 0 = full R plane, bitwise the training forward.
 * Env GNODE_R_STATE=full selects 0. Training (traj != NULL) always stores R. */
int gnode_set_r_state(int hidden);
int gnode_get_r_state(void);
/* Rollout launch structure of the tensor-core step kernels: 1 = ONE cooperative launch runs all Euler steps with a grid
 * barrier between them, 0 = one launch per step, -1 (default) = cooperative for batches of up to 32 tiles per SM.
 * Env GNODE_PERSISTENT=0/1 sets the initial value. Process-wide, like the other switches here. */
int gnode_set_persistent(int mode);
int gnode_get_persistent(void);
/* In-order relay for isolated hub rows (degree > 512; DESIGN.md 3.1): 1 (default) = on, 0 = every row is walked by one
 * half-warp. Both give BITWISE the same sums; the switch exists for that check and for A/B measurements. */
int gnode_set_hub_relay(int on);
int gnode_get_hub_relay(void);
/* Tile kernel of the reverse sweep (state VJP v = gz W on tcgen05 and weight gradient vW = gz^T X by register-blocked
 * FFMA per 128-row tile): 2 (default) = two 256-thread CTAs per SM, the two halves of a tile in sequence, next unit
 * prefetched behind the adjoint's read-modify-write; 1 = the round-1 one-CTA kernel. Env GNODE_BWD_VJP sets the initial
 * value. Process-wide. Gradients of the two agree to fp32 summation-order noise. */
int gnode_set_bwd_kernel(int kernel);
int gnode_get_bwd_kernel(void);
/* debug: per-phase SM-cycle sums of the step kernel collected while env GNODE_DBG has bit 7 set; resets them */
int gnode_debug_phase_cycles(long long* out8);
/* number of CUDA kernels this library has launched in the calling process (bench.py gpu_launches) */
int64_t gnode_launch_count(void);

/* ---- graphs ---------------------------------------------------------------
 * Replaces the host-resident scipy CSR the reference keeps in ODEfunc.A /
 * ODEfunc.A_list (ode_nn_ngraph_sim.py:41, ode_nn_ngraphs.py:41, built by
 * nx.adjacency_matrix at ode_nn.py:413) and its per-step re-expansion to COO.
 * rowptr[n+1], colidx[nnz] are HOST int32 CSR arrays; stored values are ignored
 * (every stored entry counts once, as in the reference; per-edge weights are passed to
 * the _weighted rollout calls instead, see below). Columns are sorted per
 * row at creation so the neighbour sum runs in ascending-column order, the order
 * of the reference's CPU scatter_add_. The transposed pattern is built here too
 * (backward); undirected graphs share one copy. */
int gnode_graph_create(int32_t n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
                       gnode_graph_t* out);
int gnode_graph_destroy(gnode_graph_t g);
int gnode_graph_info(gnode_graph_t g, int32_t* n, int64_t* nnz, int32_t* max_degree, int32_t* symmetric);

/* ---- batches --------------------------------------------------------------
 * Replaces scipy.sparse.block_diag(a) + LongTensor(idx).to(device), executed by
 * the reference on the host at EVERY Euler step (ode_nn_ngraph_sim.py:68-71,
 * ode_nn_ngraphs.py:65-71). Built once per distinct instance list. */
int gnode_batch_create(const gnode_graph_t* inst_graphs, int32_t n_inst, gnode_batch_t* out);
int gnode_batch_destroy(gnode_batch_t b);
int64_t gnode_batch_rows(gnode_batch_t b);

/* ---- a7: neighbour aggregation -------------------------------------------
 * out[r,:] = sum over stored (r,c) of in[c,:]   (transpose != 0: over stored (c,r)).
 * Replaces the gather / repeat / scatter_add_ at ode_nn_ngraph_sim.py:73,
 * ode_nn_ngraphs.py:73. in/out: [M,H]. */
int gnode_aggregate(gnode_batch_t b, const float* in, float* out, int transpose, void* stream);

/* ---- a5-a8: one evaluation of the ODE right-hand side ----------------------
 * Replaces ODEfunc.forward(t, y) (ode_nn_ngraph_sim.py:58-96, ode_nn_ngraphs.py:54-83).
 * y, dy: [3,M,H] (S,I,R planes); beta,gamma: [M]; scratch: [M,H] floats. */
int gnode_odefunc_eval(gnode_batch_t b, const float* y, const float* beta, const float* gamma,
                       const gnode_params_t* p, float* dy, float* scratch, void* stream);

/* ---- a1-a9: the whole rollout ---------------------------------------------
 * Replaces ODEBlock.forward (ode_nn_ngraph_sim.py:148-188, ode_nn_ngraphs.py:124-152)
 * including torchdiffeq's fixed-grid Euler loop (odeint(..., method='euler')).
 *   x      [M, ldx] fp32, ldx >= 5: columns S0 I0 R0 beta gamma (rest ignored)
 *   T      number of grid points (len(integration_time)); dt_host[T-1] HOST floats
 *          dt_k = (float)(t_{k+1} - t_k)
 *   traj   [T,3,M,H] or NULL. NULL = inference (states ping-pong in the workspace)
 *   probs  [T,M,3]  softmax probabilities (S,I,R) of every grid state
 *   workspace: gnode_rollout_workspace_bytes(b, traj != NULL) bytes, 256-B aligned */
size_t gnode_rollout_workspace_bytes(gnode_batch_t b, int with_traj);
int gnode_rollout_forward(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                          int32_t T, const float* dt_host, float* traj, float* probs,
                          void* workspace, size_t workspace_bytes, void* stream);

/* The same rollout emitting only selected grid points: out_steps (HOST int32[n_out], strictly ascending indices in
 * [0,T)) names the grid points whose probabilities are written, probs is [n_out,M,3]; NULL = all T (n_out ignored).
 * This is get_sir_t_nodes_torch's selection x_rk[int(i/deltaT)] (ode_nn.py:249-261; callers
 * ode_nn_ngraph_sim.py:230-232,259-261,285-287) moved into the rollout: the decoder + softmax of the other grid points
 * is never computed and never stored. */
int gnode_rollout_forward_sel(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                              int32_t T, const float* dt_host, const int32_t* out_steps, int32_t n_out,
                              float* traj, float* probs, void* workspace, size_t workspace_bytes, void* stream);

/* ---- N4: compact trial descriptors ------------------------------------------
 * Replaces the dense [N, 3+H] fp32 input block per trial that main() builds on the host and ships to the device
 * (ode_nn_ngraph_sim.py:371-390: I0[seeds] = 1, S0 = 1 - I0, R0 = 0, bg[:,0] = beta, bg[:,1] = gamma;
 * ode_nn_ngraphs.py:326-345) and ODEBlock.forward unpacks again (:149-150). Instance i of the batch is described by
 *   seeds[seed_ptr[i] .. seed_ptr[i+1])  instance-local node ids infected at t = 0 (DEVICE int32; seed_ptr[n_inst+1];
 *                                        ids outside [0, n_i) are ignored)
 *   beta[i], gamma[i]                    DEVICE fp32, one per instance.
 * gnode_expand_trials writes the five live columns {S0, I0, R0, beta, gamma} of every row into x [M, ldx] (ldx >= 5;
 * the remaining columns are not touched) -- the training path keeps that compact x for the reverse sweep.
 * gnode_rollout_forward_trials gives the probabilities of expansion (ldx = GNODE_TRIAL_LDX, in the workspace) +
 * gnode_rollout_forward_sel, bit for bit, without ever forming the dense block when it rolls out for inference
 * (traj == NULL, T > 1, default step kernel and R state): every row of y_0 is one of two vectors (SURVEY a2), so the
 * encoder, its transform and the decoder of grid point 0 are evaluated for two rows into a small table, a seed bitmap is
 * set from the descriptors, and Euler step 0 runs from table + bitmap (neither y_0 nor I'_0 is written); cooperative
 * rollouts of small batches keep an encoder launch, which is then a stream of stores. Env GNODE_TRIALS_ENCODE=dense | fill
 * selects the expansion path / the store-stream encoder for A/B. The workspace size is the same in all cases. */
#define GNODE_TRIAL_LDX 8
int gnode_expand_trials(gnode_batch_t b, const int32_t* seeds, const int32_t* seed_ptr, const float* beta,
                        const float* gamma, float* x, int64_t ldx, void* stream);
size_t gnode_rollout_trials_workspace_bytes(gnode_batch_t b, int with_traj);
int gnode_rollout_forward_trials(gnode_batch_t b, const int32_t* seeds, const int32_t* seed_ptr, const float* beta,
                                 const float* gamma, const gnode_params_t* p, int32_t T, const float* dt_host,
                                 const int32_t* out_steps, int32_t n_out, float* traj, float* probs,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* ---- a10: backward (reverse sweep over the stored trajectory) --------------
 * Replaces torchdiffeq OdeintAdjointMethod.backward + autograd of the encoder /
 * decoder (entered from loss.backward(), ode_nn_ngraph_sim.py:245).
 *   grad_probs [T,M,3] = dL/dprobs;  grads_out [GNODE_GRAD_COUNT] (overwritten)
 *   workspace: gnode_backward_workspace_bytes(b) bytes */
size_t gnode_backward_workspace_bytes(gnode_batch_t b);
int gnode_rollout_backward(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                           int32_t T, const float* dt_host, const float* traj,
                           const float* grad_probs, int32_t grad_mode, float* grads_out,
                           void* workspace, size_t workspace_bytes, void* stream);

/* The same with a sparse cotangent: grad_probs is [n_out,M,3] for the grid points out_steps (as in
 * gnode_rollout_forward_sel); grid points without a cotangent skip the decoder's backward, and reverse steps beyond the
 * last selected grid point (zero adjoint) are not run. NULL = dense [T,M,3]. */
int gnode_rollout_backward_sel(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                               int32_t T, const float* dt_host, const float* traj, const float* grad_probs,
                               const int32_t* out_steps, int32_t n_out, int32_t grad_mode, float* grads_out,
                               void* workspace, size_t workspace_bytes, void* stream);

/* ---- training with auxiliary storage (round 2) ---------------------------------
 * The reverse sweep of torchdiffeq's adjoint re-evaluates f at every stored state (OdeintAdjointMethod.backward), i.e.
 * it recomputes I' = sigmoid(linear(I_j)) and repeats the neighbour gather A I' of ode_nn_ngraph_sim.py:62-73. The
 * forward already holds both: it writes I'_{k+1} for the next step's gather and sums AI_k row by row. With an `aux`
 * buffer of gnode_rollout_aux_bytes(b, T) bytes ([T][2][Mr + 1][H] fp32, Mr = M rounded up to 128) the forward keeps
 * I'_k of every grid point (no extra traffic) and AI_k (256 B per row and step more), and the reverse sweep runs three
 * launches with ONE neighbour gather per step instead of four launches with two.
 *   aux_filled (HOST int32, out): 1 if the buffer was filled (default step kernel with tensor maps available), else 0
 *   -- pass aux to gnode_rollout_backward_aux only when it is 1, NULL otherwise. aux == NULL: exactly the _sel calls. */
size_t gnode_rollout_aux_bytes(gnode_batch_t b, int32_t T);
int gnode_rollout_forward_aux(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                              int32_t T, const float* dt_host, const int32_t* out_steps, int32_t n_out,
                              float* traj, float* aux, int32_t* aux_filled, float* probs, void* workspace,
                              size_t workspace_bytes, void* stream);
int gnode_rollout_backward_aux(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                               int32_t T, const float* dt_host, const float* traj, const float* aux,
                               const float* grad_probs, const int32_t* out_steps, int32_t n_out, int32_t grad_mode,
                               float* grads_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- input gradients: dL/d{S0, I0, R0, beta, gamma} -------------------------------
 * The reference's autograd reaches every input column that enters the computation: S0, I0, R0 through the encoder
 * relu(linearS1(c)) (ode_nn_ngraph_sim.py:151-156), beta and gamma through the bg block of the ODE state, which f reads
 * (:60) and whose adjoint builds up over torchdiffeq's reverse sweep. Per reverse step at state y_j with cotangent
 * a = (aS, aI, aR) and step dt (the same state and dt as the parameter VJP; ADJOINT: y_i with a_i, DISCRETE: exact
 * back-propagation of the Euler loop):
 *   dL/dbeta[r]  += dt * sum_h (aI - aS) AI S'       dL/dgamma[r] += dt * sum_h (aR - aI) I'
 * and after the sweep, with the final adjoint a_0 and y_0 = relu(c w1 + b1):  dL/dc[r] = sum_h a0[r,h] [y0 > 0] w1[h].
 * Reverse sweep with optional parameter and input gradients.
 *   grads_out  [GNODE_GRAD_COUNT] or NULL: no parameter gradient (the weight-gradient phase is skipped)
 *   grad_x     [M, ldgx] or NULL (ldgx >= 5): columns 0..4 overwritten with dL/d{S0, I0, R0, beta, gamma}, other
 *              columns untouched; at least one of grads_out / grad_x non-NULL.
 * grad_x == NULL is gnode_rollout_backward_aux, bit for bit. Same workspace (gnode_backward_workspace_bytes). Every row's
 * gradient is summed in a fixed order without atomics: bitwise reproducible. */
int gnode_rollout_backward_input(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p, int32_t T,
                                 const float* dt_host, const float* traj, const float* aux, const float* grad_probs,
                                 const int32_t* out_steps, int32_t n_out, int32_t grad_mode, float* grads_out,
                                 float* grad_x, int64_t ldgx, void* workspace, size_t workspace_bytes, void* stream);

/* ---- edge gradients: dL/dw per stored adjacency entry ------------------------------
 * The forward is the reference's binary adjacency; the gradient is that of the weighted neighbour sum
 * AI[r] = sum_c w_rc I'[c], taken at w = 1 (what contact reduction, edge removal and structural attribution rank by).
 * Per reverse step, at the same state and dt as the parameter VJP (ADJOINT: y_i with a_i; DISCRETE: exact
 * back-propagation of the Euler loop), with gAI = beta (aI - aS) S':
 *   dL/dw_rc += dt * sum_h gAI[r,h] I'[c,h]          for every stored entry (r, c) of A
 * Row sums tie it to grad_x: sum over row r's entries of dL/dw_rc = beta[r] * dL/dbeta[r].
 *   grad_edge  [nnz_total] or NULL: overwritten with dL/dw. Layout: instance after instance (in batch order), inside an
 *              instance the graph's CSR order after gnode_graph_create's per-row column sort.
 * Arguments otherwise as gnode_rollout_backward_input (which is this call with grad_edge == NULL, bit for bit); at least
 * one of grads_out / grad_x / grad_edge non-NULL. Same workspace. One more row kernel per reverse step when grad_edge is
 * non-NULL; one lane per edge adds its fixed-order dot product (no atomics): bitwise reproducible. */
int gnode_rollout_backward_edges(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p, int32_t T,
                                 const float* dt_host, const float* traj, const float* aux, const float* grad_probs,
                                 const int32_t* out_steps, int32_t n_out, int32_t grad_mode, float* grads_out,
                                 float* grad_x, int64_t ldgx, float* grad_edge, void* workspace, size_t workspace_bytes,
                                 void* stream);

/* ---- weighted contact graphs: per-edge weights in the neighbour sum --------------------
 * The rollout with AI[r] = sum over stored (r, c), in ascending column order, of fl(w_rc * I'[c]): every product rounded
 * on its own, then added in the binary sum's order. So w = 1 gives the binary rollout's bits and w = 0 those of a graph
 * built without that entry (I' is finite). Weights may take any finite value.
 *   edge_w  DEVICE fp32 [nnz_total], in the batch's edge order (that of grad_edge above); read at every call, so values
 *           written in place between calls are honoured (also by a replayed reverse sweep).
 * gnode_rollout_forward_weighted: the arguments of gnode_rollout_forward_aux plus edge_w; edge_w == NULL is that call,
 * bit for bit. The weighted neighbour sum runs on the default step kernel (5) with tensor maps, one launch per step or
 * the persistent cooperative launch; any other step-kernel setting, or a driver without tensor maps, returns
 * GNODE_ERR_UNSUPPORTED. With aux, the stored AI_k is the weighted sum.
 * gnode_rollout_backward_weighted: the arguments of gnode_rollout_backward_edges plus edge_w (the weights of the forward
 * that stored traj / aux); grad_edge then receives dL/dw at those weights. The transposed gather of the sweep,
 * sum_c w_cr gAI[c], reads the weights in transpose order: a kernel of the enqueued sequence permutes edge_w into the
 * workspace by each graph's transpose map (kept at gnode_graph_create, uploaded on the first weighted call -- a blocking
 * copy, made before any stream capture). Workspace: gnode_backward_weighted_workspace_bytes(b) (the unweighted size
 * plus nnz_total floats). edge_w == NULL is gnode_rollout_backward_edges, bit for bit. */
int gnode_rollout_forward_weighted(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                   int32_t T, const float* dt_host, const int32_t* out_steps, int32_t n_out,
                                   float* traj, float* aux, int32_t* aux_filled, float* probs, const float* edge_w,
                                   void* workspace, size_t workspace_bytes, void* stream);
size_t gnode_backward_weighted_workspace_bytes(gnode_batch_t b);
int gnode_rollout_backward_weighted(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p, int32_t T,
                                    const float* dt_host, const float* traj, const float* aux, const float* grad_probs,
                                    const int32_t* out_steps, int32_t n_out, int32_t grad_mode, float* grads_out,
                                    float* grad_x, int64_t ldgx, float* grad_edge, const float* edge_w, void* workspace,
                                    size_t workspace_bytes, void* stream);

/* Per-instance sums of grad_x columns 3 and 4 (instance i = rows [row0_i, row0_i + n_i)), in a fixed order:
 * the gradient of compact trial descriptors' beta[i], gamma[i] (N4). grad_beta, grad_gamma: DEVICE float[n_inst]. */
int gnode_trials_grad(gnode_batch_t b, const float* grad_x, int64_t ldgx, float* grad_beta, float* grad_gamma,
                      void* stream);

/* ---- N1: L1 loss on the sub-sampled prediction and its cotangent, fused -------
 * Replaces, per mini-batch, get_sir_t_nodes_torch x3 (60 row copies device -> CPU tensor, ode_nn.py:257-259), the
 * cat / transpose / .to(device) and nn.L1Loss on [:,1:,:] (ode_nn_ngraph_sim.py:230-234, ode_nn_ngraphs.py:216-220),
 * and the autograd of all of it: with probs [n_out,M,3] (fp32, the selected grid points, time-major as the rollout
 * writes them) and labels [M,n_out,3] (fp64, node-major as the reference's y.view(-1, maxTime, 3)),
 *   loss = mean over m, t >= skip, c of |probs[t,m,c] - labels[m,t,c]|      (float64 accumulation, like the reference's
 *                                                                            promoted L1Loss)
 *   grad_probs[t,m,c] = sign(probs - labels) * scale / count  for t >= skip, 0 for t < skip;  count = M (n_out-skip) 3.
 * loss_out: DEVICE double[1]; grad_probs may be NULL (evaluation). scratch: gnode_l1_scratch_bytes() bytes. The sum is
 * taken in a fixed order (per-block partial sums, then one block): bitwise reproducible. */
size_t gnode_l1_scratch_bytes(void);
int gnode_l1_loss_grad(const float* probs, const double* labels, int64_t M, int32_t n_out, int32_t skip, float scale,
                       double* loss_out, float* grad_probs, void* scratch, void* stream);

/* ---- N3: Monte-Carlo SIR labels ------------------------------------------------
 * Replaces sir_torch (ode_nn.py:30-88; called from load_SIR_labels, ode_nn_ngraph_sim.py:198): `sims` independent
 * discrete-time SIR simulations of T-1 steps from the seed set on graph g. Per step, with the nodes infected at its
 * start: every (infected u, susceptible v) edge transmits with probability beta, every infected u recovers with
 * probability gamma. One CTA per simulation, bit-packed state in shared memory, Philox4x32-10 keyed by
 * (rng_seed; simulation, step, edge / node): the counts are a pure function of the arguments.
 *   seeds   DEVICE int32[n_seeds] node ids (0-based positions in the CSR)
 *   counts  DEVICE double[3][T][n]: number of simulations in which node v is S / I / R at step t, t >= 1; the t = 0
 *           rows hold the 0/1 initial state (the reference assigns them instead of accumulating, ode_nn.py:54-55).
 *           Labels = counts / sims, as load_SIR_labels divides.
 *   workspace: gnode_mc_sir_workspace_bytes(g, T) bytes. Graphs of more than ~540k nodes are not supported. */
size_t gnode_mc_sir_workspace_bytes(gnode_graph_t g, int32_t T);
int gnode_mc_sir(gnode_graph_t g, const int32_t* seeds, int32_t n_seeds, float beta, float gamma, int32_t sims,
                 int32_t T, uint64_t rng_seed, double* counts, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GNODE_B200_H */
