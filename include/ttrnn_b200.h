/*
 * ttrnn_b200 -- C ABI of the B200 (sm_100a) tensor-train recurrent engine.
 *
 * The reference (onucharles/tensorized-rnn) has no FFI: its boundary for this
 * path is the PyTorch nn.Module API (SURVEY.md section 8b).  This header is the
 * C-ABI a maintainer binds in place of the reference's Python hot loop; each
 * entry point names the reference code it replaces.  The Python mirror of the
 * module API (tensorized_rnn_b200/) binds exactly these symbols through ctypes;
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer to FP32
 *     data unless stated otherwise; the library never allocates or frees device
 *     memory (the caller owns every buffer, sized by the *_workspace_bytes calls)
 *   - all tensors are dense row-major: x (B, T, I), out (B, T, H), states (B, H)
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued, never synced.
 *     ttrnn_rnn_forward / ttrnn_rnn_backward may fork library-owned streams from it
 *     (row groups, backward overlap) and always join them back with an event before
 *     they return: for the caller the call stays ordered on `stream`
 *   - return 0 on success; non-zero = error, text via ttrnn_last_error()
 *   - there is no CPU path: without a CUDA device every compute call fails
 */
#ifndef TTRNN_B200_H
#define TTRNN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TTRNN_ABI_VERSION 4   /* 2: + cell step, ih route query, static kernel table; 3: execution plan carried by
                                 ttrnn_rnn_workspace, GEMM probe, GE2E head, dense cells; 4: row groups in the plan
                                 (ttrnn_rnn_row_groups, ttrnn_rnn_workspace_bytes_ex), per-step logging entry points,
                                 per-launch timing records -- additive: every ABI 3 signature is unchanged.  Still 4 with
                                 per-layer states: one more flag value (TTRNN_WS_LAYER_STATES) and two new symbols
                                 (ttrnn_dense_rnn_forward_ex / _backward_ex); no existing signature or default changes.
                                 Still 4 with bidirectional stacks: two new symbols (ttrnn_time_reverse_add,
                                 ttrnn_bidir_join), nothing existing changes.  Still 4 with inter-layer dropout: one more
                                 flag value (TTRNN_WS_DROPOUT), one struct and three new symbols (ttrnn_rnn_forward_dropout,
                                 ttrnn_rnn_backward_dropout, ttrnn_dropout_apply).  Still 4 with projected LSTM stacks:
                                 one more flag value (TTRNN_WS_PROJ), one struct and four new symbols
                                 (ttrnn_rnn_param_count_proj, ttrnn_rnn_workspace_bytes_proj, ttrnn_rnn_forward_proj,
                                 ttrnn_rnn_backward_proj).  Still 4 with projected dense LSTM stacks: four new symbols
                                 (ttrnn_dense_rnn_param_count_proj, ttrnn_dense_rnn_workspace_bytes_proj,
                                 ttrnn_dense_rnn_forward_proj, ttrnn_dense_rnn_backward_proj); nothing existing changes.
                                 Still 4 with variable-length rows: one more flag value (TTRNN_WS_LENGTHS) and seven new
                                 symbols (ttrnn_rnn_forward_lengths, ttrnn_rnn_backward_lengths,
                                 ttrnn_dense_rnn_forward_lengths, ttrnn_dense_rnn_backward_lengths,
                                 ttrnn_time_reverse_add_lengths, ttrnn_bidir_join_lengths, ttrnn_rnn_describe_ex); nothing
                                 existing changes */
#define TTRNN_MAX_CORES   6
#define TTRNN_MAX_LAYERS  8

#define TTRNN_CELL_LSTM 0   /* gates i, f, g, o  (tensorized_rnn/lstm.py:23-41)  */
#define TTRNN_CELL_GRU  1   /* gates r, z, n     (tensorized_rnn/gru.py:25-50)   */

/* One TT matrix W (M x N), M = prod(out_modes), N = prod(in_modes).
 * Core k is stored as the reference stores `weight_t` parameters
 * (t3nsor/layers.py:113, t3nsor/ops.py:47-51): shape
 * (ranks[k], out_modes[k], in_modes[k], ranks[k+1]), contiguous, cores
 * concatenated in order k = 0..d-1.  ranks[0] = ranks[d] = 1. */
typedef struct ttrnn_tt_shape {
    int32_t d;
    int32_t in_modes[TTRNN_MAX_CORES];
    int32_t out_modes[TTRNN_MAX_CORES];
    int32_t ranks[TTRNN_MAX_CORES + 1];
} ttrnn_tt_shape;

/* A stack of TT-LSTM / TT-GRU layers run over a whole sequence:
 * replaces LSTM.forward (tensorized_rnn/lstm.py:101-135) / GRU.forward
 * (tensorized_rnn/gru.py:104-136) with TT weights from tt_lstm.py:16-40 /
 * gru.py:148-172.
 *
 * Parameter blob layout (FP32, contiguous), per layer l = 0..L-1:
 *   [ih cores 0..d-1][ih bias (G*H) if has_bias][hh cores 0..d-1][hh bias (G*H) if has_bias]
 * which is the order of the reference's state_dict keys
 *   cell{l}.input_weights.parameters.{k}, cell{l}.input_weights.bias,
 *   cell{l}.hidden_weights.parameters.{k}, cell{l}.hidden_weights.bias.
 * Gradients come back in a blob of the same layout. */
typedef struct ttrnn_rnn_desc {
    int32_t cell;          /* TTRNN_CELL_*                                   */
    int32_t num_layers;    /* L                                              */
    int32_t input_size;    /* I                                              */
    int32_t hidden_size;   /* H                                              */
    int32_t has_bias;      /* both TTLinears of every cell carry a bias or none */
    int32_t seq_len;       /* T  (>= 1)                                      */
    int64_t batch;         /* B  (>= 1)                                      */
    ttrnn_tt_shape ih[TTRNN_MAX_LAYERS];   /* (G*H) x I for l = 0, (G*H) x H above */
    ttrnn_tt_shape hh[TTRNN_MAX_LAYERS];   /* (G*H) x H                      */
} ttrnn_rnn_desc;

#define TTRNN_PLAN_WORDS 24
typedef struct ttrnn_rnn_workspace {
    int64_t saved_bytes;        /* forward -> backward activations (training only) */
    int64_t fwd_scratch_bytes;  /* scratch for one forward call                    */
    int64_t bwd_scratch_bytes;  /* scratch for one backward call                   */
    /* Execution plan, written by ttrnn_rnn_workspace_bytes(): an opaque snapshot of every tuning option that
     * decides a buffer layout or a kernel route (chunk length, kept-activation mode, ih route, rows per CTA ...).
     * ttrnn_rnn_forward / ttrnn_rnn_backward run from THIS copy, never from the process-wide options, so
     * changing an option between a forward and its backward cannot change how `saved` is interpreted.
     * Pass the same struct to the forward and to its backward. */
    int64_t plan[TTRNN_PLAN_WORDS];
} ttrnn_rnn_workspace;

int         ttrnn_abi_version(void);
const char *ttrnn_last_error(void);            /* thread-local, never NULL */

/* number of floats in the parameter blob of `desc`; < 0 on a malformed desc */
int64_t ttrnn_rnn_param_count(const ttrnn_rnn_desc *desc);

int ttrnn_rnn_workspace_bytes(const ttrnn_rnn_desc *desc, ttrnn_rnn_workspace *ws);
/* The same with flags (they combine).  TTRNN_WS_WHOLE_BATCH: plan one row group, so that every layer's h_t / c_t
 * sequence is one (B,T,H) block of `saved` (required by ttrnn_rnn_saved_layout / ttrnn_rnn_backward_logged).
 * TTRNN_WS_LAYER_STATES: the forward / backward calls that run from this plan take PER-LAYER states, the contract of
 * torch.nn.LSTM: h0, c0, hT, cT, d_hT, d_cT, d_h0 and d_c0 are (L, B, H), layer l's block starting at l * B * H.  Each
 * may be NULL (an input state NULL = zeros).  Layer l starts from its own (h0, c0), returns its own (h_T, c_T), the
 * upstream d_hT / d_cT of layer l enters that layer's BPTT at its last step, and d_h0 / d_c0 receive each layer's own
 * gradient (not summed).  With it a stack can run one sequence in pieces: the final states of one call are the initial
 * states of the next.  The flag changes no kernel route, buffer size or result of the shared-state contract. */
#define TTRNN_WS_WHOLE_BATCH 1
#define TTRNN_WS_LAYER_STATES 2
/* TTRNN_WS_DROPOUT: the plan is for ttrnn_rnn_forward_dropout / ttrnn_rnn_backward_dropout (below).  `saved` grows by
 * (L-1) * B * T * H floats, the masked inputs of layers 1 .. L-1, and the forward scratch by one (B, T, H) block; every
 * other size, offset and route is the one of the plan without the flag.  ttrnn_rnn_forward / ttrnn_rnn_backward /
 * ttrnn_rnn_backward_logged reject a plan that carries it. */
#define TTRNN_WS_DROPOUT 4
int ttrnn_rnn_workspace_bytes_ex(const ttrnn_rnn_desc *desc, int32_t flags, ttrnn_rnn_workspace *ws);

/* Forward over the whole stack.  h0 / c0 may be NULL (zeros); one (h0, c0) seeds
 * every layer (lstm.py:120-121) unless the plan carries TTRNN_WS_LAYER_STATES (see above).  c0 / cT / d_c* are ignored for GRU.
 * `ws` = the struct ttrnn_rnn_workspace_bytes() filled for this desc (sizes + execution plan).
 * `saved` NULL = inference (nothing kept for backward).  Returns outputs of the
 * last layer for every t, and (h_T, c_T) of the last layer (lstm.py:135). */
int ttrnn_rnn_forward(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws,
                      const float *x, const float *h0, const float *c0,
                      const float *params, float *out, float *hT, float *cT,
                      void *saved, void *scratch, void *stream);

/* BPTT through the stack: what autograd does for the reference
 * (SURVEY.md section 8a-10).  d_out (B,T,H), d_hT, d_cT: upstream gradients (any may be
 * NULL = zero).  d_params is OVERWRITTEN with the gradient blob.  d_x (B,T,I) may
 * be NULL.  d_h0 / d_c0 (B,H) may be NULL; they receive the SUM over layers
 * because every layer shares the same initial state (per layer under TTRNN_WS_LAYER_STATES). */
int ttrnn_rnn_backward(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws,
                       const float *x, const float *h0, const float *c0,
                       const float *params, const float *out, const void *saved,
                       const float *d_out, const float *d_hT, const float *d_cT,
                       float *d_params, float *d_x, float *d_h0, float *d_c0,
                       void *scratch, void *stream);

/* log_grads=True (tensorized_rnn/lstm.py:35-39,66-80, gru.py:47-48,76-85, rnn_utils.py:127-172): the reference hooks
 * every cell call and logs, per layer and timestep, mean_b ||v||^2 and mean_b log ||v||^2 of h_t, c_t and of the
 * gradients reaching them.  Fused form: the training forward already keeps every layer's h_t / c_t sequence
 * (ttrnn_rnn_saved_layout says where: float offsets into `saved`; hs_off = -1 means the last layer, whose sequence is
 * `out`; cs_off = -1 for GRU), ttrnn_rnn_backward_logged additionally makes the BPTT kernel of layer l write the TOTAL
 * gradient of h_t (and c_t, LSTM) of every step -- what the reference's tensor hooks on hy / cy receive -- into
 * dh_log / dc_log, (L,B,T,H) each (dc_log may be NULL), and ttrnn_step_norms reduces a (B,T,H) block to the two logged
 * statistics: out[0:T] = mean_b ||v[b,t]||^2, out[T:2T] = mean_b log ||v[b,t]||^2. */
int ttrnn_rnn_saved_layout(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws, int32_t layer,
                           int64_t *hs_off, int64_t *cs_off);
int ttrnn_rnn_backward_logged(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws,
                              const float *x, const float *h0, const float *c0,
                              const float *params, const float *out, const void *saved,
                              const float *d_out, const float *d_hT, const float *d_cT,
                              float *d_params, float *d_x, float *d_h0, float *d_c0,
                              void *scratch, void *stream, float *dh_log, float *dc_log);
int ttrnn_step_norms(const float *v, int64_t B, int32_t T, int32_t H, float *out, void *stream);

/* Inter-layer dropout, the `dropout` argument of torch.nn.LSTM / GRU: the output sequence of every layer but the last is
 * multiplied by mask / (1 - p) before the next layer reads it; mask is Bernoulli(1 - p) per element.  The final states
 * are never masked.  The mask is a pure function of (seed, offset, boundary k = the layer whose output it masks, GLOBAL
 * batch row b, t, feature j): Philox4x32-10 with key = seed and counter = (e / 4 as 64 bits with k in bits 48..63,
 * offset), e = (b * T + t) * F + j, element e kept when its 32-bit word is below (1 - p) * 2^32.  So it does not depend on
 * row groups, time chunks, rows per CTA or streams, and the backward regenerates it from (seed, offset): nothing of the
 * mask is stored.  p must be in [0, 1]; p = 1 zeroes the input of the layers above the first (and its gradient).
 *
 * ttrnn_rnn_forward_dropout / ttrnn_rnn_backward_dropout: ttrnn_rnn_forward / _backward with the mask applied between
 * the layers.  The plan must carry TTRNN_WS_DROPOUT when dp->p > 0 (a plan with it also runs p = 0: the mask keeps every
 * element); a forward and its backward take the same `dp`.
 *
 * ttrnn_dropout_apply: the mask of boundary `boundary` over a (B, T, F) block whose first row is global row `row0`.
 *   backward == 0: y = x * mask / (1 - p); unless y_rev is NULL also y_rev[b,t] = y[b,T-1-t] (the input of a
 *                  bidirectional layer's reverse direction).  y may alias x.
 *   backward != 0: y = (x + rev(y_rev)) * mask / (1 - p), y_rev read as the gradient of the reversed copy (NULL = zero):
 *                  the adjoint of the forward.  y may alias x, not y_rev.
 * Multiplying a ones block gives the mask / (1 - p) itself. */
typedef struct ttrnn_dropout {
    float p;              /* drop probability, 0 <= p <= 1          */
    int32_t reserved;     /* 0                                      */
    uint64_t seed;        /* Philox key                             */
    uint64_t offset;      /* Philox counter words 2-3               */
} ttrnn_dropout;
int ttrnn_rnn_forward_dropout(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws,
                              const float *x, const float *h0, const float *c0,
                              const float *params, float *out, float *hT, float *cT,
                              void *saved, void *scratch, void *stream, const ttrnn_dropout *dp);
int ttrnn_rnn_backward_dropout(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws,
                               const float *x, const float *h0, const float *c0,
                               const float *params, const float *out, const void *saved,
                               const float *d_out, const float *d_hT, const float *d_cT,
                               float *d_params, float *d_x, float *d_h0, float *d_c0,
                               void *scratch, void *stream, const ttrnn_dropout *dp);
int ttrnn_dropout_apply(int64_t B, int32_t T, int32_t F, int64_t row0, int32_t boundary, int32_t backward,
                        const ttrnn_dropout *dp, const float *x, float *y, float *y_rev, void *stream);

/* Projected LSTM stacks (LSTMP), the `proj_size` of torch.nn.LSTM: each layer computes m_t = o_t * tanh(c_t) (H wide) and
 * outputs h_t = W_hr m_t (P < H wide), which is also the next step's hh input.  W_hr of layer l is a TT matrix P x H
 * without bias; the recurrent kernels contract it between the gate math of one step and the hh chain of the next.
 *
 *   - desc->cell must be TTRNN_CELL_LSTM; desc->hh[l] is 4H x P, desc->ih[l] for l >= 1 is 4H x P.
 *   - Parameter blob, per layer: [ih cores][ih bias][hh cores][hh bias][hr cores], the order of the state_dict keys
 *     ..., cell{l}.hidden_weights.bias, cell{l}.projection_weights.parameters.{k}.
 *   - Every h-state buffer is P wide: out (B, T, P), h0, hT, d_hT, d_h0 (B, P).  The c-state buffers c0, cT, d_cT, d_c0
 *     stay (B, H).  Under TTRNN_WS_LAYER_STATES the layer stride is B * P for the h states and B * H for the c states.
 *   - The plan comes from ttrnn_rnn_workspace_bytes_proj (flags as for ttrnn_rnn_workspace_bytes_ex; TTRNN_WS_PROJ is
 *     implied, TTRNN_WS_WHOLE_BATCH has no effect: a projected plan is always one row group).  ttrnn_rnn_forward /
 *     _backward / _forward_dropout / _backward_dropout / _backward_logged / ttrnn_rnn_saved_layout refuse such a plan, and
 *     ttrnn_rnn_workspace_bytes_ex refuses the flag; the _proj calls refuse a plan without it, a GRU descriptor, a NULL
 *     `pj` and hr shapes that are not P x H.
 *   - `dp` may be NULL (no dropout).  With TTRNN_WS_DROPOUT the masked layer inputs kept in `saved` take
 *     (L-1) * B * T * P floats and the mask covers the P-wide layer output.
 *   - Projected layers run on the runtime-shape recurrent kernels (k_rnn_fwd_proj / k_rnn_bwd_proj); no statically
 *     specialised kernel and no rank padding applies to them. */
#define TTRNN_WS_PROJ 8
typedef struct ttrnn_rnn_proj {
    int32_t proj_size;                   /* P >= 1, P < hidden_size; desc->cell must be TTRNN_CELL_LSTM */
    int32_t reserved;                    /* 0                                                           */
    ttrnn_tt_shape hr[TTRNN_MAX_LAYERS]; /* W_hr of layer l: P x H                                      */
} ttrnn_rnn_proj;
int64_t ttrnn_rnn_param_count_proj(const ttrnn_rnn_desc *desc, const ttrnn_rnn_proj *pj);
int ttrnn_rnn_workspace_bytes_proj(const ttrnn_rnn_desc *desc, const ttrnn_rnn_proj *pj, int32_t flags,
                                   ttrnn_rnn_workspace *ws);
int ttrnn_rnn_forward_proj(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws,
                           const float *x, const float *h0, const float *c0,
                           const float *params, float *out, float *hT, float *cT,
                           void *saved, void *scratch, void *stream, const ttrnn_rnn_proj *pj, const ttrnn_dropout *dp);
int ttrnn_rnn_backward_proj(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws,
                            const float *x, const float *h0, const float *c0,
                            const float *params, const float *out, const void *saved,
                            const float *d_out, const float *d_hT, const float *d_cT,
                            float *d_params, float *d_x, float *d_h0, float *d_c0,
                            void *scratch, void *stream, const ttrnn_rnn_proj *pj, const ttrnn_dropout *dp);

/* Bidirectional stacks (the contract of torch.nn.LSTM(bidirectional=True)).  The library has no whole-stack
 * bidirectional call: the reverse direction of a layer is the ordinary one-layer ttrnn_rnn_forward / _backward (or
 * ttrnn_dense_rnn_*) run on the layer input reversed in time, whose outputs then come back reversed in time.  These two
 * memory-bound calls move the (B, T, .) blocks between the directions.  Every output element takes at most one FP32 add.
 *
 * ttrnn_time_reverse_add: y[b,t,:] = a[b,t,:] + r[b,T-1-t,:] over (B, T, F); a or r may be NULL (= zero).  With a NULL
 * it reverses a layer-0 input for the reverse direction; with both it forms the layer-0 input gradient
 * d_x = d_x_forward + reverse(d_x_reverse).  y must not alias a or r.
 *
 * ttrnn_bidir_join, H = hidden size, out_f / out_r = the forward / reverse direction's outputs (B, T, H), the latter in
 * reversed time:
 *   backward == 0: p = out_f, q = out_r (both required); writes the next layer's input u = y (B, T, 2H),
 *                  y[b,t] = [out_f[b,t] | out_r[b,T-1-t]], and, unless v is NULL (the last layer), v = y_rev (B, T, 2H),
 *                  y_rev[b,s] = y[b,T-1-s], the input of the next layer's reverse direction;
 *   backward != 0: p = dy, q = dy_rev (the gradients of y and y_rev; either may be NULL = zero); writes
 *                  u = d_out_f[b,t] = dy[b,t,:H] + dy_rev[b,T-1-t,:H] and v = d_out_r[b,s] = dy[b,T-1-s,H:] + dy_rev[b,s,H:],
 *                  (B, T, H) each.
 * Outputs must not alias inputs. */
int ttrnn_time_reverse_add(int64_t B, int32_t T, int32_t F, const float *a, const float *r, float *y, void *stream);
int ttrnn_bidir_join(int64_t B, int32_t T, int32_t H, int32_t backward, const float *p, const float *q, float *u,
                     float *v, void *stream);

/* Variable-length rows (DESIGN.md §4.22), the PackedSequence input of torch.nn.LSTM / GRU in its padded form: row b of a
 * (B, T, .) batch is len_b steps long, 1 <= len_b <= T.  `lengths` is a DEVICE array of B int32.
 * PRECONDITION, not checked on the device: 1 <= lengths[b] <= T for every b; and the padded inputs x[b, t >= len_b] must be
 * finite (their products with zero gate gradients enter dW_ih).
 *
 * No recurrent kernel sees the lengths.  After every write of the ih projection (forward and backward recompute) the gate
 * pre-activations of each padded (b, t) are overwritten so that the row is frozen: LSTM i = -inf, f = +inf, g = o = 0
 * (c_t = c_{t-1} exactly), GRU z = +inf, r = n = 0 (h_t = h_{t-1} exactly).  So every route that reads a materialised ih
 * projection runs unchanged; the rank-one input mode (I = 1, layer 0) builds its projection inside the kernel and is not
 * taken under lengths.  What the calls return, torch's contract:
 *   - out[b, t] = 0 for t >= len_b; the caller's d_out there is ignored (never written);
 *   - h_n of every layer (hT, also per layer under TTRNN_WS_LAYER_STATES) is the state after step len_b - 1, and c_n (LSTM)
 *     likewise; their gradients enter at that step;
 *   - d_x[b, t] = 0 for t >= len_b.
 *
 * TTRNN_WS_LENGTHS: the plan is for ttrnn_rnn_forward_lengths / ttrnn_rnn_backward_lengths (it combines with the other
 * flags of ttrnn_rnn_workspace_bytes_ex and ttrnn_rnn_workspace_bytes_proj).  The backward scratch grows by one (B, T, W)
 * block, W the output width; every other entry point refuses such a plan, and the _lengths calls refuse a plan without it.
 * There is no logged (log_grads) form.
 *
 * ttrnn_rnn_forward_lengths / _backward_lengths: the arguments of the _proj calls with `pj` optional (NULL = unprojected;
 * it must be given exactly when the plan was sized with TTRNN_WS_PROJ), `dp` optional (NULL = no dropout), then lengths.
 * ttrnn_dense_rnn_forward_lengths / _backward_lengths: the arguments of the dense _proj calls, proj_size 0 = unprojected,
 * then lengths; flags as for the dense _ex calls (TTRNN_WS_LENGTHS may be passed and changes nothing); the workspace
 * sizes are those of ttrnn_dense_rnn_workspace_bytes (_proj with proj_size > 0).
 * ttrnn_time_reverse_add_lengths / ttrnn_bidir_join_lengths: ttrnn_time_reverse_add / ttrnn_bidir_join with every row
 * reversed over its own length, x'[b, t] = x[b, len_b - 1 - t] for t < len_b; every output position t >= len_b is 0. */
#define TTRNN_WS_LENGTHS 16
int ttrnn_rnn_forward_lengths(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws,
                              const float *x, const float *h0, const float *c0,
                              const float *params, float *out, float *hT, float *cT,
                              void *saved, void *scratch, void *stream, const ttrnn_rnn_proj *pj, const ttrnn_dropout *dp,
                              const int32_t *lengths);
int ttrnn_rnn_backward_lengths(const ttrnn_rnn_desc *desc, const ttrnn_rnn_workspace *ws,
                               const float *x, const float *h0, const float *c0,
                               const float *params, const float *out, const void *saved,
                               const float *d_out, const float *d_hT, const float *d_cT,
                               float *d_params, float *d_x, float *d_h0, float *d_c0,
                               void *scratch, void *stream, const ttrnn_rnn_proj *pj, const ttrnn_dropout *dp,
                               const int32_t *lengths);
int ttrnn_time_reverse_add_lengths(int64_t B, int32_t T, int32_t F, const float *a, const float *r, float *y,
                                   const int32_t *lengths, void *stream);
int ttrnn_bidir_join_lengths(int64_t B, int32_t T, int32_t H, int32_t backward, const float *p, const float *q, float *u,
                             float *v, const int32_t *lengths, void *stream);

/* Stand-alone TT linear map y = x W^T + bias over `rows` rows:
 * replaces TTLinear.forward (t3nsor/layers.py:121-127) -> tt_dense_matmul
 * (t3nsor/ops.py:54-93).  bias may be NULL. */
int64_t ttrnn_ttlinear_param_count(const ttrnn_tt_shape *shape);
int64_t ttrnn_ttlinear_workspace_bytes(const ttrnn_tt_shape *shape, int64_t rows);
int ttrnn_ttlinear_forward(const ttrnn_tt_shape *shape, int64_t rows, const float *x,
                           const float *cores, const float *bias, float *y,
                           void *scratch, void *stream);
/* d_cores / d_bias are OVERWRITTEN; d_x and d_bias may be NULL. */
int ttrnn_ttlinear_backward(const ttrnn_tt_shape *shape, int64_t rows, const float *x,
                            const float *cores, const float *dy,
                            float *d_x, float *d_cores, float *d_bias,
                            void *scratch, void *stream);

/* One cell step from the two pre-activation blocks a = W_ih x + b_ih and u = W_hh h + b_hh,
 * both (B, G*H): the gate math and state update of LSTMCell.forward
 * (tensorized_rnn/lstm.py:26-32) / GRUCell.forward (tensorized_rnn/gru.py:33-44).  Serves the
 * module mirror's cell-step mode, i.e. the reference features that need one module call per
 * timestep: is_naive=True (TTLinearSet, tensorized_rnn/tt_linearset.py:27-38) and
 * log_grads=True (hooks of tensorized_rnn/lstm.py:35-39,66-80, gru.py:47-48,76-85).
 * LSTM: h_prev may be NULL; GRU: c_prev / c / dc / dc_prev are ignored. */
int ttrnn_cell_forward(int32_t cell, int64_t B, int32_t H, const float *a, const float *u,
                       const float *h_prev, const float *c_prev, float *h, float *c, void *stream);
/* Backward of one step (SURVEY.md section 8a-10).  dh / dc may be NULL (= zero).  da, du (B, G*H),
 * dh_prev (direct term only: GRU dh*z, LSTM zero) and dc_prev are OVERWRITTEN.  dc_total (optional,
 * LSTM) receives dL/dc_t including the path through h_t = o * tanh(c_t): the value a tensor hook
 * on the reference's `cy` sees (lstm.py:38-39), which log_grads records. */
int ttrnn_cell_backward(int32_t cell, int64_t B, int32_t H, const float *a, const float *u,
                        const float *h_prev, const float *c_prev, const float *dh, const float *dc,
                        float *da, float *du, float *dh_prev, float *dc_prev, float *dc_total,
                        void *stream);

/* Dense LSTM / GRU baselines through the same engine (SURVEY.md 8f-3): the reference's `LSTM` / `GRU` modules with dense
 * nn.Linear weights (tensorized_rnn/lstm.py:7-41,44-135, gru.py:11-50,52-136), selected by pmnist_test.py without --tt and
 * by SpeakerEncoder(compression=None).  Same forward / backward contract as ttrnn_rnn_forward / _backward.
 * Parameter blob, per layer: [W_ih (G*H x in)] [b_ih (G*H): GRU with bias only] [W_hh (G*H x H)] [b_hh (G*H) with bias]
 * -- the reference's state_dict order cell{l}.input_weights.weight [.bias], cell{l}.hidden_weights.weight [.bias]
 * (the dense LSTMCell gives its input map no bias, lstm.py:17-18).  The ih projection, dX and both weight gradients are
 * batched over the whole sequence as tensor-core GEMMs; the recurrence is one GEMM + one fused gate kernel per step.
 * hidden_size must be a multiple of 128 (GEMM tile width); d_x needs input_size % 128 == 0. */
typedef struct ttrnn_dense_desc {
    int32_t cell, num_layers, input_size, hidden_size, has_bias, seq_len;
    int64_t batch;
} ttrnn_dense_desc;
int64_t ttrnn_dense_rnn_param_count(const ttrnn_dense_desc *desc);
int ttrnn_dense_rnn_workspace_bytes(const ttrnn_dense_desc *desc, int64_t *saved_bytes, int64_t *scratch_bytes);
/* `saved` is required (training and inference): it holds the pre-activation blocks of every step. */
int ttrnn_dense_rnn_forward(const ttrnn_dense_desc *desc, const float *x, const float *h0, const float *c0,
                            const float *params, float *out, float *hT, float *cT,
                            void *saved, void *scratch, void *stream);
/* `saved` is consumed (overwritten with gradients): one backward per forward. */
int ttrnn_dense_rnn_backward(const ttrnn_dense_desc *desc, const float *x, const float *h0, const float *c0,
                             const float *params, const float *out, void *saved,
                             const float *d_out, const float *d_hT, const float *d_cT,
                             float *d_params, float *d_x, float *d_h0, float *d_c0,
                             void *scratch, void *stream);
/* The same with flags: TTRNN_WS_LAYER_STATES makes every state buffer (L, B, H), as for ttrnn_rnn_forward.  Pass the same
 * flags to a forward and its backward.  (Under that flag d_h0 / d_c0 of a layer are written where its h0 / c0 is given.) */
int ttrnn_dense_rnn_forward_ex(const ttrnn_dense_desc *desc, const float *x, const float *h0, const float *c0,
                               const float *params, float *out, float *hT, float *cT,
                               void *saved, void *scratch, void *stream, int32_t flags);
int ttrnn_dense_rnn_backward_ex(const ttrnn_dense_desc *desc, const float *x, const float *h0, const float *c0,
                                const float *params, const float *out, void *saved,
                                const float *d_out, const float *d_hT, const float *d_cT,
                                float *d_params, float *d_x, float *d_h0, float *d_c0,
                                void *scratch, void *stream, int32_t flags);
/* Projected dense LSTM stacks (LSTMP), the `proj_size` of torch.nn.LSTM: each layer computes m_t = o_t * tanh(c_t) (H wide)
 * and outputs h_t = W_hr m_t (P < H wide, no bias), which is also the next step's hh input.  Each call takes the arguments
 * of its counterpart above (the _ex form for forward / backward) plus proj_size = P.
 *   - desc->cell must be TTRNN_CELL_LSTM; 1 <= P < hidden_size and P % 128 == 0 (P is N of the per-step projection GEMM
 *     and of the dh carry GEMM).  proj_size = 0 is refused: that is the unprojected stack of the calls above.
 *   - Parameter blob, per layer: [W_ih (4H x in)] [W_hh (4H x P)] [b_hh (4H) with bias] [W_hr (P x H)], the state_dict
 *     order; `in` is P for layers >= 1 (torch.nn.LSTM: weight_ih_l{l}, weight_hh_l{l}, bias_hh_l{l}, weight_hr_l{l}, with
 *     bias_ih_l{l} = 0).
 *   - Every h-state buffer is P wide: out (B, T, P), h0, hT, d_hT, d_h0 (B, P).  The c-state buffers c0, cT, d_cT, d_c0
 *     stay (B, H).  Under TTRNN_WS_LAYER_STATES the layer stride is B * P for the h states and B * H for the c states.
 *   - Per step, the forward runs the hh GEMM (K = P), the gate kernel (writes c_t and m_t) and h_t = m_t W_hr^T; the
 *     backward forms dh_t, runs dm_t = dh_t W_hr, the gate backward and the carry du_t W_hh.  dW_hr = sum_t dh_t^T m_t
 *     is one GEMM over all B * T rows after the loop. */
int64_t ttrnn_dense_rnn_param_count_proj(const ttrnn_dense_desc *desc, int32_t proj_size);
int ttrnn_dense_rnn_workspace_bytes_proj(const ttrnn_dense_desc *desc, int64_t *saved_bytes, int64_t *scratch_bytes,
                                         int32_t proj_size);
int ttrnn_dense_rnn_forward_proj(const ttrnn_dense_desc *desc, const float *x, const float *h0, const float *c0,
                                 const float *params, float *out, float *hT, float *cT,
                                 void *saved, void *scratch, void *stream, int32_t flags, int32_t proj_size);
int ttrnn_dense_rnn_backward_proj(const ttrnn_dense_desc *desc, const float *x, const float *h0, const float *c0,
                                  const float *params, const float *out, void *saved,
                                  const float *d_out, const float *d_hT, const float *d_cT,
                                  float *d_params, float *d_x, float *d_h0, float *d_c0,
                                  void *scratch, void *stream, int32_t flags, int32_t proj_size);
/* Variable-length rows of a dense stack: see TTRNN_WS_LENGTHS above. */
int ttrnn_dense_rnn_forward_lengths(const ttrnn_dense_desc *desc, const float *x, const float *h0, const float *c0,
                                    const float *params, float *out, float *hT, float *cT,
                                    void *saved, void *scratch, void *stream, int32_t flags, int32_t proj_size,
                                    const int32_t *lengths);
int ttrnn_dense_rnn_backward_lengths(const ttrnn_dense_desc *desc, const float *x, const float *h0, const float *c0,
                                     const float *params, const float *out, void *saved,
                                     const float *d_out, const float *d_hT, const float *d_cT,
                                     float *d_params, float *d_x, float *d_h0, float *d_c0,
                                     void *scratch, void *stream, int32_t flags, int32_t proj_size, const int32_t *lengths);

/* GE2E head on the device (SURVEY.md 8f-4): the part of the speaker-encoder training step the reference runs on the CPU
 * after every RNN pass (experiments/speaker_verification/encoder/main.py:279-280 moves the embeddings to `loss_device`).
 *
 * ttrnn_embed_forward: embeds = relu(x) / ||relu(x)||_2 per row (speaker_encoder.py:86-89); x, y (rows, E),
 * inv_norm (rows) is kept for the backward.  ttrnn_embed_backward: dx from dy. */
int ttrnn_embed_forward(int64_t rows, int32_t E, const float *x, float *y, float *inv_norm, void *stream);
int ttrnn_embed_backward(int64_t rows, int32_t E, const float *x, const float *y, const float *inv_norm,
                         const float *dy, float *dx, void *stream);
/* GE2E softmax loss of `embeds` (S speakers, U utterances each, E features; row = s * U + u), training form of
 * SpeakerEncoder.similarity_matrix / .loss (speaker_encoder.py:93-141, 143-156, enrollment_embeds = None): inclusive and
 * exclusive centroids, sim[(s,u), j], logits = wb[0] * sim + wb[1], mean cross-entropy against the speaker index.
 * wb: device pointer to {similarity_weight, similarity_bias}; loss: device scalar; sim_out (optional, S*U x S): the scaled
 * similarity matrix wb[0] * sim + wb[1] that SpeakerEncoder.similarity_matrix returns (speaker_encoder.py:139).  `workspace` (ttrnn_ge2e_workspace_bytes) carries centroids / probabilities to the backward,
 * which writes d_embeds (S*U x E) and d_wb[2] for an upstream gradient *dloss (device scalar). */
int64_t ttrnn_ge2e_workspace_bytes(int32_t S, int32_t U, int32_t E);
int ttrnn_ge2e_loss_forward(int32_t S, int32_t U, int32_t E, const float *embeds, const float *wb, float *loss,
                            float *sim_out, void *workspace, void *stream);
int ttrnn_ge2e_loss_backward(int32_t S, int32_t U, int32_t E, const float *embeds, const float *wb,
                             const float *dloss, void *workspace, float *d_embeds, float *d_wb, void *stream);

/* Utterance-level embeddings (SpeakerEncoder.embed_utterances, DESIGN.md §4.21): every fixed-length window of every utterance
 * goes through one stack call; these two steps surround it.  All pointers are device pointers.
 *
 * ttrnn_partials_gather: builds the window block out (W, P, F) from the packed frames (total_frames, F) of the utterances
 * concatenated in order.  Window w copies the rows win_first[w] .. win_first[w] + win_valid[w] - 1 to out[w, 0 .. valid-1, :]
 * and writes zeros to out[w, valid .. P-1, :].  A pure copy (bit-exact).
 * PRECONDITION, not checked on the device: for every w, 0 <= win_first[w], 1 <= win_valid[w] <= P and
 * win_first[w] + win_valid[w] <= total_frames.
 *
 * ttrnn_segment_mean_normalize_forward: rows x (R, E) in n_seg consecutive segments, seg_off (n_seg + 1, int64) with
 * seg_off[0] = 0 and seg_off[n_seg] = R.  y (n_seg, E): y[s] = m / ||m||_2 with m the mean of rows seg_off[s] ..
 * seg_off[s+1] - 1; inv_norm (n_seg) = 1 / ||m||_2, kept for the backward.  ttrnn_segment_mean_normalize_backward writes
 * dx (R, E): dx[r] = (dy[s] - y[s] (y[s] . dy[s])) * inv_norm[s] / count_s for every row r of segment s.
 * PRECONDITION, not checked on the device: seg_off non-decreasing; a segment is empty when two offsets are equal, and then
 * its y row is NaN (0 / 0).  Sums run in a fixed order without atomics: two calls are bit-identical. */
int ttrnn_partials_gather(int64_t W, int32_t P, int32_t F, const float *frames, int64_t total_frames,
                          const int64_t *win_first, const int32_t *win_valid, float *out, void *stream);
int ttrnn_segment_mean_normalize_forward(int64_t n_seg, int32_t E, const float *x, const int64_t *seg_off,
                                         float *y, float *inv_norm, void *stream);
int ttrnn_segment_mean_normalize_backward(int64_t n_seg, int32_t E, const int64_t *seg_off, const float *y,
                                          const float *inv_norm, const float *dy, float *dx, void *stream);

/* Measurement helpers (bench.py only).
 * ttrnn_ffma_probe: dependent-chain-free FP32 FFMA loop on every SM; writes the
 * number of FLOPs executed to *flops_out (host) and leaves a checksum in sink
 * (device, >= 4 bytes).  Time it with CUDA events to get the FP32 roofline peak. */
int ttrnn_ffma_probe(int32_t iters, float *sink, double *flops_out, void *stream);
/* counts kernels launched by this library since the last reset (host counter) */
int64_t ttrnn_launch_count(int32_t reset);
/* Per-kernel device timing for the roofline report.  ttrnn_kernel_timing(1) makes every launch
 * of the main kernel groups record a CUDA-event pair on its own stream (bounded pool; extra
 * launches are simply not recorded); ttrnn_kernel_timing(0) stops.  ttrnn_kernel_times()
 * synchronises the recorded events, adds their elapsed milliseconds into ms[kind] and the
 * number of recorded launches into count[kind], and clears the pool.  Kinds: */
#define TTRNN_K_TTLINEAR_FWD 0
#define TTRNN_K_RNN_FWD      1
#define TTRNN_K_RNN_BWD      2
#define TTRNN_K_TTLINEAR_BWD 3
#define TTRNN_K_GEMM_FWD     4   /* dense-route ih projection (tensor-core or FFMA row GEMM)          */
#define TTRNN_K_GEMM_DX      5   /* dense-route dX = delta * W                                         */
#define TTRNN_K_GEMM_DW      6   /* dense-route core-gradient accumulation dW^T = X^T delta (ih and hh) */
#define TTRNN_K_KINDS        7
int ttrnn_kernel_timing(int32_t enable);
int ttrnn_kernel_times(double *ms /*[TTRNN_K_KINDS]*/, int64_t *count /*[TTRNN_K_KINDS]*/);
/* Per-launch records of the last ttrnn_kernel_times() call: 6 doubles per record = {kind, rows per CTA, grid size (CTAs),
 * batch rows of the launch, timesteps of the launch, milliseconds}; all but kind and milliseconds are 0 for the kinds
 * that are not recurrent kernels, except that a statically specialised TT-matvec kernel (kinds 0 and 3) reports its rows
 * per CTA, grid and rows (batch rows x timesteps of the chunk).
 * Returns the number of records (buf NULL: just the count).  bench.py reports the recurrent kernels per variant from it. */
int64_t ttrnn_kernel_launch_records(double *buf, int64_t cap_records);

/* Which contraction order the batched ih projection of `layer` uses: 0 = TT chain core by core
 * (t3nsor/ops.py:81-90), 1 = dense route (W_ih formed once per call from the cores, then one dense
 * FP32 contraction per row; chosen when I*G*H <= dense_ih_ratio % of the chain's multiply-adds),
 * 2 = rank-one input mode (I = 1).  Also reports both costs per row.  < 0 on a malformed desc. */
int ttrnn_rnn_ih_route(const ttrnn_rnn_desc *desc, int32_t layer, int64_t *chain_macs_per_row,
                       int64_t *dense_macs_per_row);

/* Execution plan of `desc` under the current options, as text: first line "chunk_steps=.. sms=.. tc_gemm=.. rank_padded=.. bwd_overlap=..", then one
 * line per layer of key=value pairs (ih_route, ih_fwd_tc / ih_dw_tc = tensor-core GEMMs used, fwd_kernel, fwd_rows =
 * batch rows per CTA, save_mode = 2 with kept gate activations else 0, and with training != 0: bwd_kernel, bwd_rows, bwd_phase_rows, optional second phase,
 * hh_dw, hh_dw_tc).  Needs a CUDA device (the plan depends on its SM count).  Returns characters written, < 0 on error. */
int ttrnn_rnn_describe(const ttrnn_rnn_desc *desc, int32_t training, char *buf, int32_t cap);
/* The same for the plan that ttrnn_rnn_workspace_bytes_ex(desc, flags, .) would size: TTRNN_WS_WHOLE_BATCH plans one row group
 * and TTRNN_WS_LENGTHS leaves out the rank-one input mode (I = 1), which variable-length rows do not take; the other flags
 * change no route.  TTRNN_WS_PROJ is refused (projected stacks run on the runtime-shape kernels only). */
int ttrnn_rnn_describe_ex(const ttrnn_rnn_desc *desc, int32_t flags, int32_t training, char *buf, int32_t cap);
/* Row-group split of `desc` under the current options (round 2, "row_groups"): multi-layer stacks whose batch does not
 * fill whole waves of CTAs are cut into two independent row groups that run the stack on two streams, so that the SMs
 * a layer-pass of one group leaves idle run the next layer of the other (the reference has no counterpart: its layer
 * loop, lstm.py:123-133, is sequential over the whole batch).  Returns the number of groups (1 or 2; < 0 on error) and
 * their row counts.  sms > 0 plans for that SM count without touching a device (tests); sms <= 0 asks the device. */
int ttrnn_rnn_row_groups(const ttrnn_rnn_desc *desc, int32_t sms, int64_t *rows /*[2]*/);
/* launches of the tcgen05 (tensor-core, 3xTF32) GEMM kernels since the last reset (subset of ttrnn_launch_count) */
int64_t ttrnn_tc_launch_count(int32_t reset);

/* Host-only: text table of the statically specialised kernels compiled into the library, one line per
 * kernel "kind|name|rows_per_cta|shared_memory_bytes|fits" (fits = 1 when it is within the 227 KB opt-in limit
 * and can be selected).  Returns the number of characters written, < 0 on a bad buffer. */
int ttrnn_static_kernel_table(char *buf, int32_t cap);
/* Host-only: the same kernels in the same order, one line per kernel with the key that identifies it:
 * "kind|name|rows_per_cta|cell|mode|saved|split|merged" (cell = TTRNN_CELL_*, mode = input mode 0 projected /
 * 1 rank-one, saved = 2 when the BPTT kernel consumes kept gate activations, split = 1 for dX-only BPTT kernels and for
 * the TT-matvec backward kernels without dX, merged = 1 for the chain with cores 0 and 1 contracted; -1 where a column
 * does not apply to the TT-matvec kernels).  Returns the number of characters written, < 0 on a bad buffer. */
int ttrnn_static_kernel_keys(char *buf, int32_t cap);
/* Host-only: launches of every statically specialised kernel since the last reset, one counter per line of
 * ttrnn_static_kernel_table (and ttrnn_static_kernel_keys) in their order; copies min(cap, entries) counters into
 * counts (may be NULL), zeroes them when reset != 0.  Returns the number of entries. */
int ttrnn_static_kernel_launches(int64_t *counts, int32_t cap, int32_t reset);

/* Tuning knobs (process-wide; also read from the environment at load time):
 *   "rows_per_cta"  batch rows owned by one CTA of the recurrent kernels (0 = auto)
 *   "chunk_steps"   timesteps per ih-projection chunk (0 = auto, bounded by memory)
 *   "chunk_bytes"   byte budget of one ih-projection chunk (default 4 GiB)
 *   "static_kernels" 0 = always use the runtime-shape kernels
 *   "static_rows_fwd" / "static_rows_bwd"  force the rows-per-CTA variant of the static kernels
 *   "save_u_bytes"  budget for keeping only the hh pre-activations (G*H floats per row and step) so that
 *                   backward skips the final stage of the chain recompute (default 16 GiB; 0 = recompute)
 *   "row_plan"      0 = one kernel variant per BPTT launch (default 1: a tail variant with fewer rows per
 *                   CTA may run the rows that do not fill a whole wave)
 *   "gemm_wide"     1 = 128 x 256 CTA tiles for the dense-route row GEMMs (default 0: measured slower)
 *   "split_kept"    kept gates: 0 = never use the dX-only BPTT variants (gate gradients + dX chain in the recurrent
 *                   kernel, hh core gradients accumulated densely outside); default 1 where registered (cfg3 shape)
 *   "dense_hh_dw"   split backward only: 0 = hh core gradients by a second chain pass per row instead of the dense
 *                   accumulation dW_hh^T = H_prev^T delta + projection onto the cores (default 1)
 *   "dense_ih"      0 = never take the dense route of the ih projection (default 1)
 *   "dense_ih_ratio" dense route allowed while I*G*H * 100 <= chain multiply-adds * ratio (default 130)
 *   "rank_pad"      1 (default) = a stack whose inner TT ranks are not multiples of 4 runs on the statically specialised
 *                   kernels with zero-padded cores when every padded hh chain has one registered (e.g. the reference's GE2E
 *                   default n_cores 2 / rank 2); 0 = runtime-shape kernels
 *   "tc_gemm"       1 (default) = the dense-route GEMMs run on the tensor cores (tcgen05.mma kind::tf32, error-compensated
 *                   3xTF32 split, TMA-staged operands, TMEM accumulators) where the shape fits; 0 = FP32 FFMA kernels
 *   "tc_red_ts"     1 (default) = the reduction GEMM takes its A operand from TMEM (tcgen05.st + the TS form of tcgen05.mma),
 *                   which leaves room for five raw TMA stages; 0 = both operands from shared memory (3 % slower, same results)
 *   "tc_rows_ts"    1 (default) = the row GEMMs (ih projection, dX) with K >= 128 take their A operand from TMEM as well;
 *                   0 = both operands from shared memory for every K (4-8 % slower at K >= 256, same results)
 *   "bwd_overlap"   1 (default) = multi-layer backward of a single-chunk plan: the weight-gradient work of layer l (dW GEMMs,
 *                   projections onto the cores, partial folds) runs on an internal second stream under the BPTT kernel of
 *                   layer l - 1, planned for the SMs that kernel leaves idle; the second stream is forked from and joined back
 *                   into the caller's stream inside ttrnn_rnn_backward (capturable).  Costs a second set of the per-layer
 *                   backward scratch buffers.  0 = everything on the caller's stream
 *   "merge_cores"   d3 r8 LSTM chains: run static kernels with TT cores 0 and 1 contracted into one core while staging
 *                   (same parameters and gradients, one chain stage fewer).  1 (default) = the dX-only BPTT kernels only:
 *                   forward results stay bit-identical to 0, gradients differ by rounding; 2 = the forward kernels as well
 *                   (faster, but h_t is rounded differently); 0 = the three-core chain.  Stamped into the workspace plan.
 * returns 0 if the key is known. */
int ttrnn_set_option(const char *key, int64_t value);

#ifdef __cplusplus
}
#endif
#endif /* TTRNN_B200_H */
