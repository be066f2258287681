/* nint.h -- C ABI of the B200-native Smart-NINT ConvLSTM hot path (libnint.so, sm_100a).
 *
 * The reference (smhassanerfani/nasa-niswan) has no FFI layer: its boundary for this path is the
 * Python class surface of model.py.  Each entry point below names the reference code it replaces
 * (file:line into the upstream repository).  Plain pointers and sizes only; every pointer is a
 * DEVICE pointer unless it says "host"; `stream` is a cudaStream_t passed as void*.
 * All functions return 0 on success and a non-zero code on failure; nint_last_error() returns a
 * thread-local description.  There is no CPU fallback: without a CUDA device every compute call
 * fails.
 *
 * Tensors crossing the boundary keep the reference's layouts:
 *   x      [B,T,C,H,W] fp32            (model.py:253-255)
 *   h, c   [B,Hc,H,W]  fp32            (model.py:216-217, 258-262)
 *   weight [4*Hc, C+Hc, k, k] fp32, bias [4*Hc]     (model.py:207-211; gate order i,f,g,o model.py:221)
 *   head   weight [1,Hc_last,1,1], bias [1]         (model.py:251)
 *   pred   [B,1,H,W] fp32 ; seq [B,T,H,W] fp32      (model.py:274 ; commented variant model.py:264,272)
 */
#ifndef NINT_H_
#define NINT_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NINT_MAX_LAYERS 8
#define NINT_DTYPE_BF16 0 /* bf16 operands, fp32 accumulation and cell state */
#define NINT_DTYPE_TF32 1 /* tf32 operands (fp32 storage), fp32 accumulation */

typedef struct nint_plan nint_plan;

/* Geometry of one ConvLSTM (model.py:235-251: ConvLSTM(input_channels, hidden_channels[],
 * kernel_size[], num_layers)) plus the batch/sequence shape of the calls it will serve. */
typedef struct nint_config {
  int32_t batch, seq_len, height, width; /* B, T, H, W of x (model.py:255) */
  int32_t in_channels;                   /* C */
  int32_t num_layers;                    /* L <= NINT_MAX_LAYERS */
  int32_t hidden[NINT_MAX_LAYERS];       /* Hc_l: any size in [1, 256] (model.py:207 takes any int); run internally padded
                                            to a multiple of 16 (64 above 64) with zero weights: results unchanged */
  int32_t ksize[NINT_MAX_LAYERS];        /* odd (model.py:204: padding = k // 2) */
  int32_t dtype;                         /* NINT_DTYPE_* */
  int32_t training;                      /* 1: keep gates/c/h of every step for BPTT */
  int32_t return_sequence;               /* 1: also apply the head at every t (model.py:264,272) */
  int32_t flags;                         /* NINT_FLAG_* */
} nint_config;

/* NINT_FLAG_DETERMINISTIC: gradients are bit-reproducible run to run (utils.py:77-88 asks cuDNN for the same): split-K
 * partial sums go to per-split buffers and are reduced in a fixed order instead of fp32 atomics.
 * NINT_FLAG_INPUT_GRAD: training plans also keep what nint_backward_input / nint_cell_backward need (the reference's
 * autograd yields x.grad and the gradient w.r.t. an explicit initial state, model.py:216-231).
 * NINT_FLAG_STATE_GRAD: training plans also keep what nint_backward_bptt_state / nint_backward_initial_state need (per
 * layer an fp32 [B,H,W,hc] buffer for dL/dh_T, and the dgrad scratch of dL/dh0).
 * NINT_FLAG_TANGENT: training plans also keep what nint_forward_tangent[_bank] needs (the input tangent
 * [T,B,H,W,cx_pad] in the operand format, per layer a 2-slot dh ring [2,B,H,W,hc_pad] of the operand format and a dc
 * buffer [B,H,W,hc] fp32, and one fp32 [B,H,W,4*max hc] dump of the tangent gate GEMM).  Plans without it have the
 * same workspace and issue the same launches.
 * NINT_FLAG_SECOND_ORDER: training plans also keep what nint_backward_second_order[_bank] needs, on top of what
 * NINT_FLAG_TANGENT keeps (the flag implies it): per layer the tangent gate GEMM's fp32 dump of every step
 * [T,B,H,W,4hc] and the tangent dc of every step [T+1,B,H,W,hc] fp32 (in place of the single dump and dc buffer), the
 * pass's dgates and their tangents [2,B,H,W,4hc] in the operand format, its running dc and tangent [2,B,H,W,hc] fp32,
 * and one fp32 dgrad dump [2,B,H,W,max(cin_rows, hc)]. */
#define NINT_FLAG_DETERMINISTIC 1
#define NINT_FLAG_INPUT_GRAD 2
#define NINT_FLAG_STATE_GRAD 4
#define NINT_FLAG_TANGENT 8
#define NINT_FLAG_SECOND_ORDER 16
/* NINT_FLAG_PARAM_TANGENT: training plans also keep a parameter direction for nint_forward_tangent[_bank] (the flag
 * implies NINT_FLAG_TANGENT): per layer the direction's weight panels packed like the forward's and its q-order fp32
 * bias [4*hc], and the head's direction (dw [Hc_last], db).  Together with NINT_FLAG_SECOND_ORDER the plan also keeps
 * what the parameter terms of nint_backward_second_order[_bank] and nint_backward_second_order_params need: per layer
 * the direction's dgrad panels, the tangent dh of every step [T+1,B,H,W,hc_pad] E (slot 0 = dh0; in place of the
 * 2-slot ring) and the pass's dgates and their tangents of every step [T][2B,H,W,4hc] E (in place of one step), and
 * the head's reductions.  Plans without it have the same workspace and issue the same launches. */
#define NINT_FLAG_PARAM_TANGENT 32
#define NINT_X_FP32 0
#define NINT_X_BF16 1

int nint_version(void);
const char* nint_last_error(void);

/* ---- plan life cycle (host-side object; owns no device memory) */
int nint_plan_create(const nint_config* cfg, nint_plan** out);
void nint_plan_destroy(nint_plan* plan);
/* device workspace the caller must provide (torch allocates it): activations, saved gates/states,
 * packed weights, gradient accumulators */
size_t nint_plan_workspace_bytes(const nint_plan* plan);
/* attaches the workspace (256-byte aligned device pointer), zero-fills it and encodes the TMA
 * tensor maps */
int nint_plan_bind(nint_plan* plan, void* workspace, size_t bytes, void* stream);

/* ---- parameters: repack the fp32 OIHW masters (state_dict names layers.{l}.conv.weight/bias,
 * conv.weight/bias; utils.py:27,39) into tensor-core operand panels.  Call after every
 * optimizer step. */
int nint_plan_set_weights(nint_plan* plan, int layer, const float* weight, const float* bias, void* stream);
int nint_plan_set_head(nint_plan* plan, const float* weight, const float* bias, void* stream);

/* ---- recurrent state.  model.py:258-262 starts every forward from zeros (the default);
 * ConvLSTMCell.forward (model.py:216-217) takes an explicit (h, c).  A state set here is the initial state of every
 * later forward until nint_plan_reset_state; nint_plan_get_state reads the final state of the last forward.  On bf16
 * plans h enters the GEMM rounded to bf16 (like every h_t), on tf32 plans rounded to tf32; c stays fp32. */
int nint_plan_reset_state(nint_plan* plan, void* stream);
int nint_plan_set_state(nint_plan* plan, int layer, const float* h, const float* c, void* stream);
int nint_plan_get_state(nint_plan* plan, int layer, float* h, float* c, void* stream);

/* ---- ConvLSTM.forward (model.py:253-274): T x L fused cell steps + head.
 * pred [B,1,H,W]; seq [B,T,H,W] or NULL (requires return_sequence). */
int nint_forward(nint_plan* plan, const float* x, float* pred, float* seq, void* stream);
/* The same with x [B,T,C,H,W] given as bf16 (x_dtype = NINT_X_BF16; bf16 plans only): a host loader that stages its
 * windows in bf16 halves the host-to-device bytes of train.py:92, and the values the tensor cores see are identical
 * (the fp32 path rounds x to bf16 as it packs it). */
int nint_forward_ex(nint_plan* plan, const void* x, int x_dtype, float* pred, float* seq, void* stream);

/* ---- frame bank: the B200 form of dataset.py:551-637 (E33OMA90D_CRNN keeps the whole record in RAM and makes its
 * windows with sliding_window_view, consecutive windows sharing T-1 frames).  Here the record lives once in HBM in the
 * model's own operand layout -- bank [n_frames][H][W][c_pad] of bf16 (bf16 plans) or tf32-rounded fp32, channels-last,
 * padding lanes zero except lane `ones_lane` = 1.0 (nint_plan_input_layout) -- and a batch is B window start indices:
 * sample b reads frames win_start[b] .. win_start[b] + T - 1 straight through the TMA descriptors (no per-step copy or
 * packing pass).  win_start: device int32 [B]; it and the bank must stay valid until the backward of the step is
 * queued.  nint_pack_frames builds a bank from frames [n_frames,C,H,W] (fp32 or bf16); nint_fuse_inputs_bank builds it
 * from the raw fields (below). */
int nint_plan_input_layout(const nint_plan* plan, int* c_pad, int* ones_lane, int* elem_bytes);
int nint_pack_frames(int dtype, const void* frames, int x_dtype, long long n_frames, int channels, int height, int width,
                     int c_pad, int ones_lane, void* bank, void* stream);
int nint_forward_bank(nint_plan* plan, const void* bank, long long n_frames, const int* win_start, float* pred,
                      float* seq, void* stream);

/* ---- BPTT of the last nint_forward (replaces autograd over model.py:216-274, train.py:109).
 * dpred [B,1,H,W], dseq [B,T,H,W] or NULL.  grad_weight[l] / grad_bias[l] are host arrays of
 * device pointers with the parameters' shapes; gradients are WRITTEN (not accumulated). */
int nint_backward(nint_plan* plan, const float* dpred, const float* dseq, float* const* grad_weight,
                  float* const* grad_bias, float* grad_head_weight, float* grad_head_bias, void* stream);
/* The same in two stages, so a data-parallel caller can all-reduce one layer's gradient bucket while the next
 * layer's weight gradient is still being computed (train.py has no DDP; SURVEY.md section 8e):
 * nint_backward_bptt = head gradients + the reverse-time loop (leaves dgates of every step in the workspace),
 * nint_backward_wgrad = weight / bias gradient of ONE layer over all T steps; any layer order, each layer once. */
int nint_backward_bptt(nint_plan* plan, const float* dpred, const float* dseq, float* grad_head_weight,
                       float* grad_head_bias, void* stream);
int nint_backward_wgrad(nint_plan* plan, int layer, float* grad_weight, float* grad_bias, void* stream);
/* nint_backward_bptt with upstream gradients of the final state as well: dh_T[l], dc_T[l] [B,Hc_l,H,W] are dL/dh_T and
 * dL/dc_T of layer l (host arrays of L device pointers; either array and any entry may be NULL = zero).  dpred and dseq
 * may both be NULL when a state gradient is given.  State gradients need a plan created with NINT_FLAG_STATE_GRAD. */
int nint_backward_bptt_state(nint_plan* plan, const float* dpred, const float* dseq, const float* const* dh_T,
                             const float* const* dc_T, float* grad_head_weight, float* grad_head_bias, void* stream);
/* Gradient w.r.t. the initial state of the last forward (after nint_backward_bptt[_state]; plans created with
 * NINT_FLAG_STATE_GRAD): dh0[l], dc0[l] [B,Hc_l,H,W] fp32 (host arrays of L device pointers; either array and any entry
 * may be NULL = not wanted).  dh0 = dgates_0 (*) flip(W_h), dc0 = dc_0 * f_0. */
int nint_backward_initial_state(nint_plan* plan, float* const* dh0, float* const* dc0, void* stream);
/* Gradient w.r.t. the input, dx [B,T,C,H,W] fp32 (x.grad of the reference's autograd through model.py:219-220); after
 * nint_backward_bptt, plans created with NINT_FLAG_INPUT_GRAD. */
int nint_backward_input(nint_plan* plan, float* dx, void* stream);
/* The input gradient of a frame-bank forward, added into the frames it read: after nint_backward_bptt[_state] of a plan
 * created with NINT_FLAG_INPUT_GRAD whose last forward was nint_forward_bank, dframes[win_start[b] + t] += dL/dx[b][t]
 * for every (b, t).  dframes: fp32 [n_frames][C][H][W] (NCHW, the layout of nint_fuse_inputs' output), n_frames the
 * bank's.  ACCUMULATES (several backwards add up, like .grad of a leaf).  Order: steps in increasing t, within a step
 * samples in increasing b, so an element receives its contributions in (t, b) order -- deterministic, also for
 * repeated window starts (no atomics).  Frames outside [0, n_frames) are skipped, as the forward reads them as zeros. */
int nint_backward_input_bank(nint_plan* plan, float* dframes, void* stream);

/* ---- tangent-linear model: forward-mode derivative (J v) of the last forward w.r.t. its input windows and its initial
 * state, at fixed parameters.  Per step and layer: da_t = W (*) [dx_t, dh_{t-1}] (no bias), then the cell's
 * linearisation at the gates the forward saved, dc_t = f dc_{t-1} + c_{t-1} df + g di + i dg and
 * dh_t = tanh(c_t) do + o (1 - tanh^2(c_t)) dc_t; dpred = head_w . dh_T, dseq[:, t] = head_w . dh_t (no head bias).
 * The gates are the saved operand-format values BPTT uses too; dh_t enters the next GEMM rounded to the operand format
 * like h_t.  Training plans created with NINT_FLAG_TANGENT, after nint_forward (explicit windows) and before a backward
 * (BPTT consumes the saved gates).  G, c and h of the forward stay intact: several tangents and then one backward of
 * the same forward may follow.
 * dx: [B,T,C,H,W] fp32 or bf16 (dx_dtype = NINT_X_*; bf16 on bf16 plans only), or NULL = zero input tangent.
 * dh0[l], dc0[l]: tangent of layer l's initial state [B,Hc_l,H,W] fp32 (host arrays of L device pointers; either array
 * and any entry may be NULL = zero).  Outputs: dpred [B,1,H,W], dseq [B,T,H,W] (return_sequence plans), dh_T[l], dc_T[l]
 * [B,Hc_l,H,W] fp32 -- all WRITTEN, any may be NULL (host arrays as for dh0). */
int nint_forward_tangent(nint_plan* plan, const void* dx, int dx_dtype, const float* const* dh0, const float* const* dc0,
                         float* dpred, float* dseq, float* const* dh_T, float* const* dc_T, void* stream);
/* The same after nint_forward_bank: dbank [n_frames][H][W][c_pad] holds the tangent frames in the bank's layout with
 * the constant-1 lane 0 (nint_pack_frames / nint_fuse_inputs_bank with ones_lane = -1), n_frames the bank's, and the
 * windows are cut at the forward's win_start. */
int nint_forward_tangent_bank(nint_plan* plan, const void* dbank, long long n_frames, const float* const* dh0,
                              const float* const* dc0, float* dpred, float* dseq, float* const* dh_T,
                              float* const* dc_T, void* stream);

/* ---- parameter-space tangent: the direction dtheta = (dW_l, db_l per layer, dw_head, db_head) that later
 * nint_forward_tangent[_bank] calls include next to (dx, dh0, dc0), giving J (dx, dh0, dc0, dtheta).  Per step and layer
 * the tangent gate GEMM gains dW (*) [x_t, h_{t-1}] + db over the forward's own operands (one more GEMM launch, added
 * into the tangent GEMM's fp32 dump), and the head gains dw_head . h_t + db_head.  Shapes as nint_plan_set_weights /
 * nint_plan_set_head; dbias NULL = zero.  A layer or head without a direction set
 * has zero direction and costs nothing; nint_plan_clear_param_tangent clears them all (the tangent pass then issues
 * exactly the launches of a plan without the flag).  Training plans created with NINT_FLAG_PARAM_TANGENT.  Setting or
 * clearing a direction after a tangent pass makes a following nint_backward_second_order[_bank] fail until the tangent
 * pass is run again.  On plans that also have NINT_FLAG_SECOND_ORDER the second-order pass takes the direction's terms:
 * deta_t gains dW_h^T (*) a_{t+1} + dW_x(above)^T (*) a_t (one EPI_RAW_ACC dgrad over the primal dgates), the top
 * layer's u dw_head, H v w.r.t. x gains dW_x^T (*) a_t and w.r.t. h0 dW_h^T (*) a_0. */
int nint_plan_set_weight_tangent(nint_plan* plan, int layer, const float* dweight, const float* dbias, void* stream);
int nint_plan_set_head_tangent(nint_plan* plan, const float* dweight, const float* dbias, void* stream);
int nint_plan_clear_param_tangent(nint_plan* plan, void* stream);
/* Parameter outputs of the last nint_backward_second_order[_bank] on a plan created with NINT_FLAG_SECOND_ORDER |
 * NINT_FLAG_PARAM_TANGENT, for the joint direction (dx, dh0, dc0, dtheta) of the tangent pass it followed:
 *   grad_W_l = sum_t wgrad(a_t, comb_t), grad_b_l = sum_t a_t; (H v)_W_l = sum_t wgrad(da_t, comb_t) + wgrad(a_t, dcomb_t),
 *   (H v)_b_l = sum_t da_t; head: grad w = sum u h, grad b = sum u, (H v)_w = sum du h + u dh, (H v)_b = sum du
 * (a, da = the pass's dgates and their tangents, comb_t = [x_t, h_{t-1}], dcomb_t its tangent; sums over every t with a
 * head seed).  The second-order pass reduces the head terms while it holds u and du, so this call takes no seeds.
 * Host arrays of L device pointers with the parameters' shapes (arrays and entries may be NULL = not wanted; a layer's
 * bias is written with its weight), head outputs [Hc_last] / [1]; all WRITTEN.  Refused before a second-order pass of
 * the current forward, tangent pass and direction.  Deterministic plans give bit-reproducible outputs. */
int nint_backward_second_order_params(nint_plan* plan, float* const* grad_weight, float* const* grad_bias,
                                      float* const* hvp_weight, float* const* hvp_bias, float* grad_head_weight,
                                      float* grad_head_bias, float* hvp_head_weight, float* hvp_head_bias, void* stream);

/* ---- second-order adjoint: the Hessian-vector product H v = d/de grad_z L(z + e v) of a loss L of the last forward's
 * outputs w.r.t. its input windows and initial state z, at fixed parameters, as forward-over-reverse.  One reverse pass
 * carries the adjoint (eta = dL/dh_t, kappa = dL/dc_t, da_t = dL/dgates_t) and its tangent in the direction of the
 * last nint_forward_tangent[_bank] together: per step (descending) and layer (top first), eta and its tangent are one
 * dgrad of da_{t+1} and its tangent (+ the layer above's x part at t, + the head term u w_head / du w_head), then the
 * cell's adjoint and its linearisation at the saved gates and tangents (DESIGN.md section 10, f8).
 * u = dL/dpred: dpred [B,1,H,W] or dseq [B,T,H,W] (return_sequence plans; one of the two); du = its tangent
 * d2L/dpred2 . dpred_tangent: ddpred / ddseq likewise (NULL = zero).  Outputs, any may be NULL, all WRITTEN: dx (the
 * gradient) and ddx (H v) w.r.t. x [B,T,C,H,W] fp32; dh0[l], dc0[l], ddh0[l], ddc0[l] [B,Hc_l,H,W] fp32 w.r.t. the initial
 * state (host arrays of L device pointers; arrays and entries may be NULL).
 * Training plans created with NINT_FLAG_SECOND_ORDER, after nint_forward and nint_forward_tangent of that forward and
 * before a backward.  The pass writes only its own buffers: more (tangent, second-order) pairs and then one backward of
 * the same forward may follow. */
int nint_backward_second_order(nint_plan* plan, const float* dpred, const float* dseq, const float* ddpred,
                               const float* ddseq, float* dx, float* ddx, float* const* dh0, float* const* dc0,
                               float* const* ddh0, float* const* ddc0, void* stream);
/* The same after nint_forward_bank / nint_forward_tangent_bank: the gradient and H v w.r.t. the frames are ADDED into
 * dframes / ddframes fp32 [n_frames][C][H][W] (either may be NULL) by the kernel nint_backward_input_bank uses: steps in
 * DEcreasing t (the pass runs backwards in time), within a step samples in increasing b -- deterministic, no atomics. */
int nint_backward_second_order_bank(nint_plan* plan, const float* dpred, const float* dseq, const float* ddpred,
                                    const float* ddseq, float* dframes, float* ddframes, float* const* dh0,
                                    float* const* dc0, float* const* ddh0, float* const* ddc0, void* stream);

/* ---- ConvLSTMCell as a differentiable unit (model.py:216-231): one step from an explicit state, and its backward.
 * Plans with seq_len = 1, num_layers = 1, training = 1, NINT_FLAG_INPUT_GRAD.  nint_cell_forward = set_state + one
 * fused step + get_state; nint_cell_backward takes dL/dh', dL/dc' [B,Hc,H,W] (either may be NULL = zero) and writes
 * dx [B,C,H,W], dh, dc [B,Hc,H,W], grad_weight, grad_bias (any output may be NULL). */
int nint_cell_forward(nint_plan* plan, const float* x, const float* h, const float* c, float* h_out, float* c_out,
                      void* stream);
int nint_cell_backward(nint_plan* plan, const float* dh_out, const float* dc_out, float* dx, float* dh, float* dc,
                       float* grad_weight, float* grad_bias, void* stream);

/* ---- preprocessing fusion (north-star item 4; SURVEY.md section 8f rank 2).  Stacks the first `levels` model
 * levels of a 3-D forcing levels3d [frames,levels,H,W] with the 2-D emission field emis2d [frames,H,W] as the last
 * channel (dataset.py:526), z-scores every channel with mean/std [levels+1] (dataset.py:520-529), appends the
 * n_static already z-scored static attribute fields statics [n_static,H,W] to every frame (dataset.py:100-122,
 * 532-533; NULL / 0 for none) and adds the geophysical halo -- cyclic in longitude, reflected in latitude
 * (dataset.py:67-98, 535-536) -- giving out [frames,levels+1+n_static,padded_height,padded_width] fp32, the
 * model's input layout.  mode 0: true reflect
 * (dataset.py:38-53); mode 1: bug-compatible with the shipped RNN dataset (np.fliplr flips channels, dataset.py:96).
 * Same error conditions as dataset.py:80,98.  PARITY UNPINNED upstream for levels > 1 (no shipped code). */
int nint_fuse_inputs(const float* levels3d, const float* emis2d, const float* mean, const float* std,
                     const float* statics, int n_static, long long frames, int levels, int height, int width,
                     int padded_height, int padded_width, int mode, float* out, void* stream);
/* The same fusion written straight into the frame-bank layout (dtype = NINT_DTYPE_*): bank
 * [frames][padded_height][padded_width][c_pad], no fp32 NCHW intermediate, no second packing pass. */
int nint_fuse_inputs_bank(const float* levels3d, const float* emis2d, const float* mean, const float* std,
                          const float* statics, int n_static, long long frames, int levels, int height, int width,
                          int padded_height, int padded_width, int mode, int dtype, int c_pad, int ones_lane,
                          void* bank, void* stream);
/* Adjoint of nint_fuse_inputs for one set of shapes and one mode: dframes [frames][levels+1+n_static][Hp][Wp] (dL/d of
 * its output) -> d_levels3d [frames][levels][H][W], d_emis2d [frames][H][W] and d_statics [n_static][H][W] (summed over
 * every frame).  Outputs are WRITTEN, not accumulated; any may be NULL (not wanted).  Every source element sums its
 * halo preimages (interior position, cyclic longitude copies, reflected -- or in mode 1 channel-reversed -- latitude
 * halo rows) in fp32 in increasing padded row, then padded column (statics: over the frames in order, then rows, then
 * columns), and the z-scored channels divide that sum by std[c] (IEEE), as autograd of (v - mean) / std does.
 * Deterministic, no atomics.  Same error conditions as nint_fuse_inputs. */
int nint_fuse_inputs_adjoint(const float* dframes, const float* std, long long frames, int levels, int n_static,
                             int height, int width, int padded_height, int padded_width, int mode, float* d_levels3d,
                             float* d_emis2d, float* d_statics, void* stream);

/* ---- the rest of the training step (train.py:101-110), SURVEY.md section 8f rank 1.
 * nint_loss_mse_l1: loss = MSELoss(y, p) + L1Loss(y, p) (train.py:74-75,105) with p = pred[:, 0, y0:y1, x0:x1]
 * (train.py:102 crop; pass 0, H, 0, W for none); pred [B,1,H,W], y [B, y1-y0, x1-x0]; writes the scalar loss, and
 * d loss / d pred into dpred [B,1,H,W] (zero outside the crop; NULL = value only).  stats: 5 floats of device
 * scratch, left holding {sum (p-y)^2, sum |p-y|, sum y, sum y^2, -} (enough for an on-device R^2, train.py:114).
 * nint_adam_step: torch.optim.Adam (train.py:71; no weight decay / amsgrad) over one flat fp32 buffer; `step` counts
 * from 1; grads are multiplied by grad_scale first (1 / world_size after a sum all-reduce). */
int nint_loss_mse_l1(const float* pred, const float* y, int batch, int height, int width, int crop_y0, int crop_y1,
                     int crop_x0, int crop_x1, float* dpred, float* loss, float* stats, void* stream);
int nint_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                   float beta1, float beta2, float eps, int step, float grad_scale, void* stream);
/* nint_loss_mse_l1 with the targets in a bank y [n_frames, y1-y0, x1-x0]: sample b's target is frame
 * win_start[b] + y_offset (dataset.py:600-601: y[seq_len - 1:] pairs window i with frame i + T - 1); an index outside
 * [0, n_frames) reads as a zero target (the input side reads zeros through TMA) instead of faulting. */
int nint_loss_mse_l1_bank(const float* pred, const float* ybank, long long n_frames, const int* win_start, int y_offset, int batch,
                          int height, int width, int crop_y0, int crop_y1, int crop_x0, int crop_x1, float* dpred,
                          float* loss, float* stats, void* stream);
/* nint_adam_step with the step count and learning rate in DEVICE memory: state = 4 floats {step, lr, -, -}; the call
 * increments state[0] itself.  Nothing in the launch depends on host values that change between steps, so a CUDA graph
 * of the whole training step can be replayed. */
int nint_adam_step_dev(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float* state,
                       float beta1, float beta2, float eps, float grad_scale, void* stream);

/* ---- data-parallel step tail over NVLink peer memory (SURVEY.md section 8e; the reference has no multi-GPU code).
 * Replaces ncclAllReduce + nint_adam_step_dev by ONE kernel: cross-rank barrier, sum of every rank's gradients read
 * straight from the peers' memory in rank order (bit-identical on all ranks), Adam on this rank's parameters.
 * peer_buffers: HOST array of `world` device pointers -- the same symmetric allocation as mapped for each rank
 * ([rank] is this GPU's own).  Layout of the allocation: two gradient slots of n fp32 used alternately (the caller
 * writes step s's gradients to the slot at slot_offset_bytes, alternating by step parity) and a zero-initialised flag
 * block of 32 uint32 at flags_offset_bytes.  seq: step number, increasing from 1 on every rank.  state as in
 * nint_adam_step_dev.  Every rank must make the call for a step; a rank that never arrives traps the waiters after
 * ~20 s instead of hanging them. */
int nint_dp_allreduce_adam(const void* const* peer_buffers, long long slot_offset_bytes, long long flags_offset_bytes,
                           int rank, int world, unsigned seq, float* params, float* exp_avg, float* exp_avg_sq,
                           long long n, float* state, float beta1, float beta2, float eps, float grad_scale, void* stream);

/* ---- measurement.  Kernel classes: 0 = fused gate-conv forward, 1 = dgrad + gate backward,
 * 2 = wgrad, 3 = everything else (layout packing, head, gradient unpacking); -1 = all.
 * nint_launch_count: kernels launched by this library in the calling process so far.
 * nint_plan_profile(plan, 1) brackets every later launch of the plan with CUDA events on the
 * launching stream; nint_plan_profile_read waits for them and returns, per class, the summed
 * device time in ms and the launch count since the last read (arrays of 4). */
long long nint_launch_count(int kernel_class);
int nint_plan_profile(nint_plan* plan, int enable);
int nint_plan_profile_read(nint_plan* plan, double* ms, long long* count);

/* ---- test hook: raw gate pre-activations of layer 0 at t = 0 without bias,
 * out [B,H,W,4*Hc] fp32 in kernel column order (see nint_gate_column). */
int nint_debug_raw_gates(nint_plan* plan, const float* x, float* out, void* stream);
/* debug timeline: with NINT_DEBUG_FLAGS & 8, CTA 0 of every conv launch records clock64() stamps per warp role
 * (8 roles x 1024 stamps; later launches overwrite earlier ones).  Copies them to `host`, optionally clears. */
int nint_debug_read_trace(long long* host, int n, int clear);
/* Post-mortem of a time-fused conv launch's step hand-off (a wait that lasts ~2 s traps instead of hanging the GPU, and
 * a trap destroys the context): the first call arms a host-mapped record, later calls -- also after a failed launch --
 * return {code (0 = none, 3 = hand-off timed out), block, thread, (step << 32) | image, counter value}. */
int nint_debug_fail_record(unsigned long long* out5);
/* reference gate channel n = gate*Hc + c for kernel column q of a layer with Hc hidden channels */
int nint_gate_column(int q, int hidden);
/* pixel tile chosen for a grid (host-only helper, no device needed) */
int nint_pick_tile(int height, int width, int* tile_w, int* tile_h);

#ifdef __cplusplus
}
#endif
#endif /* NINT_H_ */
