// Internal host/device interface between the C-ABI layer (nint_api.cu) and the kernels.
//
// Layout conventions shared by every kernel (DESIGN.md "Data layout in HBM"):
//   * activations are channels-last, [slot][B][H][W][C_pad] of E (E = bf16, or fp32 holding
//     tf32-rounded values), C_pad a multiple of 32 channels; the conv kernels walk K in 64-byte
//     chunks (32 bf16 / 16 tf32 elements), wgrad in 32-channel panels;
//   * a pixel tile is tile_w x tile_h <= 128 pixels of one image, row = ty * tile_w + tx;
//   * the 4*hc gate channels of a layer are stored in "q-order": hidden channel c = 16*grp + c16,
//       q = grp * 64 + gate * 16 + c16  <->  reference channel n = gate * hc + c
//     (gate order i,f,g,o: model.py:221): the four gates of a 16-channel group are 64 contiguous columns,
//     i.e. one 128-byte (bf16) TMA box row per pixel for the epilogue, and any multiple of 16 hidden
//     channels is a contiguous N slice (n-block) of the forward GEMM.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

// Experiment knobs (ConvGemmParams / WgradParams::debug_flags: skip the epilogue's memory work, issue no MMAs, issue them
// twice, timeline stamps, ...) are compiled in only with -DNINT_KNOBS=1 (`python -m nasa_niswan_b200.build --knobs` ->
// libnint_knobs.so, selected with NINT_LIB).  In the product build the flags read as 0 at compile time: a run-time
// branch inside the single-thread MMA loops costs the default path dearly (DESIGN.md section 6: -12 % for one).
#ifndef NINT_KNOBS
#define NINT_KNOBS 0
#endif
#define NINT_DBG(p) (NINT_KNOBS ? (p).debug_flags : 0)

namespace nint {

// EPI_RAW_ACC: EPI_RAW that adds the accumulators into the dump instead of overwriting it (a second GEMM summed into the
// first one's dump: the parameter tangent's dW (*) comb_t on top of W (*) dcomb_t)
enum : int { EPI_FWD = 0, EPI_BWD = 1, EPI_RAW = 2, EPI_RAW_ACC = 3 };
__host__ __device__ constexpr bool epi_is_raw(int epi) { return epi == EPI_RAW || epi == EPI_RAW_ACC; }

// One K-segment of an implicit-GEMM convolution: an activation tensor read through a 5-D TMA
// map (box = one chunk x tile_w x tile_h pixels; out-of-image pixels are zero-filled by TMA =
// the conv's zero padding, model.py:204-211) and its packed weights read through a 3-D map
// [(nb*nchunks + chunk)*taps + tap][n_tile rows][chunk elements] (box = this CTA's rows of one weight stage).
struct alignas(64) ConvSegment {
  CUtensorMap tmap_act;
  CUtensorMap tmap_w;
  int slot;
  int ksize;
  int nchunks;
  int wsel;   // host only: which packed weight tensor of the layer (nint_api.cu get_w_map)
  int ts;     // taps per weight stage of THIS segment (divides ksize^2; conv_halo_plan); taps_per_stage is the largest
  // frame-bank input (nint_forward_bank): tmap_act is [n_frames][H][W][C] and image b of the launch reads frame
  // win_start[b] + slot (slot = time step); null = the plan's own [slot][B][H][W][C] tensor
  const int* win_start;
  int bank_frames;
};

struct alignas(64) ConvGemmParams {
  ConvSegment seg[2];
  int nseg;
  int B, H, W;   // B = images of THIS launch: images [b0, b0 + B) of the plan's batch (sub-batch-major schedules)
  int b0;
  int tile_w, tile_h;
  int tiles_x, tiles_y;
  int n_tile;    // UMMA N (accumulator columns per tile)
  int n_blocks;  // N slices of the gate columns (forward: 4*hc / n_tile); a cluster owns one slice
  int num_stages;
  // halo variant (nint_conv_halo.cu): activation buffers, cluster size, descriptor base-offset policy
  int na_bufs, a_buf_bytes, cluster, taps_per_stage;
  int group, a_halo_bytes;  // tiles per group (side-by-side accumulators), bytes of one halo chunk
  int acc_cols, n_acc;      // TMEM columns of one accumulator buffer (group * n_tile), number of buffers (2 or 4)
  int plan_g, plan_ns;      // experiment knobs for conv_halo_plan: cap on tiles per group / epilogue stages (0 = auto)
  int w_resident;           // 1: num_stages covers a tile's whole K walk; weights are loaded once per CTA
  int debug_flags;          // experiments: 1 = epilogue does no memory ops / math, 2 = no MMA issue
  int pdl;                  // 1: programmatic dependent launch (prologue overlaps the previous launch's tail)
  // ---- TMA-staged epilogue I/O (nint_epilogue.cuh): 5-D maps (channel, x, y, image, slot) of the layer's
  // c history (fp32), h history (E), saved gates (E, q-order) and running dc (fp32); slot < 0 = absent
  CUtensorMap tm_c, tm_h, tm_g, tm_dc;
  int slot_c_in, slot_c_out, slot_h_out, slot_g;   // FWD: c_{t-1}, c_t, h_t, gates_t;  BWD: slot_g = gates_t / dgates_t
  int slot_c_prev, has_dc_in;                      // BWD: c_{t-1}, dc_t present (c_t is recomputed from c_{t-1} and the gates)
  int e_stages, e_stage_bytes, e_off_c, e_off_c2, e_off_dc, e_off_h;
  int c_ring;               // forward: slots of the separate c_{t-1} -> c_t ring (0 for the backward kernel)
  uint32_t idesc;
  int hc, hc_pad;  // hidden channels of this layer / padded channel count of its h tensor
  int hcb;         // hidden channels per n-block (n_tile / 4)
  // ---- EPI_FWD: LSTM cell update (model.py:221-229)
  const float* bias_q;  // [4*hc], q-order; null = the bias is folded into the GEMM (layer 0 with the constant-1 input lane)
  // ---- EPI_BWD: gate backward (SURVEY 8 a10); accumulator = dh (absent when nseg == 0); dgates overwrite
  // the saved gates in place
  const float* head_dpred;  // optional [B,H,W] (+ stride): dh += head_dpred * head_w[c]
  long long head_dpred_bstride;  // elements between images of head_dpred
  const float* head_w;      // [hc]
  // tf32 mode: dgates are rounded to tf32 (the MMA operand format) when stored; the bias gradient -- a plain sum of
  // dgates that can nearly cancel -- also gets the sum of the rounding residuals: [gridDim.x][4 quadrants][4*hc] fp32,
  // every (CTA, pixel quadrant) adds into its own slots (deterministic), reduced by unpack_wgrad_kernel
  float* db_resid;
  const float* dh_ext;      // optional [B,H,W,hc] fp32 channels-last: dh += dh_ext (standalone cell backward, model.py:216-231)
  // ---- EPI_RAW: dump fp32 accumulators [B,H,W,n_blocks*n_tile] (debug / generic conv); EPI_RAW_ACC adds into it
  float* raw_out;
  // ---- time-fused launch: n_steps > 1 consecutive time steps of one layer run as ONE persistent launch.  The tile walk
  // covers n_steps x tiles (step-major); in step s every slot field advances by its `d_*` (forward +1, BPTT -1; fields in
  // ring_bits live in a 2-slot ring).  Step s of image b may only start once every tile of image b of step s-1 has been
  // stored: step_done[(s-1) * B + b] counts the storer warps that have finished a tile (zeroed before the launch) and
  // reaches step_target.  Tile-level dependencies instead of a grid-wide drain between launches: the pipeline of a CTA
  // never empties across steps.
  int n_steps;
  int d_seg[2], d_c_in, d_c_out, d_h_out, d_g, d_c_prev;
  int ring_bits;            // bit 0/1: seg[0/1].slot, 2: slot_c_in, 3: slot_c_out, 4: slot_h_out (slot & 1 after the advance)
  int c_prev_none_step;     // BWD: step whose c_{t-1} is the zero initial state (-1: none)
  long long head_dpred_sstride;   // elements between consecutive steps of head_dpred
  unsigned* step_done;
  unsigned step_target;
};

// 8x16 pixel tiles, activation chunk + halo loaded once and re-read by every tap (nint_conv_halo.cu).
// conv_halo_plan fills the shared-memory plan (epilogue stages, item group, halo buffers, weight stages)
// from nseg, seg[].ksize, n_tile, hc, cluster, slot_*; non-zero = does not fit.
int conv_halo_plan(int epi, int dtype, ConvGemmParams& p);
int conv_halo_smem_bytes(const ConvGemmParams& p);
cudaError_t launch_conv_halo(int epi, int dtype, const ConvGemmParams& p, int num_sms, cudaStream_t stream);
// debug timeline (debug_flags & 8): 8 roles x 1024 clock64 stamps written by CTA 0 of the last traced launch
cudaError_t read_trace(long long* host, int n);
cudaError_t fail_record(unsigned long long* out5);
cudaError_t clear_trace();

// ---- wgrad (nint_wgrad.cu):  dW[tap][q][col] += sum_pixels dgates[pix][q] * comb[pix + tap][col]
constexpr int kMaxWgradGroups = 32;
struct alignas(64) WgradParams {
  CUtensorMap tmap_dg;    // dgates [T][B][H][W][4*hc]        (A, MN-major, M = q)
  CUtensorMap tmap_b[2];  // x-part tensor, h-part tensor      (B, MN-major, N = channel)
  int slot_b0[2];         // slot of step 0 for each b tensor
  int nchunks_b[2];       // 32-channel panels per b segment
  int T, B, H, W;
  int tile_w, tile_h, tiles_x, tiles_y;
  int ksize;
  int m_blocks;           // ceil(4*hc / 128)
  int n_groups;
  int group_tap0[kMaxWgradGroups + 1];  // taps [group_tap0[g], group_tap0[g+1]) belong to group g
  int bias_group;         // tap group whose CTAs also accumulate the bias gradient with a ones-panel MMA (-1: none --
                          // the x tensor carries a constant 1.0 in a padding channel and db falls out of the centre tap)
  int group_splits[kMaxWgradGroups];    // split-K factor over pixel tiles, per tap group (in proportion to its MMA cost)
  int group_unit0[kMaxWgradGroups + 1]; // first CTA (cluster, for the pair kernel) of each group; [n_groups] = grid units
  int ncols;              // row pitch of dw_acc = all padded input + hidden channels of the layer
  int acc_cols;           // accumulator columns per tap of THIS launch = (sum nchunks_b) * 32 (one column block)
  int col0;               // first dw_acc column of the block
  int real_cols;          // columns of the block that exist in dw_acc (<= acc_cols; the rest is MMA padding)
  int chan0[2];           // first channel of the block inside the x-part / h-part tensor
  int a_bufs, b_stages;
  int halo;               // 1: 8x16 tiles, B panels hold the tile + k//2 halo and every tap re-reads them in place
  int b_panel_bytes;      // bytes between consecutive B panels of a stage
  int debug_flags;        // experiments: 2 = no MMA issue, 4 = issue every MMA twice
  int pair;               // 1: CTA-pair kernel (bf16, 4*hc % 256 == 0): m_blocks counts 256-q blocks, tmap_dg has 64-q
                          // boxes (SWIZZLE_128B) and tmap_b b_pw-channel halo boxes (SWIZZLE_32B / 64B / 128B)
  int b_pw;               // pair kernel: channels per B panel (16 / 32 / 64)
  uint32_t idesc, idesc_bias;
  int hc4;                // 4*hc
  const int* win_start;   // frame-bank input: tmap_b[0] is [n_frames][H][W][C]; image b at step t reads frame win_start[b] + t
  float* dw_part;         // deterministic mode: per-split partial sums [max splits][taps][4*hc][ncols] (plain stores) or null
  float* db_part;         // deterministic mode: [max splits][4*hc] or null
  float* dw_acc;          // [taps][4*hc][ncols] fp32, atomically accumulated (pre-zeroed)
  float* db_acc;          // [4*hc] fp32 (q-order) or null
};
int wgrad_b_panel_bytes(int dtype, int halo, int ksize);
int wgrad_smem_bytes(int dtype, int bpanels, int a_bufs, int b_stages, int b_panel_bytes);
void wgrad_pick_buffers(int dtype, int bpanels, int b_panel_bytes, int* a_bufs, int* b_stages);
int wgrad_pair_supported(int dtype, int hc4, int cx_pad, int ncols, int ksize);
int wgrad_pair_panel_width(int cx_pad, int ncols);          // channels per B panel of the pair kernel: 16 / 32 / 64
int wgrad_pair_b_stages(int cx_pad, int ncols, int ksize);  // B stages that fit (0: pair kernel not possible)
int wgrad_pair_b_stages_tf32(int n_mma, int ksize);         // same for the tf32 variant (32-channel fp32 panels)
cudaError_t launch_wgrad(int dtype, const WgradParams& p, cudaStream_t stream);

// ---- pointwise / layout kernels (nint_pointwise.cu)
// x [B,T,C,H,W] fp32 or bf16 (model.py:255) -> X [T][B][H][W][c_pad] E (pad channels zero)
// ones_lane >= C: that padding channel is set to 1.0 (bias gradient through the wgrad GEMM), -1: none
cudaError_t launch_pack_input(int dtype, const void* x, int x_bf16, void* X, int B, int T, int C, int H, int W, int c_pad,
                              int ones_lane, cudaStream_t s);
// frames [N][C][H][W] fp32 or bf16 -> frame bank [N][H][W][c_pad] E (nint_forward_bank)
cudaError_t launch_pack_frames(int dtype, const void* src, int src_bf16, void* bank, long long N, int C, int H, int W,
                               int c_pad, int ones_lane, cudaStream_t s);
// NCHW fp32 <-> NHWC E (state import / export for the cell API)
cudaError_t launch_pack_state(int dtype, const float* src_nchw, void* dst_nhwc, int B, int C, int H, int W,
                              int c_pad, cudaStream_t s);
cudaError_t launch_unpack_state(int dtype, const void* src_nhwc, float* dst_nchw, int B, int C, int H, int W,
                                int c_pad, cudaStream_t s);
cudaError_t launch_nchw_to_nhwc_f32(const float* src, float* dst, int B, int C, int H, int W, int c_pad, cudaStream_t s);
cudaError_t launch_nhwc_to_nchw_f32(const float* src, float* dst, int B, int C, int H, int W, int c_pad, cudaStream_t s);
// OIHW fp32 master weights [4*hc_real][cin + hc_real][k][k] -> packed operand panels of a layer whose hidden size is
// padded to hc >= hc_real (padding channels: zero weights, zero bias -> their h and c stay exactly zero)
cudaError_t launch_pack_weights_fwd(int dtype, const float* w, const float* bias, void* wpack_x, void* wpack_h,
                                    float* bias_q, int cin, int hc_real, int hc, int hcb, int k, int cx_pad, int hc_pad,
                                    int bias_lane, cudaStream_t s);
cudaError_t launch_pack_weights_bwd(int dtype, const float* w, void* wpack_dx, void* wpack_dh, int cin, int cin_rows,
                                    int hc_real, int hc, int k, cudaStream_t s);
// 1x1 head (model.py:251,274)
cudaError_t launch_head_fwd(int dtype, const void* h, const float* w, const float* b, float* out, long long npix_per_img,
                            int B, int hc, int hc_pad, long long out_bstride, cudaStream_t s);
// tangent of the head with a parameter direction: out = db + sum_c dh[pix][c] w[c] + h[pix][c] dw[c] (one pass over
// the primal and the tangent h; model.py:274 differentiated in (h, w, b))
cudaError_t launch_head_tangent(int dtype, const void* h, const void* dh, const float* w, const float* dw, const float* db,
                                float* out, long long npix_per_img, int B, int hc, int hc_pad, long long out_bstride,
                                cudaStream_t s);
// part: null (fp32 atomics) or head_bwd_blocks(B) * (hc + 1) floats of scratch (deterministic fixed-order sum)
int head_bwd_blocks(int B);
cudaError_t launch_head_bwd(int dtype, const void* h, const float* dpred, long long dpred_bstride, float* dw, float* db,
                            long long npix_per_img, int B, int hc, int hc_pad, float* part, cudaStream_t s);
// dw_acc [taps][4hc (q)][ncols] -> grad weight OIHW [4hc_real][cin+hc_real][k][k]; grad bias from db_acc (q), or from
// column bias_col of the centre tap of dw_acc when bias_col >= 0; nparts > 0: dw_acc / db_acc are `nparts` partial
// slices summed in order (deterministic mode)
cudaError_t launch_unpack_wgrad(const float* dw_acc, const float* db_acc, float* gw, float* gb, int cin, int hc_real,
                                int hc, int k, int ncols, int cx_pad, int bias_col, int accumulate, int nparts,
                                const float* db_resid, int resid_slots, cudaStream_t s);
// fp32 accumulator dump [B][H][W][ncols] (EPI_RAW) -> gradient tensor [B][(T)][C][H][W] fp32 (dx / dh of the cell API)
cudaError_t launch_unpack_raw(const float* raw, float* dst, int B, int C, int H, int W, int ncols, long long dst_bstride,
                              cudaStream_t s);
// the same dump of step t added into the frames the windows read: dframes[win_start[b] + t][C][H][W] += raw[b], samples
// in increasing b per element (repeated starts accumulate in that order), frames outside [0, n_frames) skipped
cudaError_t launch_accum_frames(const float* raw, float* dframes, const int* win_start, int B, int C, int H, int W,
                                int ncols, int t, long long n_frames, cudaStream_t s);

// tangent-linear cell step (nint_forward_tangent): raw = the tangent GEMM's EPI_RAW dump [npix][4*hc] (q-order, i/f/o
// columns halved like the packed forward weights), gates = the forward's activated gates of this step [npix][4*hc] E,
// c_prev / c_cur = c_{t-1} / c_t [npix][hc] fp32; dc_in = dc_{t-1}, dc_out = dc_t [npix][hc] fp32 (the same buffer:
// updated in place), dh_out [npix][hc_pad] E gets dh_t (lanes >= hc are not written)
// dbias_q: null, or the parameter tangent's q-order bias [4*hc] (i/f/o halved like bias_q) added to raw and stored back
// into it (the dump then holds the whole tangent pre-activation) -- a separate kernel (tangent_cell_bias_kernel), so the
// launch without it is unchanged
cudaError_t launch_tangent_cell(int dtype, float* raw, const void* gates, const float* c_prev, const float* c_cur,
                                const float* dc_in, float* dc_out, void* dh_out, long long npix, int hc, int hc_pad,
                                cudaStream_t s, const float* dbias_q = nullptr);

// second-order adjoint cell step (nint_backward_second_order), per (pixel, hidden channel): eta = [2][npix][hc] fp32
// dgrad dump (dL/dh_t and its tangent; NULL = 0), u / du = dL/dpred and its tangent at this step (NULL = 0; pixel
// b*HW + i at u[b*u_bstride + i]) times head_w [hc] (top layer only), gates / traw = the forward's activated gates and
// the tangent GEMM's dump of this step [npix][4hc] (traw: i/f/o halved), c_prev / c_cur and dc_prev / dc_cur = c and
// its tangent at t-1 / t [npix][hc] fp32; kappa [2][npix][hc] fp32 (dL/dc and its tangent) is updated in place,
// da_out [2][npix][4hc] E gets dL/dgates_t and its tangent in the fused backward's q-order and scaling
cudaError_t launch_soa_cell(int dtype, const float* eta, const float* u, long long u_bstride, const float* du,
                            long long du_bstride, const float* head_w, const void* gates, const float* traw,
                            const float* c_prev, const float* c_cur, const float* dc_prev, const float* dc_cur,
                            float* kappa, void* da_out, long long npix, long long HW, int hc, cudaStream_t s,
                            const float* dhead_w = nullptr);   // dhead_w: the head weight's tangent (soa_cell_dhead_kernel)

// preprocessing fusion: stack levels + emission, z-score, cyclic-longitude / reflect-latitude halo
cudaError_t launch_fuse_inputs(const float* lev, const float* emis, const float* mean, const float* stdv,
                               const float* statics, int S, float* out, long long N, int L, int H, int W, int Hp, int Wp,
                               int mode, cudaStream_t s);
// the same, written as the frame bank [N][Hp][Wp][c_pad] E (channels-last operand layout, ones lane)
cudaError_t launch_fuse_inputs_bank(int dtype, const float* lev, const float* emis, const float* mean, const float* stdv,
                                    const float* statics, int S, void* out, long long N, int L, int H, int W, int Hp, int Wp,
                                    int mode, int c_pad, int ones_lane, cudaStream_t s);
// adjoint of launch_fuse_inputs: dframes [N][L+1+S][Hp][Wp] -> d_lev [N][L][H][W], d_emis [N][H][W], d_statics [S][H][W]
// (summed over the frames); any output may be null
cudaError_t launch_fuse_inputs_adjoint(const float* dframes, const float* stdv, long long N, int L, int S, int H, int W,
                                       int Hp, int Wp, int mode, float* d_lev, float* d_emis, float* d_statics,
                                       cudaStream_t s);
// fused training loss MSE + L1 on the cropped prediction (value + gradient); stats = 5 floats of scratch;
// y_index != null: the target of sample b is image y_index[b] + y_offset of y (frame bank)
cudaError_t launch_loss_mse_l1(const float* pred, const float* y, float* dpred, float* stats, float* loss, int B, int H,
                               int W, int y0, int y1, int x0, int x1, const int* y_index, int y_offset, long long y_frames,
                               cudaStream_t s);
// Adam step over a flat fp32 parameter buffer
cudaError_t launch_adam(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                        float eps, int step, float grad_scale, cudaStream_t s);
// the same with {step, lr, bc1, sqrt(bc2)} in device memory (`state`, 4 floats): capturable in a CUDA graph
cudaError_t launch_adam_dev(float* p, const float* g, float* m, float* v, long long n, float* state, float beta1,
                            float beta2, float eps, float grad_scale, cudaStream_t s);

// fused cross-rank barrier + gradient all-reduce over NVLink peer memory + Adam (nint_dp.cu)
cudaError_t launch_dp_allreduce_adam(const void* const* peer_bases, long long slot_offset_bytes, long long flags_offset_bytes,
                                     int rank, int world, unsigned seq, float* params, float* m, float* v, long long n,
                                     float* state, float beta1, float beta2, float eps, float grad_scale, cudaStream_t s);

// q-order helper (host + device)
__host__ __device__ inline int q_to_n(int q, int hc) { return ((q >> 4) & 3) * hc + (q >> 6) * 16 + (q & 15); }

}  // namespace nint
