// C-ABI layer (include/nint.h): plan geometry, workspace carving, TMA tensor-map encoding and
// the host-side step loops of ConvLSTM.forward (model.py:253-274) and its BPTT.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "../../include/nint.h"
#include "nint_kernels.h"

namespace {

using namespace nint;
enum : int { BF16 = 0, TF32 = 1 };

thread_local char g_err[512] = "";
int fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}
#define CK(expr)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// kernel classes for the launch counter / CUDA-event profile
enum : int { K_FWD = 0, K_BWD = 1, K_WGRAD = 2, K_OTHER = 3, K_NCLS = 4 };
constexpr int kResidCtas = 160;   // upper bound on the CTAs of one conv launch (one per SM)
// tf32 rounding residuals of the bias gradient are tracked for SHORT sums only (up to 2^20 pixel-steps per bias
// element): there the rounding does not average out (tiny cases sat at 1.4e-3..2.5e-3 of the 1e-3 bar); on long sums
// (cfg 2 at B=32: 5 M pixel-steps, bias gradients at 1e-4..7e-4) the warp reductions would cost the tf32 backward
// kernel 40 % (306 -> 430 us per launch, measured) for nothing.
constexpr long long kResidMaxPixelSteps = 1LL << 20;
long long g_launches[K_NCLS] = {0, 0, 0, 0};

struct Profile {
  bool on = false;
  std::vector<cudaEvent_t> pool;
  std::vector<int> cls;  // class of pair i (events 2i, 2i+1)
  std::vector<int> weight;  // time steps the launch of pair i covers (1; n for a time-fused conv launch)
  size_t used = 0;       // pairs in flight
};

struct Layer {
  int cin, hc_real, hc, k, taps;   // cin / hc_real: the reference's channel counts (model.py:207); hc: hc_real padded to the
                                   // kernels' granularity (16; 64 above 64) with zero weights -- results are unchanged
  int cin_rows;                    // rows (N) of the dx dgrad operand: padded width of the tensor dx flows into
  int cx_pad, hc_pad, chx, chh;  // padded channels / 64-byte chunks of the x and h segments
  int hcb, n_blocks, n_tile;
  int nslots_h, nslots_c;
  // workspace pointers
  uint8_t* Hs = nullptr;   // [nslots_h][B][H][W][hc_pad] E
  float* Cs = nullptr;     // [nslots_c][B][H][W][hc]
  uint8_t* G = nullptr;    // [T][B][H][W][4hc] E   (training)
  float* dC = nullptr;     // [B][H][W][hc]         (training)
  float* dh_ext = nullptr; // [B][H][W][hc] upstream dL/dh_T (NINT_FLAG_STATE_GRAD)
  uint8_t* tH = nullptr;   // NINT_FLAG_TANGENT: [2][B][H][W][hc_pad] E ring of dh (slot t & 1 = dh_{t-1})
  float* tC = nullptr;     // NINT_FLAG_TANGENT: [B][H][W][hc] running dc; NINT_FLAG_SECOND_ORDER: [T+1] slots (slot t = dc_{t-1})
  CUtensorMap tm_tH, tm_tH_up;   // tH as this layer's recurrent segment / as the x segment of layer l+1
  // NINT_FLAG_SECOND_ORDER: the tangent gate GEMM's dump of every step [T][B][H][W][4hc] fp32; the second-order pass's
  // dgates and their tangents [2][B][H][W][4hc] E (one step: the pass reads da_{t+1} before it writes da_t), seen by
  // tm_sA as 2B images so one dgrad launch covers both; its running dc (kappa) and tangent [2][B][H][W][hc] fp32
  float* tR = nullptr;
  uint8_t* sA = nullptr;
  float* sK = nullptr;
  CUtensorMap tm_sA;
  uint8_t *wx = nullptr, *wh = nullptr, *wdx = nullptr, *wdh = nullptr;
  float *bias_q = nullptr, *dw_acc = nullptr, *db_acc = nullptr;
  // NINT_FLAG_PARAM_TANGENT: the parameter direction dW packed like wx / wh (same panels, i/f/o halved) and its bias in
  // q-order; dw_set: a direction is set for this layer (else dW = 0 and the tangent pass runs no dW GEMM); dbias_add:
  // the tangent cell adds tbias_q (the bias is not folded into the dW GEMM through the constant-1 lane)
  uint8_t *twx = nullptr, *twh = nullptr;
  float* tbias_q = nullptr;
  bool dw_set = false, dbias_add = false;
  // NINT_FLAG_PARAM_TANGENT + NINT_FLAG_SECOND_ORDER: dW's dgrad panels (laid out as wdx / wdh) for the second-order
  // pass's dW^T terms, and the wgrad views of the parameter outputs: the pass's (a, da) history as dgates operand
  // (primal view / tangent view: images [0, B) / [B, 2B) of every [2B] step slot) and the dh history as the h part /
  // as the x part of layer l+1 (32-channel boxes, CTA-pair boxes)
  uint8_t *twdx = nullptr, *twdh = nullptr;
  CUtensorMap tmw_sA[2], tmp_sA[2], tmw_tH, tmw_tH_up, tmp_tH, tmp_tH_up;
  float* db_resid = nullptr;   // tf32 training plans: [kResidCtas][4][4hc] sums of the dgates rounding residuals (nint_kernels.h)
  size_t dw_acc_bytes = 0;   // one slice [taps][4hc][ncols]; deterministic mode keeps det_splits slices
  int det_splits = 0;
  int ncols = 0;
  CUtensorMap tm_H, tm_G;
  // weight maps depend on the launch's shared-memory plan (taps per stage): encoded on first use, cached
  struct WMap { int ts = 0, rows = 0, n_tile = 0; CUtensorMap map; };
  std::vector<WMap> wmaps[8];   // 0: wx, 1: wh, 2: wdx, 3: wdh, 4: twx, 5: twh, 6: twdx, 7: twdh
  CUtensorMap tm_H_up;       // Hs[l] read as the x segment of layer l+1 (halo of k_{l+1})
  CUtensorMap tmw_H, tmw_G;  // wgrad views (32-channel boxes; differ from tm_* in tf32 mode only)
  CUtensorMap tmw_H_up;      // Hs[l] as the x part of layer l+1's wgrad (halo of k_{l+1})
  CUtensorMap tmp_G, tmp_H, tmp_H_up;        // CTA-pair wgrad views: 64-q dgates boxes (SWIZZLE_128B), 16-channel halo boxes (SWIZZLE_32B)
  // wgrad runs one launch per column block of dW (columns = padded input channels, then hidden channels): a block
  // is what one CTA (pair) can hold as operand panels in shared memory and as an MMA N (<= 256)
  struct WgBlock {
    int col0 = 0, cols = 0;      // dw_acc columns [col0, col0 + cols)
    int n_mma = 0;               // MMA N / accumulator columns per tap (>= cols: the tf32 pair kernel pads to whole panels)
    int nch_x = 0, nch_h = 0;    // 32-channel panels taken from the x-part / h-part tensor
    int chan0_x = 0, chan0_h = 0;
    bool pair = false;
    int pw = 16, a_bufs = 0, b_stages = 0;
  };
  std::vector<WgBlock> wg_blocks;
  CUtensorMap tme_C, tme_H, tme_G, tme_dC;  // epilogue I/O boxes (16 | 64 channels x 8 x 16 pixels; nint_epilogue.cuh)
  bool weights_set = false;
  bool bias_folded = false;   // the forward bias rides in the GEMM through the input's constant-1 lane
  // launch parameters that do not change from step to step (shared-memory plan, tensor maps, descriptors): built on
  // first use, then only the slot indices are patched per launch.  fwd[have_state][bank], bwd[has dgates_{t+1} segment]
  struct CachedConv { bool valid = false; ConvGemmParams g; };
  CachedConv fwd_cache[2][2], bwd_cache[2];
};

}  // namespace

struct nint_plan {
  nint_config cfg;
  int L, B, T, H, W, dtype, esize, ce;
  int tile_w, tile_h, tiles_x, tiles_y;
  int num_sms = 148;
  Layer layer[NINT_MAX_LAYERS];
  size_t ws_bytes = 0;
  uint8_t* ws = nullptr;
  uint8_t* X = nullptr;  // [T][B][H][W][cx_pad0] E
  CUtensorMap tm_X, tmw_X, tmp_X;
  // frame-bank input (nint_forward_bank): maps over the caller's [n_frames][H][W][cx_pad0] tensor, re-encoded when the
  // bank pointer or length changes
  bool x_bank = false;
  const void* bank_ptr = nullptr;
  long long bank_frames = 0;
  const int* win_start = nullptr;
  CUtensorMap tmb_X, tmbw_X, tmbp_X;
  float *head_w = nullptr, *head_b = nullptr;
  float* raw = nullptr;      // NINT_FLAG_INPUT_GRAD / _STATE_GRAD: [B][H][W][max(cx_pad0, hc0, hc_l)] fp32 dgrad dump
  float* dh_ext = nullptr;   // NINT_FLAG_INPUT_GRAD, cell plans: upstream dL/dh' as [B][H][W][hc] fp32
  float* head_part = nullptr;  // deterministic mode: per-block partial sums of the head gradient
  // NINT_FLAG_TANGENT: input tangent [T][B][H][W][cx_pad0] E, the tangent GEMM's fp32 dump [B][H][W][4 * max hc], a zero
  // head bias; maps over tX and over the caller's tangent bank (re-encoded when its pointer or length changes)
  bool tangent = false;
  uint8_t* tX = nullptr;
  float* traw = nullptr;
  float* tzero = nullptr;
  CUtensorMap tm_tX, tmb_tX;
  const void* tbank_ptr = nullptr;
  long long tbank_frames = 0;
  // NINT_FLAG_SECOND_ORDER: [2][B][H][W][max(cin_rows0, hc_l)] fp32 dgrad dump of the pass (primal, then tangent);
  // tangent_kept: the per-step tangent dumps belong to the last forward
  bool second_order = false, tangent_kept = false;
  float* sraw = nullptr;
  // NINT_FLAG_PARAM_TANGENT: the head's parameter direction (dw [hc], db) and whether one is set; param_in_tangent:
  // the last tangent pass included a parameter direction (the second-order pass has no parameter terms yet)
  bool param_tangent = false, dhead_set = false, param_in_tangent = false;
  float *thead_w = nullptr, *thead_b = nullptr;
  // both flags: the tangent pass keeps dh of every step (tH [T+1] slots, slot 0 = dh0) and the second-order pass
  // (a, da) of every step (sA [T][2B]); head_sums = the pass's head reductions {grad w [hc], grad b, hvp w [hc], hvp b};
  // soa_params: the last second-order pass belongs to the current forward and tangent (the params call may run)
  bool hist = false, soa_params = false;
  float* head_sums = nullptr;
  CUtensorMap tmw_tX, tmp_tX, tmbw_tX, tmbp_tX;
  unsigned* step_done = nullptr;   // [T][B] tile counters of a time-fused conv launch (ConvGemmParams::step_done)
  // consecutive time steps of a layer as ONE persistent launch whose tiles wait on the previous step's tiles of the same
  // image (ConvGemmParams::n_steps).  -1: automatic -- BPTT launches are fused while they are short (bwd_should_fuse),
  // forward launches never (with PDL the forward kernel runs at its steady-state rate from start to end, and the
  // storers' wait for write completion costs it more than the drain it saves: DESIGN.md section 6).  NINT_FUSE_STEPS=
  // 0 / 1 / 2 / 3 forces nothing / forward / BPTT / both.
  int fuse_steps = -1;
  bool head_set = false;
  bool zero_init = true;
  bool fwd_done = false;
  bool gates_valid = false; // the saved activated gates of the last forward are intact (BPTT overwrites them in place)
  bool bptt_done = false;   // dgates of the last forward are in place: nint_backward_wgrad may run
  bool deterministic = false, input_grad = false, state_grad = false;
  // Programmatic dependent launch of the conv kernels (NINT_PDL=1 switches it on).  OFF by default: it buys 0.4-0.6 % at
  // cfg 2, but with the last build of round 2 the one-launch-per-step schedule of the reference's three-layer recipe
  // died with "unspecified launch failure" at a random step in 4 of 8 (and 5 of 12) 150-step runs with it and in 0 of
  // 8 without it (same box, alternating: tools/gpurun/r2_run_fz.sh; DESIGN.md section 6).  Cause unknown.
  int pdl = 0;
  int sub_batch = 0;        // > 0: sub-batch-major schedule (images [b0, b0 + sub_batch) run all T steps before the next
                            // slice, so a step's recurrent operands are still in L2 when the next step reads them)
  int final_slot_h = 0, final_slot_c = 0;
  int cluster = 2;        // 2: CTA pairs (tcgen05 cta_group::2) where the layer geometry allows, 1: single CTAs
  int debug_flags = 0;
  int ones_lane = -1;     // padding channel of X that holds 1.0 (bias gradient through the wgrad GEMM), -1: no spare channel
  int plan_g = 0, plan_ns = 0;   // NINT_PLAN_G / NINT_PLAN_NS: experiment knobs of the backward kernel's shared-memory plan
  Profile prof;
};

namespace {

// every kernel launch of the library goes through here: counts it and, when the plan is being
// profiled, brackets it with CUDA events on the launching stream
template <typename F>
int launch(nint_plan* p, int cls, cudaStream_t st, const char* what, F&& f) {
  cudaEvent_t e1 = nullptr;
  if (p && p->prof.on) {
    Profile& pr = p->prof;
    if (pr.pool.size() < 2 * (pr.used + 1)) {
      cudaEvent_t a, b;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return fail("cudaEventCreate failed");
      pr.pool.push_back(a);
      pr.pool.push_back(b);
    }
    e1 = pr.pool[2 * pr.used + 1];
    if (pr.cls.size() <= pr.used) pr.cls.resize(pr.used + 1), pr.weight.resize(pr.used + 1);
    pr.cls[pr.used] = cls;
    pr.weight[pr.used] = 1;
    cudaEventRecord(pr.pool[2 * pr.used], st);
    ++pr.used;
  }
  cudaError_t e = f();
  if (e1) cudaEventRecord(e1, st);
  if (e != cudaSuccess) return fail("%s failed: %s", what, cudaGetErrorString(e));
  ++g_launches[cls];
  return 0;
}
#define LAUNCH(plan, cls, st, call) \
  do { if (launch(plan, cls, st, #call, [&]() { return (call); })) return 1; } while (0)

// the kernels work on 8 x 16 pixel tiles (UMMA M = 128 rows; 8-pixel rows = one 512-byte swizzle atom of the
// halo buffers); grids that are not multiples are handled by TMA's out-of-bounds fill / clipping
int pick_tile(int H, int W, int* tw_out, int* th_out) {
  (void)H; (void)W;
  *tw_out = 8;
  *th_out = 16;
  return 0;
}

// wgrad = true: 32-channel box; tf32 then needs the 128B swizzle with 32-byte atoms (the MN-major tf32
// UMMA layout), bf16 is the same 64-byte box either way.
// slot_images: images between consecutive slots (0: B; a view of B images out of larger slots)
int encode_act_map(CUtensorMap* m, int dtype, void* base, int C, int W, int H, int B, int slots, int ce, int tw,
                   int th, bool wgrad = false, int halo = 0, long long slot_images = 0) {
  tw += 2 * halo;
  th += 2 * halo;
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail("cuTensorMapEncodeTiled not available (no CUDA driver?)");
  const cuuint64_t es = dtype == BF16 ? 2 : 4;
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B, (cuuint64_t)slots};
  cuuint64_t strides[4] = {C * es, (cuuint64_t)W * C * es, (cuuint64_t)H * W * C * es,
                           (cuuint64_t)(slot_images ? slot_images : B) * H * W * C * es};
  cuuint32_t box[5] = {(cuuint32_t)(wgrad ? 32 : ce), (cuuint32_t)tw, (cuuint32_t)th, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUtensorMapSwizzle sw = (wgrad && dtype == TF32) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = enc(m, dtype == BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, base,
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(activation C=%d W=%d H=%d B=%d slots=%d) -> %d", C, W, H, B, slots, (int)r);
  return 0;
}

// general activation box: `box_c` channels x (tw + 2*halo) x (th + 2*halo) pixels with an explicit swizzle
int encode_act_box(CUtensorMap* m, int dtype, void* base, int C, int W, int H, int B, int slots, int box_c, int tw,
                   int th, int halo, CUtensorMapSwizzle sw, long long slot_images = 0) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail("cuTensorMapEncodeTiled not available (no CUDA driver?)");
  const cuuint64_t es = dtype == BF16 ? 2 : 4;
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B, (cuuint64_t)slots};
  cuuint64_t strides[4] = {C * es, (cuuint64_t)W * C * es, (cuuint64_t)H * W * C * es,
                           (cuuint64_t)(slot_images ? slot_images : B) * H * W * C * es};
  cuuint32_t box[5] = {(cuuint32_t)box_c, (cuuint32_t)(tw + 2 * halo), (cuuint32_t)(th + 2 * halo), 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, dtype == BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, base,
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(box C=%d box_c=%d halo=%d) -> %d", C, box_c, halo, (int)r);
  return 0;
}

// epilogue I/O box: `box_c` channels x 8 x 16 pixels of a channels-last tensor with element size `es`;
// the swizzle span equals the box row (32 / 64 / 128 bytes) so per-pixel 16-byte accesses are conflict free
int encode_io_map(CUtensorMap* m, bool fp32, void* base, int C, int W, int H, int B, int slots, int box_c) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail("cuTensorMapEncodeTiled not available (no CUDA driver?)");
  const cuuint64_t es = fp32 ? 4 : 2;
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B, (cuuint64_t)slots};
  cuuint64_t strides[4] = {C * es, (cuuint64_t)W * C * es, (cuuint64_t)H * W * C * es,
                           (cuuint64_t)B * H * W * C * es};
  cuuint32_t box[5] = {(cuuint32_t)box_c, 8, 16, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const int row_bytes = box_c * (int)es;
  CUtensorMapSwizzle sw;
  if (row_bytes == 32) sw = CU_TENSOR_MAP_SWIZZLE_32B;
  else if (row_bytes == 64) sw = CU_TENSOR_MAP_SWIZZLE_64B;
  else if (row_bytes == 128) sw = CU_TENSOR_MAP_SWIZZLE_128B;
  else return fail("encode_io_map: unsupported box row of %d bytes", row_bytes);
  CUresult r = enc(m, fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(io C=%d W=%d H=%d B=%d slots=%d box=%d) -> %d", C, W, H, B, slots, box_c, (int)r);
  return 0;
}

// packed weight panels [chunk-tap index][n_tile rows][ce elements] seen as a 3-D tensor; a box is the `w_rows`
// rows one CTA holds (all of N, or half in CTA-pair mode) of `ts` consecutive taps = one weight stage
int encode_w_map(CUtensorMap* m, int dtype, void* base, long long chunk_taps, int ce, int n_tile, int w_rows, int ts) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail("cuTensorMapEncodeTiled not available (no CUDA driver?)");
  const cuuint64_t es = dtype == BF16 ? 2 : 4;
  cuuint64_t dims[3] = {(cuuint64_t)ce, (cuuint64_t)n_tile, (cuuint64_t)chunk_taps};
  cuuint64_t strides[2] = {ce * es, (cuuint64_t)n_tile * ce * es};
  cuuint32_t box[3] = {(cuuint32_t)ce, (cuuint32_t)w_rows, (cuuint32_t)ts};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, dtype == BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base,
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(weights chunk_taps=%lld n_tile=%d rows=%d ts=%d) -> %d", chunk_taps, n_tile, w_rows, ts, (int)r);
  return 0;
}

// UMMA instruction descriptor (kind::f16 / kind::tf32, fp32 accumulate); see nint_common.cuh
uint32_t idesc_of(int dtype, int m, int n, int a_mn, int b_mn) {
  const uint32_t fmt = dtype == BF16 ? 1u : 2u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(a_mn & 1) << 15) | ((uint32_t)(b_mn & 1) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

size_t act_bytes(const nint_plan* p, int slots, int c) {
  return static_cast<size_t>(slots) * p->B * p->H * p->W * c * p->esize;
}

// carve (or just measure, when base == nullptr) the workspace
size_t carve(nint_plan* p, uint8_t* base) {
  size_t off = 0;
  auto take = [&](size_t bytes) -> uint8_t* {
    uint8_t* r = base ? base + off : nullptr;
    off += align_up(bytes, 1024);
    return r;
  };
  const bool tr = p->cfg.training != 0;
  const size_t npix = static_cast<size_t>(p->B) * p->H * p->W;
  p->X = take(act_bytes(p, p->T, p->layer[0].cx_pad));
  for (int l = 0; l < p->L; ++l) {
    Layer& y = p->layer[l];
    y.Hs = take(act_bytes(p, y.nslots_h, y.hc_pad));
    y.Cs = reinterpret_cast<float*>(take(static_cast<size_t>(y.nslots_c) * npix * y.hc * 4));
    y.G = tr ? take(act_bytes(p, p->T, 4 * y.hc)) : nullptr;
    y.dC = tr ? reinterpret_cast<float*>(take(npix * y.hc * 4)) : nullptr;
    const size_t wrow = static_cast<size_t>(p->ce) * p->esize;  // 64 bytes
    y.wx = take(static_cast<size_t>(y.n_blocks) * y.taps * y.chx * y.n_tile * wrow);
    y.wh = take(static_cast<size_t>(y.n_blocks) * y.taps * y.chh * y.n_tile * wrow);
    y.bias_q = reinterpret_cast<float*>(take(4 * y.hc * 4));
    if (tr) {
      const int nch = 4 * y.hc / p->ce;
      y.wdx = (l > 0 || p->input_grad || p->second_order) ? take(static_cast<size_t>(y.taps) * nch * y.cin_rows * wrow) : nullptr;
      y.wdh = take(static_cast<size_t>(y.taps) * nch * y.hc * wrow);
      y.dw_acc_bytes = static_cast<size_t>(y.taps) * 4 * y.hc * y.ncols * 4;
      const size_t slices = p->deterministic ? static_cast<size_t>(y.det_splits) : 1;
      y.dw_acc = reinterpret_cast<float*>(take(y.dw_acc_bytes * slices));
      y.db_acc = reinterpret_cast<float*>(take(4 * y.hc * 4 * slices));
      y.db_resid = p->dtype == TF32 ? reinterpret_cast<float*>(take(static_cast<size_t>(kResidCtas) * 4 * 4 * y.hc * 4)) : nullptr;
    }
  }
  const Layer& top = p->layer[p->L - 1];
  p->head_w = reinterpret_cast<float*>(take(top.hc * 4));
  p->head_b = reinterpret_cast<float*>(take(16));
  if (tr && p->deterministic)
    p->head_part = reinterpret_cast<float*>(take(static_cast<size_t>(head_bwd_blocks(p->B)) * (top.hc_real + 1) * 4));
  p->step_done = reinterpret_cast<unsigned*>(take(static_cast<size_t>(p->T) * p->B * 4));
  // dgrad dump: dx / the cell's dh (layer 0) and dh0 of every layer (nint_backward_initial_state)
  int raw_cols = 0;
  if (tr && p->input_grad) raw_cols = p->layer[0].cin_rows > p->layer[0].hc ? p->layer[0].cin_rows : p->layer[0].hc;
  if (tr && p->state_grad)
    for (int l = 0; l < p->L; ++l) raw_cols = raw_cols > p->layer[l].hc ? raw_cols : p->layer[l].hc;
  if (raw_cols > 0) p->raw = reinterpret_cast<float*>(take(npix * raw_cols * 4));
  if (tr && p->input_grad) p->dh_ext = reinterpret_cast<float*>(take(npix * p->layer[0].hc * 4));
  if (tr && p->state_grad)
    for (int l = 0; l < p->L; ++l) p->layer[l].dh_ext = reinterpret_cast<float*>(take(npix * p->layer[l].hc * 4));
  if (tr && p->tangent) {
    p->tX = take(act_bytes(p, p->T, p->layer[0].cx_pad));
    int max_hc = 0;
    for (int l = 0; l < p->L; ++l) {
      Layer& y = p->layer[l];
      y.tH = take(act_bytes(p, p->hist ? p->T + 1 : 2, y.hc_pad));
      y.tC = reinterpret_cast<float*>(take(npix * y.hc * 4 * (p->second_order ? p->T + 1 : 1)));
      if (p->second_order) y.tR = reinterpret_cast<float*>(take(static_cast<size_t>(p->T) * npix * 4 * y.hc * 4));
      max_hc = max_hc > y.hc ? max_hc : y.hc;
    }
    if (!p->second_order) p->traw = reinterpret_cast<float*>(take(npix * 4 * max_hc * 4));
    p->tzero = reinterpret_cast<float*>(take(16));
  }
  if (tr && p->param_tangent) {
    const size_t wrow = static_cast<size_t>(p->ce) * p->esize;
    for (int l = 0; l < p->L; ++l) {
      Layer& y = p->layer[l];
      y.twx = take(static_cast<size_t>(y.n_blocks) * y.taps * y.chx * y.n_tile * wrow);
      y.twh = take(static_cast<size_t>(y.n_blocks) * y.taps * y.chh * y.n_tile * wrow);
      y.tbias_q = reinterpret_cast<float*>(take(4 * y.hc * 4));
    }
    p->thead_w = reinterpret_cast<float*>(take(top.hc * 4));
    p->thead_b = reinterpret_cast<float*>(take(16));
  }
  if (tr && p->hist) {
    const size_t wrow = static_cast<size_t>(p->ce) * p->esize;
    for (int l = 0; l < p->L; ++l) {
      Layer& y = p->layer[l];
      const int nch = 4 * y.hc / p->ce;
      y.twdx = take(static_cast<size_t>(y.taps) * nch * y.cin_rows * wrow);
      y.twdh = take(static_cast<size_t>(y.taps) * nch * y.hc * wrow);
    }
    p->head_sums = reinterpret_cast<float*>(take(static_cast<size_t>(2 * (top.hc + 1) + 1) * 4));
  }
  if (tr && p->second_order) {
    int cols = p->layer[0].cin_rows;
    for (int l = 0; l < p->L; ++l) {
      Layer& y = p->layer[l];
      y.sA = take(act_bytes(p, p->hist ? 2 * p->T : 2, 4 * y.hc));
      y.sK = reinterpret_cast<float*>(take(2 * npix * y.hc * 4));
      cols = cols > y.hc ? cols : y.hc;
    }
    p->sraw = reinterpret_cast<float*>(take(2 * npix * cols * 4));
  }
  return off;
}

inline uint8_t* slot_ptr(const nint_plan* p, uint8_t* base, int slot, int c) {
  return base + act_bytes(p, 1, c) * slot;
}
inline float* cslot_ptr(const nint_plan* p, const Layer& y, int slot) {
  return y.Cs + static_cast<size_t>(slot) * p->B * p->H * p->W * y.hc;
}
// the tangent pass's dc before step `slot` (dc_{slot-1}): one running buffer, or the per-step history of second-order plans
inline float* tc_slot(const nint_plan* p, const Layer& y, int slot) {
  return p->second_order ? y.tC + static_cast<size_t>(slot) * p->B * p->H * p->W * y.hc : y.tC;
}

void fill_common(const nint_plan* p, const Layer& y, ConvGemmParams& g) {
  memset(&g, 0, sizeof(g));
  g.debug_flags = p->debug_flags;
  g.pdl = p->pdl;
  g.plan_g = p->plan_g; g.plan_ns = p->plan_ns;
  g.B = p->B; g.b0 = 0; g.H = p->H; g.W = p->W;
  g.tile_w = p->tile_w; g.tile_h = p->tile_h; g.tiles_x = p->tiles_x; g.tiles_y = p->tiles_y;
  g.hc = y.hc; g.hc_pad = y.hc_pad; g.hcb = y.hcb;
  g.n_steps = 1;
  g.c_prev_none_step = -1;
}

// turn g (set up for its first step) into a time-fused launch of n_steps consecutive steps: zero the tile counters
int arm_fused(nint_plan* p, ConvGemmParams& g, int n_steps, int storer_warps, cudaStream_t st) {
  g.n_steps = n_steps;
  g.step_done = p->step_done;
  g.step_target = static_cast<unsigned>(p->tiles_x * p->tiles_y * g.n_blocks * storer_warps);
  if (reinterpret_cast<uint8_t*>(p->step_done) < p->ws ||
      reinterpret_cast<uint8_t*>(p->step_done + static_cast<size_t>(n_steps) * p->B) > p->ws + p->ws_bytes)
    return fail("internal: step counters outside the workspace (%p, ws %p + %zu)", (void*)p->step_done, (void*)p->ws, p->ws_bytes);
  CK(cudaMemsetAsync(p->step_done, 0, static_cast<size_t>(n_steps) * p->B * 4, st));
  return 0;
}

// CTA-pair mode (cluster of 2, tcgen05 cta_group::2; halo variant only): every CTA holds half of the N rows
// of a weight stage, which must stay a whole number of 8-row swizzle atoms with N a multiple of 32
int fwd_cluster(const nint_plan* p, int l) {
  (void)l;
  return p->cluster;   // n_tile = 4*hcb: multiple of 64
}
int bwd_cluster(const nint_plan* p, int l) {
  return p->layer[l].hc % 32 == 0 ? p->cluster : 1;    // n_tile = hc
}

// weight map of layer `y` for one K segment: which = 0 wx, 1 wh (forward, N = n_tile per n-block), 2 wdx, 3 wdh
// (dgrad, N = n_tile input channels), 4 twx, 5 twh (the parameter tangent, laid out as wx / wh); `rows` = N rows per
// CTA, `ts` = taps per weight stage
int get_w_map(nint_plan* p, Layer& y, int which, int n_tile, int rows, int ts, CUtensorMap* out) {
  for (const Layer::WMap& w : y.wmaps[which])
    if (w.ts == ts && w.rows == rows && w.n_tile == n_tile) { *out = w.map; return 0; }
  void* const bases[8] = {y.wx, y.wh, y.wdx, y.wdh, y.twx, y.twh, y.twdx, y.twdh};
  void* base = bases[which];
  if (!base) return fail("internal: packed weight tensor %d of this layer was not allocated", which);
  long long chunk_taps;
  if (which == 0 || which == 4) chunk_taps = (long long)y.n_blocks * y.chx * y.taps;
  else if (which == 1 || which == 5) chunk_taps = (long long)y.n_blocks * y.chh * y.taps;
  else chunk_taps = (long long)(4 * y.hc / p->ce) * y.taps;
  Layer::WMap w;
  w.ts = ts; w.rows = rows; w.n_tile = n_tile;
  if (encode_w_map(&w.map, p->dtype, base, chunk_taps, p->ce, n_tile, rows, ts)) return 1;
  y.wmaps[which].push_back(w);
  *out = w.map;
  return 0;
}

// images [b0, b0 + nb) of a launch (nb <= 0: the whole batch)
inline void set_batch_range(const nint_plan* p, ConvGemmParams& g, int b0, int nb) {
  g.b0 = nb > 0 ? b0 : 0;
  g.B = nb > 0 ? nb : p->B;
}

// step-independent launch parameters of layer l's gate convolution (have_state: with the h_{t-1} K segment)
int fwd_conv_params(nint_plan* p, int l, bool have_state, int epi, ConvGemmParams& g) {
  Layer& y = p->layer[l];
  const bool tr = p->cfg.training != 0;
  const bool bank = l == 0 && p->x_bank;
  Layer::CachedConv* cache = epi == EPI_FWD ? &y.fwd_cache[have_state ? 1 : 0][bank ? 1 : 0] : nullptr;
  if (cache && cache->valid) {
    g = cache->g;
  } else {
    fill_common(p, y, g);
    g.n_tile = y.n_tile;
    g.n_blocks = y.n_blocks;
    g.cluster = fwd_cluster(p, l);
    g.idesc = idesc_of(p->dtype, 128 * g.cluster, y.n_tile, 0, 0);
    // segment 0: x_t (layer 0) or the h_t of the layer below (model.py:266,271)
    int s = 0;
    g.seg[s].tmap_act = l == 0 ? (bank ? p->tmb_X : p->tm_X) : p->layer[l - 1].tm_H_up;
    g.seg[s].wsel = 0;
    g.seg[s].ksize = y.k;
    g.seg[s].nchunks = y.chx;
    ++s;
    if (have_state) {  // h_{t-1} == 0 contributes nothing: skip its K-segment (SURVEY.md K1)
      g.seg[s].tmap_act = y.tm_H;
      g.seg[s].wsel = 1;
      g.seg[s].ksize = y.k;
      g.seg[s].nchunks = y.chh;
      ++s;
    }
    g.nseg = s;
    // epilogue I/O (TMA boxes): c_{t-1} -> c_t (in place at inference), h_t, activated gates (training)
    g.tm_c = y.tme_C; g.tm_h = y.tme_H; g.tm_g = y.tme_G; g.tm_dc = y.tme_dC;
    g.slot_g = (tr && epi == EPI_FWD) ? 0 : -1;   // only its sign enters the shared-memory plan
    if (conv_halo_plan(epi, p->dtype, g)) return fail("layer %d: the conv kernel's shared-memory plan does not fit (hidden %d, k %d)", l, y.hc, y.k);
    for (int i = 0; i < g.nseg; ++i)
      if (get_w_map(p, y, g.seg[i].wsel, g.n_tile, g.n_tile / g.cluster, g.seg[i].ts, &g.seg[i].tmap_w)) return 1;
    if (cache) { cache->g = g; cache->valid = true; }
  }
  return 0;
}

// one fused cell step of layer l at time t (model.py:216-231) for images [b0, b0 + nb); n_steps > 1: steps t .. t+n_steps-1
// as ONE time-fused launch (all of them must have a recurrent state: t >= 1, or an explicit initial state)
int cell_step(nint_plan* p, int l, int t, int epi, float* raw_out, cudaStream_t st, int b0 = 0, int nb = 0, int n_steps = 1) {
  Layer& y = p->layer[l];
  const bool tr = p->cfg.training != 0;
  const bool have_state = !(t == 0 && p->zero_init);
  const bool bank = l == 0 && p->x_bank;
  ConvGemmParams g;
  if (fwd_conv_params(p, l, have_state, epi, g)) return 1;
  // ---- what changes from step to step: slots, batch range, bank indices
  const int in_slot_h = tr ? t : (t & 1);
  const int out_slot_h = tr ? t + 1 : ((t + 1) & 1);
  g.seg[0].slot = l == 0 ? t : (tr ? t + 1 : ((t + 1) & 1));
  g.seg[0].win_start = bank ? p->win_start : nullptr;
  g.seg[0].bank_frames = bank ? static_cast<int>(p->bank_frames) : 0;
  if (have_state) g.seg[1].slot = in_slot_h;
  g.slot_c_in = have_state ? (tr ? t : 0) : -1;
  g.slot_c_out = tr ? t + 1 : 0;
  g.slot_h_out = out_slot_h;
  g.slot_g = (tr && epi == EPI_FWD) ? t : -1;
  g.bias_q = (y.bias_folded && epi == EPI_FWD) ? nullptr : y.bias_q;   // folded: the GEMM adds it (set_weights decides)
  g.raw_out = raw_out;
  set_batch_range(p, g, b0, nb);
  g.n_steps = 1;
  if (n_steps > 1) {
    if (!have_state || epi != EPI_FWD || nb > 0) return fail("internal: time-fused forward launch without a recurrent state");
    g.d_seg[0] = g.d_seg[1] = g.d_h_out = g.d_g = 1;
    g.d_c_in = g.d_c_out = tr ? 1 : 0;
    g.ring_bits = tr ? 0 : ((l > 0 ? 1 : 0) | 2 | 16);   // inference: the h history is a 2-slot ring
    if (arm_fused(p, g, n_steps, 2, st)) return 1;
  }
  LAUNCH(p, (epi == EPI_FWD ? K_FWD : K_OTHER), st, launch_conv_halo(epi, p->dtype, g, p->num_sms, st));
  if (p->prof.on && p->prof.used > 0) p->prof.weight[p->prof.used - 1] = n_steps;
  return 0;
}

// dgrad convolution without the gate epilogue: raw[b][y][x][n] = sum dgates_t (*) flip(W) for the N = `n_rows` input
// channels of packed operand `wsel` (2: x part, 3: h part) of layer l; fp32 dump through the EPI_RAW epilogue
int dgrad_raw(nint_plan* p, int l, int t, int wsel, int n_rows, float* raw_out, cudaStream_t st) {
  Layer& y = p->layer[l];
  ConvGemmParams g;
  fill_common(p, y, g);
  g.n_tile = n_rows;
  g.n_blocks = 1;
  g.cluster = (n_rows % 32 == 0) ? p->cluster : 1;
  g.idesc = idesc_of(p->dtype, 128 * g.cluster, n_rows, 0, 0);
  g.seg[0].tmap_act = y.tm_G; g.seg[0].wsel = wsel; g.seg[0].slot = t;
  g.seg[0].ksize = y.k; g.seg[0].nchunks = 4 * y.hc / p->ce;
  g.nseg = 1;
  g.tm_c = y.tme_C; g.tm_h = y.tme_H; g.tm_g = y.tme_G; g.tm_dc = y.tme_dC;
  g.slot_g = g.slot_c_in = g.slot_c_out = g.slot_h_out = g.slot_c_prev = -1;
  g.raw_out = raw_out;
  if (conv_halo_plan(EPI_RAW, p->dtype, g)) return fail("layer %d: the dgrad kernel's shared-memory plan does not fit (N %d, k %d)", l, n_rows, y.k);
  if (get_w_map(p, y, wsel, g.n_tile, g.n_tile / g.cluster, g.seg[0].ts, &g.seg[0].tmap_w)) return 1;
  LAUNCH(p, K_OTHER, st, launch_conv_halo(EPI_RAW, p->dtype, g, p->num_sms, st));
  return 0;
}

}  // namespace

// Column blocks of a layer's weight gradient (Layer::WgBlock).  CTA-pair kernel (bf16, 4*hc % 256 == 0): the whole
// row when it fits (N <= 256, >= 2 B stages), else the x part and the h part as two launches.  Otherwise the
// single-CTA kernel with as few blocks of whole 32-channel panels as leave it two B stages.
static int plan_wgrad_blocks(nint_plan* p, Layer& y) {
  y.wg_blocks.clear();
  const int px = y.cx_pad / 32, ph = y.hc_pad / 32;
  auto pair_block = [&](int col0, int x_cols, int cols) {
    Layer::WgBlock b;
    b.col0 = col0; b.cols = cols;
    b.nch_x = x_cols / 32; b.nch_h = (cols - x_cols) / 32;
    b.pair = true;
    b.pw = wgrad_pair_panel_width(x_cols, cols);
    b.a_bufs = 3;
    b.b_stages = wgrad_pair_b_stages(x_cols, cols, y.k);
    b.n_mma = cols;
    return b;
  };
  // tf32 CTA-pair kernel: 32-channel fp32 panels, each CTA takes whole panels, so N is rounded up to an even panel
  // count (the extra panel lies outside the h tensor: TMA zero-fills it); it has no ones-panel bias MMA, so it
  // needs the constant-1 channel of layer 0
  if (p->cluster == 2 && p->dtype == TF32 && (4 * y.hc) % 256 == 0 && &y == &p->layer[0] && p->ones_lane >= 0) {
    const int n_mma = (y.ncols / 32 + 1) / 2 * 64;
    const int st = n_mma <= 256 ? wgrad_pair_b_stages_tf32(n_mma, y.k) : 0;
    if (st >= 2) {
      Layer::WgBlock b;
      b.col0 = 0; b.cols = y.ncols; b.n_mma = n_mma;
      b.nch_x = y.cx_pad / 32; b.nch_h = y.hc_pad / 32;
      b.pair = true; b.pw = 32; b.a_bufs = 2; b.b_stages = st;
      y.wg_blocks.push_back(b);
      return 0;
    }
  }
  if (p->cluster == 2 && p->dtype == BF16 && (4 * y.hc) % 256 == 0) {
    if (wgrad_pair_supported(p->dtype, 4 * y.hc, y.cx_pad, y.ncols, y.k)) {
      y.wg_blocks.push_back(pair_block(0, y.cx_pad, y.ncols));
      return 0;
    }
    if (wgrad_pair_supported(p->dtype, 4 * y.hc, y.cx_pad, y.cx_pad, y.k) &&
        wgrad_pair_supported(p->dtype, 4 * y.hc, 0, y.hc_pad, y.k)) {
      y.wg_blocks.push_back(pair_block(0, y.cx_pad, y.cx_pad));
      y.wg_blocks.push_back(pair_block(y.cx_pad, 0, y.hc_pad));
      return 0;
    }
  }
  const int panels = px + ph, bpb = wgrad_b_panel_bytes(p->dtype, 1, y.k);
  int per = panels, a_bufs = 0, b_stages = 0;
  for (; per >= 1; --per) {
    wgrad_pick_buffers(p->dtype, per, bpb, &a_bufs, &b_stages);
    if (per * 32 <= 256 && (b_stages >= 2 || (per == 1 && b_stages >= 1))) break;
  }
  if (per < 1) return 1;
  for (int j0 = 0; j0 < panels; j0 += per) {
    const int j1 = j0 + per < panels ? j0 + per : panels;
    Layer::WgBlock b;
    b.col0 = j0 * 32; b.cols = b.n_mma = (j1 - j0) * 32;
    b.nch_x = (j1 < px ? j1 : px) - (j0 < px ? j0 : px);
    b.nch_h = (j1 - j0) - b.nch_x;
    b.chan0_x = (j0 < px ? j0 : px) * 32;
    b.chan0_h = (j0 > px ? j0 - px : 0) * 32;
    wgrad_pick_buffers(p->dtype, j1 - j0, bpb, &b.a_bufs, &b.b_stages);
    y.wg_blocks.push_back(b);
  }
  return 0;
}

// Launch parameters of column block `bi` of layer l's weight gradient: operand maps, tap groups, split-K shares.
// Also used (with the nominal 148 SMs, before any device is known) to size the deterministic mode's partial buffers.
static int wgrad_params(nint_plan* p, int l, size_t bi, int num_sms, WgradParams& w) {
  Layer& y = p->layer[l];
  const int T = p->T;
  const Layer::WgBlock& blk = y.wg_blocks[bi];
  const int bias_col = (l == 0) ? p->ones_lane : -1;
  const long long total_tiles = static_cast<long long>(T) * p->B * p->tiles_x * p->tiles_y;
  memset(&w, 0, sizeof(w));
  w.halo = 1;
  w.debug_flags = p->debug_flags;
  w.b_panel_bytes = wgrad_b_panel_bytes(p->dtype, w.halo, y.k);
  w.slot_b0[0] = l == 0 ? 0 : 1;
  w.slot_b0[1] = 0;
  w.nchunks_b[0] = blk.nch_x;
  w.nchunks_b[1] = blk.nch_h;
  w.chan0[0] = blk.chan0_x;
  w.chan0[1] = blk.chan0_h;
  w.T = T; w.B = p->B; w.H = p->H; w.W = p->W;
  w.tile_w = p->tile_w; w.tile_h = p->tile_h; w.tiles_x = p->tiles_x; w.tiles_y = p->tiles_y;
  w.ksize = y.k;
  w.hc4 = 4 * y.hc;
  w.pair = blk.pair ? 1 : 0;
  const bool bank = l == 0 && p->x_bank;
  w.win_start = bank ? p->win_start : nullptr;
  if (w.pair && p->dtype == BF16) {
    w.tmap_dg = y.tmp_G;
    w.tmap_b[0] = l == 0 ? (bank ? p->tmbp_X : p->tmp_X) : p->layer[l - 1].tmp_H_up;
    w.tmap_b[1] = y.tmp_H;
  } else {   // single-CTA kernel, and the tf32 pair kernel: 32-channel boxes (bf16 SWIZZLE_64B / tf32 128B_ATOM_32B)
    w.tmap_dg = y.tmw_G;
    w.tmap_b[0] = l == 0 ? (bank ? p->tmbw_X : p->tmw_X) : p->layer[l - 1].tmw_H_up;
    w.tmap_b[1] = y.tmw_H;
  }
  // a block without x (or h) panels never dereferences that map, but kernel parameters must be valid maps
  if (blk.nch_x == 0) { w.tmap_b[0] = w.tmap_b[1]; w.win_start = nullptr; }
  if (blk.nch_h == 0) w.tmap_b[1] = w.tmap_b[0];
  w.m_blocks = w.pair ? w.hc4 / 256 : (w.hc4 + 127) / 128;
  w.ncols = y.ncols;
  w.acc_cols = blk.n_mma;
  w.real_cols = blk.cols;
  w.col0 = blk.col0;
  // The bias gradient is either free (layer 0: x carries 1.0 in padding channel `ones_lane`, so db is that column
  // of the centre tap) or costs 32 more accumulator columns and one N=32 MMA per K step against a panel of ones,
  // in the first column block's lightest tap group (the last one when it has room, else the first).
  // tap groups: a CTA keeps (taps in group) x acc_cols accumulator columns in TMEM (512 available)
  const int bias_cols = (bias_col >= 0 || bi > 0) ? 0 : 32;
  const int tpg = 512 / blk.n_mma;                     // taps per group
  if (tpg < 1) return fail("wgrad: %d columns exceed the accumulator", blk.n_mma);
  int ng = 0, tap = 0;
  w.group_tap0[0] = 0;
  const int rest = y.taps % tpg;
  const bool bias_last = rest > 0 && rest * blk.n_mma + bias_cols <= 512;   // a partial last group with room for the bias
  const int g0 = bias_last ? tpg : ((512 - bias_cols) / blk.n_mma < tpg ? (512 - bias_cols) / blk.n_mma : tpg);
  if (g0 < 1) return fail("wgrad: %d columns leave no room for the bias columns", blk.n_mma);
  while (tap < y.taps) {
    const int n = ng == 0 ? g0 : tpg;
    tap = tap + n > y.taps ? y.taps : tap + n;
    if (ng + 1 > kMaxWgradGroups) return fail("wgrad: too many tap groups");
    w.group_tap0[++ng] = tap;
  }
  w.bias_group = bias_cols == 0 ? -1 : (bias_last ? ng - 1 : 0);
  w.n_groups = ng;
  // split-K over pixel tiles: every group gets a share of the SMs in proportion to its MMA cycles per K step
  // (pair MMA: ~N/2 cycles with a ~40-cycle floor; 1-CTA MMA: ~N*0.67 with a ~88-cycle floor -- DESIGN.md 4)
  {
    int units = (w.pair ? num_sms / 2 : num_sms) / w.m_blocks;   // (group, split) slots
    if (units < ng) units = ng;
    auto mma_cost = [&](int n) { return w.pair ? (n / 2 > 40 ? n / 2 : 40) : (n * 2 / 3 > 88 ? n * 2 / 3 : 88); };
    int cost[kMaxWgradGroups], tot = 0;
    for (int g = 0; g < ng; ++g) {
      cost[g] = (w.group_tap0[g + 1] - w.group_tap0[g]) * mma_cost(blk.n_mma) + (g == w.bias_group ? mma_cost(32) : 0);
      tot += cost[g];
    }
    const bool even = (p->debug_flags & 64) != 0;     // experiment: the same split count for every group
    int used = 0;
    for (int g = 0; g < ng; ++g) {
      int sp = even ? units / ng : static_cast<int>(static_cast<long long>(units) * cost[g] / tot);
      if (sp < 1) sp = 1;
      w.group_splits[g] = sp;
      used += sp;
    }
    // hand the remaining slots to whichever group has the most work per split
    while (!even && used < units) {
      int best = 0;
      for (int g = 1; g < ng; ++g)
        if (static_cast<long long>(cost[g]) * w.group_splits[best] > static_cast<long long>(cost[best]) * w.group_splits[g]) best = g;
      ++w.group_splits[best];
      ++used;
    }
    w.group_unit0[0] = 0;
    for (int g = 0; g < ng; ++g) {
      if (w.group_splits[g] > total_tiles) w.group_splits[g] = static_cast<int>(total_tiles);
      w.group_unit0[g + 1] = w.group_unit0[g] + w.m_blocks * w.group_splits[g];
    }
  }
  w.b_pw = blk.pw;
  w.a_bufs = blk.a_bufs;
  w.b_stages = blk.b_stages;
  if (w.b_stages < 1) return fail("wgrad: operand panels do not fit in shared memory");
  w.idesc = idesc_of(p->dtype, w.pair ? 256 : 128, blk.n_mma, 1, 1);
  w.idesc_bias = idesc_of(p->dtype, w.pair ? 256 : 128, 32, 1, 1);
  w.dw_acc = y.dw_acc;
  w.db_acc = y.db_acc;
  w.dw_part = p->deterministic ? y.dw_acc : nullptr;
  w.db_part = p->deterministic ? y.db_acc : nullptr;
  return 0;
}
static int wgrad_max_splits(const WgradParams& w) {
  int m = 1;
  for (int g = 0; g < w.n_groups; ++g) if (w.group_splits[g] > m) m = w.group_splits[g];
  return m;
}

extern "C" {

int nint_version(void) { return 100; }
const char* nint_last_error(void) { return g_err; }
int nint_gate_column(int q, int hidden) { return q_to_n(q, hidden); }
int nint_pick_tile(int height, int width, int* tile_w, int* tile_h) {
  if (height < 1 || width < 1 || !tile_w || !tile_h) return fail("nint_pick_tile: bad arguments");
  return pick_tile(height, width, tile_w, tile_h);
}

long long nint_launch_count(int kernel_class) {
  if (kernel_class < 0) return g_launches[0] + g_launches[1] + g_launches[2] + g_launches[3];
  return kernel_class < K_NCLS ? g_launches[kernel_class] : 0;
}

int nint_plan_profile(nint_plan* p, int enable) {
  if (!p) return fail("null plan");
  p->prof.on = enable != 0;
  p->prof.used = 0;
  return 0;
}

int nint_plan_profile_read(nint_plan* p, double* ms, long long* count) {
  if (!p || !ms || !count) return fail("nint_plan_profile_read: null argument");
  Profile& pr = p->prof;
  for (int c = 0; c < K_NCLS; ++c) ms[c] = 0.0, count[c] = 0;
  for (size_t i = 0; i < pr.used; ++i) {
    CK(cudaEventSynchronize(pr.pool[2 * i + 1]));
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, pr.pool[2 * i], pr.pool[2 * i + 1]));
    ms[pr.cls[i]] += t;
    count[pr.cls[i]] += pr.weight[i];
  }
  pr.used = 0;
  return 0;
}

int nint_plan_create(const nint_config* cfg, nint_plan** out) {
  if (!cfg || !out) return fail("nint_plan_create: null argument");
  if (cfg->num_layers < 1 || cfg->num_layers > NINT_MAX_LAYERS)
    return fail("num_layers must be in [1,%d], got %d", NINT_MAX_LAYERS, cfg->num_layers);
  if (cfg->batch < 1 || cfg->seq_len < 1 || cfg->height < 1 || cfg->width < 1 || cfg->in_channels < 1)
    return fail("batch/seq_len/height/width/in_channels must be positive");
  if (cfg->dtype != BF16 && cfg->dtype != TF32) return fail("unknown dtype %d", cfg->dtype);
  nint_plan* p = new (std::nothrow) nint_plan();
  if (!p) return fail("out of host memory");
  p->cfg = *cfg;
  p->L = cfg->num_layers; p->B = cfg->batch; p->T = cfg->seq_len; p->H = cfg->height; p->W = cfg->width;
  p->dtype = cfg->dtype;
  p->esize = cfg->dtype == BF16 ? 2 : 4;
  p->ce = 64 / p->esize;
  p->deterministic = (cfg->flags & NINT_FLAG_DETERMINISTIC) != 0;
  p->input_grad = (cfg->flags & NINT_FLAG_INPUT_GRAD) != 0;
  p->state_grad = (cfg->flags & NINT_FLAG_STATE_GRAD) != 0;
  p->second_order = (cfg->flags & NINT_FLAG_SECOND_ORDER) != 0;
  p->param_tangent = (cfg->flags & NINT_FLAG_PARAM_TANGENT) != 0;
  p->hist = p->param_tangent && p->second_order && cfg->training;
  p->tangent = (cfg->flags & NINT_FLAG_TANGENT) != 0 || p->second_order || p->param_tangent;
  {  // debug / A-B knobs (documented in DESIGN.md): CTA pairs on/off, experiment flags
    const char* c = getenv("NINT_CLUSTER");
    p->cluster = c ? atoi(c) : 2;
    if (p->cluster != 1 && p->cluster != 2) p->cluster = 1;
    const char* d = getenv("NINT_DEBUG_FLAGS");
    p->debug_flags = d ? atoi(d) : 0;
    // bits other than 512 (host side: no bias folding) are kernel experiment knobs, compiled in only with -DNINT_KNOBS=1
    if (!NINT_KNOBS && (p->debug_flags & ~512)) {
      const int flags = p->debug_flags;
      delete p;
      return fail("NINT_DEBUG_FLAGS=%d needs the experiment build of the library (python -m nasa_niswan_b200.build --knobs, "
                  "then NINT_LIB=<...>/libnint_knobs.so): the product build compiles the kernel knobs out", flags);
    }
    const char* pg = getenv("NINT_PLAN_G");
    p->plan_g = pg ? atoi(pg) : 0;
    const char* pn = getenv("NINT_PLAN_NS");
    p->plan_ns = pn ? atoi(pn) : 0;
    if (const char* e = getenv("NINT_DETERMINISTIC")) p->deterministic = p->deterministic || atoi(e) != 0;
    const char* pd = getenv("NINT_PDL");
    p->pdl = pd ? (atoi(pd) != 0) : 0;   // off by default (see nint_plan::pdl)
    if (const char* e = getenv("NINT_FUSE_STEPS")) p->fuse_steps = atoi(e);   // bit 0: forward, bit 1: backward
    const char* sb = getenv("NINT_SUB_BATCH");
    p->sub_batch = sb ? atoi(sb) : 0;
    if (p->sub_batch < 0 || p->sub_batch >= p->B) p->sub_batch = 0;
  }
  pick_tile(p->H, p->W, &p->tile_w, &p->tile_h);
  p->tiles_x = (p->W + p->tile_w - 1) / p->tile_w;
  p->tiles_y = (p->H + p->tile_h - 1) / p->tile_h;
  int cin = cfg->in_channels, below_hc = 0;
  for (int l = 0; l < p->L; ++l) {
    Layer& y = p->layer[l];
    y.cin = cin; y.hc_real = cfg->hidden[l]; y.k = cfg->ksize[l]; y.taps = y.k * y.k;
    if (y.hc_real < 1 || y.hc_real > 256) {
      delete p;
      return fail("hidden_channels[%d] = %d unsupported (1 .. 256)", l, cfg->hidden[l]);
    }
    // any hidden size runs padded to the kernels' granularity (a multiple of 16, of 64 above 64): the padding channels
    // get zero weights and biases, so their c and h stay exactly zero and nothing downstream sees them (model.py:207)
    y.hc = y.hc_real <= 64 ? (y.hc_real + 15) / 16 * 16 : (y.hc_real + 63) / 64 * 64;
    if (y.k < 1 || y.k % 2 == 0 || y.k > 15) {
      delete p;
      return fail("kernel_size[%d] = %d unsupported (odd, <= 15)", l, y.k);
    }
    if (l > 0 && cin > 256) { delete p; return fail("layer %d input channels %d > 256", l, cin); }
    // x segment: layer 0 reads X (cin channels padded to 32); layer l > 0 reads the whole padded h tensor of the layer below
    y.cx_pad = l == 0 ? (y.cin + 31) / 32 * 32 : (below_hc + 31) / 32 * 32;
    y.chx = y.cx_pad / p->ce;
    y.hc_pad = (y.hc + 31) / 32 * 32;  y.chh = y.hc_pad / p->ce;
    y.cin_rows = l == 0 ? y.cx_pad : below_hc;
    // a spare padding channel of X carries 1.0: the packed forward weights are zero there (no effect on the cell),
    // and the weight-gradient GEMM then produces the bias gradient in that column for free
    if (l == 0 && y.cx_pad > y.cin && !(p->debug_flags & 128)) p->ones_lane = y.cin;
    // forward N slice (n-block) = hcb hidden channels x 4 gates.  If the whole weight slice of an n-block
    // fits in shared memory next to the halo buffers and epilogue stages (<= 112 KiB per CTA of a pair), the
    // conv kernel keeps it resident and only activations stream: weight re-reads were ~55 % of the L2 -> SM
    // traffic of the forward cell and L2 sector throughput was its bound (profiles/).
    y.hcb = y.hc < 64 ? y.hc : 64;
    if (cfg->dtype == BF16) {
      bool fits = false;
      for (int cand = y.hcb; cand >= 32 && !fits; cand >>= 1) {
        const long long w_cta = static_cast<long long>(y.cx_pad / 32 + y.hc_pad / 32) * y.taps * (4 * cand / p->cluster) * 64;
        if (y.hc % cand == 0 && w_cta <= 112 * 1024) { y.hcb = cand; fits = true; }
      }
      // weights that have to stream (5x5 taps, wide layers): N = 128 with two pixel tiles sharing every weight stage
      // moves half the weight bytes per tile of N = 256 (measured: 5x5 forward 645 -> 328 us, cfg 5 352 -> 314 ms)
      if (!fits && y.hc >= 32 && y.hc % 32 == 0) y.hcb = 32;
    }
    if (const char* e = getenv("NINT_HCB")) {   // experiment knob: force the forward n-block width (16 / 32 / 64)
      const int v = atoi(e);
      if (v >= 16 && v <= 64 && (v & (v - 1)) == 0 && y.hc % v == 0) y.hcb = v;
    }
    y.n_blocks = y.hc / y.hcb; y.n_tile = 4 * y.hcb;
    y.nslots_h = cfg->training ? p->T + 1 : 2;
    y.nslots_c = cfg->training ? p->T + 1 : 1;
    y.ncols = y.cx_pad + y.hc_pad;
    if (cfg->training && plan_wgrad_blocks(p, y)) {
      const int hc = y.hc, k = y.k;
      delete p;
      return fail("layer %d: training with hidden %d, kernel %d: not even one 32-channel wgrad operand panel fits in "
                  "shared memory", l, hc, k);
    }
    if (cfg->training && p->deterministic) {
      // partial-sum slices of the deterministic weight gradient: as many as the widest split-K of any column block
      // on a 148-SM part (checked again at launch against the real device)
      y.det_splits = 1;
      for (size_t bi = 0; bi < y.wg_blocks.size(); ++bi) {
        WgradParams w;
        if (wgrad_params(p, l, bi, 148, w)) { delete p; return 1; }
        if (wgrad_max_splits(w) > y.det_splits) y.det_splits = wgrad_max_splits(w);
      }
    }
    cin = y.hc_real;
    below_hc = y.hc;
  }
  if (p->input_grad && cfg->training && p->layer[0].cin_rows > 256) {
    delete p;
    return fail("input gradient: %d input channels exceed one MMA N (256)", cfg->in_channels);
  }
  // (layer l >= 1 reads the h tensor of layer l-1 as its x segment: ceil(hc_{l-1}/ce) chunks on both sides)
  p->ws_bytes = carve(p, nullptr);
  *out = p;
  return 0;
}

void nint_plan_destroy(nint_plan* plan) {
  if (!plan) return;
  for (cudaEvent_t e : plan->prof.pool) cudaEventDestroy(e);
  delete plan;
}

size_t nint_plan_workspace_bytes(const nint_plan* plan) { return plan ? plan->ws_bytes : 0; }

int nint_plan_input_layout(const nint_plan* plan, int* c_pad, int* ones_lane, int* elem_bytes) {
  if (!plan) return fail("null plan");
  if (c_pad) *c_pad = plan->layer[0].cx_pad;
  if (ones_lane) *ones_lane = plan->ones_lane;
  if (elem_bytes) *elem_bytes = plan->esize;
  return 0;
}

// tensor maps over an input tensor [images][H][W][cx_pad0] x `slots`: conv view, wgrad view, CTA-pair wgrad view
static int encode_input_maps(nint_plan* p, void* base, long long images, int slots, CUtensorMap* conv, CUtensorMap* wg,
                             CUtensorMap* wg_pair) {
  const int tw = p->tile_w, th = p->tile_h, ce = p->ce, pad0 = p->layer[0].k / 2;
  Layer& y = p->layer[0];
  if (images > 0x7fffffffLL) return fail("too many frames (%lld)", images);
  const int n = static_cast<int>(images);
  if (encode_act_map(conv, p->dtype, base, y.cx_pad, p->W, p->H, n, slots, ce, tw, th, false, pad0)) return 1;
  if (encode_act_map(wg, p->dtype, base, y.cx_pad, p->W, p->H, n, slots, ce, tw, th, true, pad0)) return 1;
  if (p->cfg.training && p->dtype == BF16)
    for (const Layer::WgBlock& b : y.wg_blocks) {
      if (!b.pair || b.nch_x == 0) continue;
      const CUtensorMapSwizzle sw = b.pw == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (b.pw == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
      if (encode_act_box(wg_pair, p->dtype, base, y.cx_pad, p->W, p->H, n, slots, b.pw, tw, th, pad0, sw)) return 1;
    }
  return 0;
}

static CUtensorMapSwizzle pair_swizzle(int pw) {
  return pw == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (pw == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

// wgrad views of the parameter outputs (plans with both NINT_FLAG_PARAM_TANGENT and NINT_FLAG_SECOND_ORDER), the same box
// geometries as the ordinary wgrad's maps: the input tangent, the dh history and the pass's (a, da) history
static int encode_param_wgrad_maps(nint_plan* p) {
  const int tw = p->tile_w, th = p->tile_h, ce = p->ce, T = p->T, B = p->B;
  CUtensorMap conv;
  if (encode_input_maps(p, p->tX, B, T, &conv, &p->tmw_tX, &p->tmp_tX)) return 1;
  for (int l = 0; l < p->L; ++l) {
    Layer& y = p->layer[l];
    const int pad = y.k / 2;
    for (int v = 0; v < 2; ++v) {   // images [0, B) / [B, 2B) of every [2B] slot
      uint8_t* base = y.sA + act_bytes(p, v, 4 * y.hc);
      if (encode_act_map(&y.tmw_sA[v], p->dtype, base, 4 * y.hc, p->W, p->H, B, T, ce, tw, th, true, 0, 2LL * B)) return 1;
    }
    if (encode_act_map(&y.tmw_tH, p->dtype, y.tH, y.hc_pad, p->W, p->H, B, T + 1, ce, tw, th, true, pad)) return 1;
    if (l + 1 < p->L &&
        encode_act_map(&y.tmw_tH_up, p->dtype, y.tH, y.hc_pad, p->W, p->H, B, T + 1, ce, tw, th, true, p->layer[l + 1].k / 2))
      return 1;
    bool any_pair = false;
    for (const Layer::WgBlock& b : y.wg_blocks) {
      if (!b.pair || p->dtype != BF16) continue;
      any_pair = true;
      if (b.nch_h > 0 &&
          encode_act_box(&y.tmp_tH, p->dtype, y.tH, y.hc_pad, p->W, p->H, B, T + 1, b.pw, tw, th, pad, pair_swizzle(b.pw))) return 1;
      if (b.nch_x > 0 && l > 0) {
        Layer& dn = p->layer[l - 1];
        if (encode_act_box(&dn.tmp_tH_up, p->dtype, dn.tH, dn.hc_pad, p->W, p->H, B, T + 1, b.pw, tw, th, pad, pair_swizzle(b.pw))) return 1;
      }
    }
    for (int v = 0; v < 2 && any_pair; ++v)
      if (encode_act_box(&y.tmp_sA[v], p->dtype, y.sA + act_bytes(p, v, 4 * y.hc), 4 * y.hc, p->W, p->H, B, T, 64, tw, th, 0,
                         CU_TENSOR_MAP_SWIZZLE_128B, 2LL * B)) return 1;
  }
  return 0;
}

int nint_plan_bind(nint_plan* p, void* workspace, size_t bytes, void* stream) {
  if (!p || !workspace) return fail("nint_plan_bind: null argument");
  if (bytes < p->ws_bytes) return fail("workspace too small: %zu < %zu", bytes, p->ws_bytes);
  if (reinterpret_cast<uintptr_t>(workspace) % 256) return fail("workspace must be 256-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int dev = 0, sms = 0, cc_major = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CK(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, dev));
  if (cc_major != 10) return fail("libnint needs an sm_100 device (Blackwell B200); found compute capability %d.x", cc_major);
  p->num_sms = sms;
  p->ws = static_cast<uint8_t*>(workspace);
  carve(p, p->ws);
  CK(cudaMemsetAsync(p->ws, 0, p->ws_bytes, st));
  const int tw = p->tile_w, th = p->tile_h, ce = p->ce;
  auto pad_of = [&](int l) { return p->layer[l].k / 2; };
  if (encode_input_maps(p, p->X, p->B, p->T, &p->tm_X, &p->tmw_X, &p->tmp_X)) return 1;
  p->x_bank = false; p->bank_ptr = nullptr; p->bank_frames = 0; p->win_start = nullptr;
  for (int l = 0; l < p->L; ++l) {
    Layer& y = p->layer[l];
    for (auto& a : y.fwd_cache) for (auto& c : a) c.valid = false;
    for (auto& c : y.bwd_cache) c.valid = false;
    if (encode_act_map(&y.tm_H, p->dtype, y.Hs, y.hc_pad, p->W, p->H, p->B, y.nslots_h, ce, tw, th, false, pad_of(l))) return 1;
    if (l + 1 < p->L &&
        encode_act_map(&y.tm_H_up, p->dtype, y.Hs, y.hc_pad, p->W, p->H, p->B, y.nslots_h, ce, tw, th, false, pad_of(l + 1))) return 1;
    if (encode_io_map(&y.tme_C, true, y.Cs, y.hc, p->W, p->H, p->B, y.nslots_c, 16)) return 1;
    if (encode_io_map(&y.tme_H, p->dtype == TF32, y.Hs, y.hc_pad, p->W, p->H, p->B, y.nslots_h, 16)) return 1;
    if (p->cfg.training) {
      if (encode_io_map(&y.tme_G, p->dtype == TF32, y.G, 4 * y.hc, p->W, p->H, p->B, p->T, 128 / p->esize)) return 1;
      if (encode_io_map(&y.tme_dC, true, y.dC, y.hc, p->W, p->H, p->B, 1, 16)) return 1;
    } else {
      y.tme_G = y.tme_C;   // never dereferenced (slot_g < 0), but the kernel parameter must be a valid map
      y.tme_dC = y.tme_C;
    }
    for (auto& v : y.wmaps) v.clear();
    if (p->cfg.training) {
      if (encode_act_map(&y.tm_G, p->dtype, y.G, 4 * y.hc, p->W, p->H, p->B, p->T, ce, tw, th, false, pad_of(l))) return 1;
      if (encode_act_map(&y.tmw_G, p->dtype, y.G, 4 * y.hc, p->W, p->H, p->B, p->T, ce, tw, th, true)) return 1;
      if (encode_act_map(&y.tmw_H, p->dtype, y.Hs, y.hc_pad, p->W, p->H, p->B, y.nslots_h, ce, tw, th, true, pad_of(l))) return 1;
      if (l + 1 < p->L &&
          encode_act_map(&y.tmw_H_up, p->dtype, y.Hs, y.hc_pad, p->W, p->H, p->B, y.nslots_h, ce, tw, th, true, pad_of(l + 1))) return 1;
    }
  }
  if (p->cfg.training) {
    for (int l = 0; l < p->L; ++l) {
      Layer& y = p->layer[l];
      auto sw_of = [](int pw) {
        return pw == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (pw == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
      };
      bool any_pair = false;
      for (const Layer::WgBlock& b : y.wg_blocks) {
        if (!b.pair || p->dtype != BF16) continue;   // the tf32 pair kernel reads the 32-channel tmw_* maps
        any_pair = true;
        // a pair block covers whole tensors (the full row, or the x part / the h part), so one map per tensor
        if (b.nch_h > 0 &&
            encode_act_box(&y.tmp_H, p->dtype, y.Hs, y.hc_pad, p->W, p->H, p->B, y.nslots_h, b.pw, tw, th, pad_of(l), sw_of(b.pw))) return 1;
        if (b.nch_x > 0 && l > 0) {
          Layer& dn = p->layer[l - 1];
          if (encode_act_box(&dn.tmp_H_up, p->dtype, dn.Hs, dn.hc_pad, p->W, p->H, p->B, dn.nslots_h, b.pw, tw, th, pad_of(l), sw_of(b.pw))) return 1;
        }
      }
      if (any_pair &&
          encode_act_box(&y.tmp_G, p->dtype, y.G, 4 * y.hc, p->W, p->H, p->B, p->T, 64, tw, th, 0, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    }
  }
  if (p->cfg.training && p->tangent) {   // the tangent GEMM reads its operands through the forward's box geometry
    if (encode_act_map(&p->tm_tX, p->dtype, p->tX, p->layer[0].cx_pad, p->W, p->H, p->B, p->T, ce, tw, th, false, pad_of(0))) return 1;
    const int th_slots = p->hist ? p->T + 1 : 2;
    for (int l = 0; l < p->L; ++l) {
      Layer& y = p->layer[l];
      if (encode_act_map(&y.tm_tH, p->dtype, y.tH, y.hc_pad, p->W, p->H, p->B, th_slots, ce, tw, th, false, pad_of(l))) return 1;
      if (l + 1 < p->L &&
          encode_act_map(&y.tm_tH_up, p->dtype, y.tH, y.hc_pad, p->W, p->H, p->B, th_slots, ce, tw, th, false, pad_of(l + 1))) return 1;
    }
    if (p->hist && encode_param_wgrad_maps(p)) return 1;
    p->tbank_ptr = nullptr;
    p->tbank_frames = 0;
    for (int l = 0; l < p->L && p->second_order; ++l) {
      Layer& y = p->layer[l];
      if (encode_act_map(&y.tm_sA, p->dtype, y.sA, 4 * y.hc, p->W, p->H, 2 * p->B, p->hist ? p->T : 1, ce, tw, th, false, pad_of(l))) return 1;
    }
  }
  p->tangent_kept = false;
  p->param_in_tangent = false;
  p->soa_params = false;
  p->dhead_set = false;
  for (int l = 0; l < p->L; ++l) p->layer[l].dw_set = p->layer[l].dbias_add = false;
  p->zero_init = true;
  p->fwd_done = false;
  p->gates_valid = false;
  p->bptt_done = false;
  return 0;
}

int nint_plan_set_weights(nint_plan* p, int l, const float* weight, const float* bias, void* stream) {
  if (!p || !p->ws) return fail("plan not bound");
  if (l < 0 || l >= p->L) return fail("layer %d out of range", l);
  if (!weight) return fail("null weight");
  Layer& y = p->layer[l];
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // layer 0 with a constant-1 input lane: the bias becomes that lane's centre-tap weight and the epilogue adds nothing
  y.bias_folded = l == 0 && p->ones_lane >= 0 && bias != nullptr && !(p->debug_flags & 512);
  LAUNCH(p, K_OTHER, st, launch_pack_weights_fwd(p->dtype, weight, bias, y.wx, y.wh, y.bias_q, y.cin, y.hc_real, y.hc, y.hcb, y.k, y.cx_pad, y.hc_pad,
                                                 y.bias_folded ? p->ones_lane : -1, st));
  if (p->cfg.training) LAUNCH(p, K_OTHER, st, launch_pack_weights_bwd(p->dtype, weight, y.wdx, y.wdh, y.cin, y.cin_rows, y.hc_real, y.hc, y.k, st));
  y.weights_set = true;
  return 0;
}

int nint_plan_set_head(nint_plan* p, const float* weight, const float* bias, void* stream) {
  if (!p || !p->ws) return fail("plan not bound");
  if (!weight || !bias) return fail("null head parameter");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CK(cudaMemcpyAsync(p->head_w, weight, p->layer[p->L - 1].hc_real * 4, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(p->head_b, bias, 4, cudaMemcpyDeviceToDevice, st));
  p->head_set = true;
  return 0;
}

static int param_tangent_check(nint_plan* p, const char* what) {
  if (!p || !p->ws) return fail("plan not bound");
  if (!p->cfg.training || !p->param_tangent)
    return fail("%s needs a training plan created with NINT_FLAG_PARAM_TANGENT", what);
  // the second-order pass must linearise at the direction the tangent pass it follows used
  p->tangent_kept = false;
  p->soa_params = false;
  return 0;
}

int nint_plan_set_weight_tangent(nint_plan* p, int l, const float* dweight, const float* dbias, void* stream) {
  if (param_tangent_check(p, "nint_plan_set_weight_tangent")) return 1;
  if (l < 0 || l >= p->L) return fail("layer %d out of range", l);
  if (!dweight) return fail("nint_plan_set_weight_tangent: null weight tangent");
  Layer& y = p->layer[l];
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // layer 0 with a constant-1 input lane: dbias rides in the dW GEMM over the primal x, like the forward's bias
  const bool fold = l == 0 && p->ones_lane >= 0 && !(p->debug_flags & 512);
  LAUNCH(p, K_OTHER, st, launch_pack_weights_fwd(p->dtype, dweight, dbias, y.twx, y.twh, y.tbias_q, y.cin, y.hc_real, y.hc, y.hcb,
                                                 y.k, y.cx_pad, y.hc_pad, fold ? p->ones_lane : -1, st));
  if (p->hist)
    LAUNCH(p, K_OTHER, st, launch_pack_weights_bwd(p->dtype, dweight, y.twdx, y.twdh, y.cin, y.cin_rows, y.hc_real, y.hc, y.k, st));
  y.dw_set = true;
  y.dbias_add = dbias != nullptr && !fold;
  return 0;
}

int nint_plan_set_head_tangent(nint_plan* p, const float* dweight, const float* dbias, void* stream) {
  if (param_tangent_check(p, "nint_plan_set_head_tangent")) return 1;
  if (!dweight) return fail("nint_plan_set_head_tangent: null weight tangent");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CK(cudaMemcpyAsync(p->thead_w, dweight, p->layer[p->L - 1].hc_real * 4, cudaMemcpyDeviceToDevice, st));
  if (dbias) CK(cudaMemcpyAsync(p->thead_b, dbias, 4, cudaMemcpyDeviceToDevice, st));
  else CK(cudaMemsetAsync(p->thead_b, 0, 4, st));
  p->dhead_set = true;
  return 0;
}

int nint_plan_clear_param_tangent(nint_plan* p, void* stream) {
  (void)stream;
  if (param_tangent_check(p, "nint_plan_clear_param_tangent")) return 1;
  for (int l = 0; l < p->L; ++l) p->layer[l].dw_set = p->layer[l].dbias_add = false;
  p->dhead_set = false;
  return 0;
}

int nint_plan_reset_state(nint_plan* p, void* stream) {
  if (!p || !p->ws) return fail("plan not bound");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!p->zero_init) {
    for (int l = 0; l < p->L; ++l) {
      Layer& y = p->layer[l];
      CK(cudaMemsetAsync(y.Hs, 0, act_bytes(p, 1, y.hc_pad), st));
      CK(cudaMemsetAsync(y.Cs, 0, static_cast<size_t>(p->B) * p->H * p->W * y.hc * 4, st));
    }
  }
  p->zero_init = true;
  return 0;
}

int nint_plan_set_state(nint_plan* p, int l, const float* h, const float* c, void* stream) {
  if (!p || !p->ws) return fail("plan not bound");
  if (l < 0 || l >= p->L || !h || !c) return fail("nint_plan_set_state: bad arguments");
  Layer& y = p->layer[l];
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (p->zero_init) {
    // the other layers keep an explicit zero state in slot 0
    for (int j = 0; j < p->L; ++j) {
      Layer& z = p->layer[j];
      CK(cudaMemsetAsync(z.Hs, 0, act_bytes(p, 1, z.hc_pad), st));
      CK(cudaMemsetAsync(z.Cs, 0, static_cast<size_t>(p->B) * p->H * p->W * z.hc * 4, st));
    }
  }
  LAUNCH(p, K_OTHER, st, launch_pack_state(p->dtype, h, y.Hs, p->B, y.hc_real, p->H, p->W, y.hc_pad, st));
  LAUNCH(p, K_OTHER, st, launch_nchw_to_nhwc_f32(c, y.Cs, p->B, y.hc_real, p->H, p->W, y.hc, st));
  p->zero_init = false;
  return 0;
}

int nint_plan_get_state(nint_plan* p, int l, float* h, float* c, void* stream) {
  if (!p || !p->ws) return fail("plan not bound");
  if (l < 0 || l >= p->L) return fail("layer %d out of range", l);
  if (!p->fwd_done) return fail("nint_plan_get_state before nint_forward");
  Layer& y = p->layer[l];
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (h) LAUNCH(p, K_OTHER, st, launch_unpack_state(p->dtype, slot_ptr(p, y.Hs, p->final_slot_h, y.hc_pad), h, p->B, y.hc_real, p->H, p->W, y.hc_pad, st));
  if (c) LAUNCH(p, K_OTHER, st, launch_nhwc_to_nchw_f32(cslot_ptr(p, y, p->final_slot_c), c, p->B, y.hc_real, p->H, p->W, y.hc, st));
  return 0;
}

static int check_ready(nint_plan* p) {
  if (!p || !p->ws) return fail("plan not bound");
  for (int l = 0; l < p->L; ++l)
    if (!p->layer[l].weights_set) return fail("weights of layer %d not set", l);
  if (!p->head_set) return fail("head parameters not set");
  return 0;
}

// Time-fused forward launch of layer l?  NINT_FUSE_STEPS bit 0 forces it, 0 forbids it.  Automatic: for launches of at
// most 16 rounds of tile groups per cluster and step -- all three layers of the reference's recipe (7.6 / 7.6 / 15
// rounds: -1.3 % on top of the fused BPTT), cfg 2 at B=8 (11.7 rounds: -2 % on average, noisy); at 23 rounds (B=16) the
// gain is ~2 % and at 47 (B=32) nil, and with PDL the forward runs at its steady-state rate from start to end there.
static int fwd_should_fuse(nint_plan* p, int l, bool* fuse) {
  *fuse = false;
  if (p->fuse_steps == 0) return 0;
  if (p->fuse_steps > 0) {
    *fuse = (p->fuse_steps & 1) != 0;
    return 0;
  }
  ConvGemmParams g;
  if (fwd_conv_params(p, l, true, EPI_FWD, g)) return 1;
  const int per_group = g.cluster * g.group;
  const double groups = (static_cast<double>(p->B) * p->tiles_x * p->tiles_y + per_group - 1) / per_group;
  const int clusters = p->num_sms / (g.cluster * g.n_blocks);
  *fuse = clusters > 0 && groups / clusters <= 16.0;
  return 0;
}

// the T x L fused cell steps + head of ConvLSTM.forward once the input is in place (X packed, or the bank attached)
static int forward_steps(nint_plan* p, float* pred, float* seq, cudaStream_t st) {
  const bool tr = p->cfg.training != 0;
  const long long HW = static_cast<long long>(p->H) * p->W;
  const Layer& top = p->layer[p->L - 1];
  const size_t top_img = static_cast<size_t>(HW) * top.hc_pad * p->esize;   // bytes of one image of the top layer's h
  const int SB = p->sub_batch > 0 ? p->sub_batch : p->B;
  // time-fused schedule: layer by layer, all steps of a fused layer in ONE persistent launch (after the step that starts
  // from the zero state, whose GEMM has no h segment).  Layer-major order needs the whole h history of the layer
  // below, which a training plan keeps; an inference plan keeps two slots, so only a single layer fuses there
  bool fuse_l[NINT_MAX_LAYERS];
  bool any_fused = false;
  for (int l = 0; l < p->L; ++l) {
    fuse_l[l] = false;
    if (SB >= p->B && p->T > 1 && (tr || (p->L == 1 && !seq)) && fwd_should_fuse(p, l, &fuse_l[l])) return 1;
    any_fused = any_fused || fuse_l[l];
  }
  if (any_fused) {
    for (int l = 0; l < p->L; ++l) {          // model.py:267
      int t = 0;
      if (p->zero_init || !fuse_l[l]) {
        if (cell_step(p, l, 0, EPI_FWD, nullptr, st)) return 1;
        t = 1;
      }
      if (!fuse_l[l] || p->T - t == 1) {
        for (; t < p->T; ++t)                 // model.py:265
          if (cell_step(p, l, t, EPI_FWD, nullptr, st)) return 1;
      } else if (cell_step(p, l, t, EPI_FWD, nullptr, st, 0, 0, p->T - t)) return 1;
    }
    if (seq)
      for (int t = 0; t < p->T; ++t)          // model.py:272 (commented variant)
        LAUNCH(p, K_OTHER, st, launch_head_fwd(p->dtype, slot_ptr(p, top.Hs, t + 1, top.hc_pad), p->head_w, p->head_b,
                           seq + t * HW, HW, p->B, top.hc_real, top.hc_pad, p->T * HW, st));
  } else
  for (int b0 = 0; b0 < p->B; b0 += SB) {     // sub-batch-major: every slice runs all its steps while its state is in L2
    const int nb = b0 + SB <= p->B ? SB : p->B - b0;
    for (int t = 0; t < p->T; ++t) {          // model.py:265
      for (int l = 0; l < p->L; ++l)          // model.py:267
        if (cell_step(p, l, t, EPI_FWD, nullptr, st, b0, SB < p->B ? nb : 0)) return 1;
      if (seq) {                              // model.py:272 (commented variant)
        const int slot = tr ? t + 1 : ((t + 1) & 1);
        LAUNCH(p, K_OTHER, st, launch_head_fwd(p->dtype, slot_ptr(p, top.Hs, slot, top.hc_pad) + b0 * top_img, p->head_w, p->head_b,
                           seq + b0 * p->T * HW + t * HW, HW, nb, top.hc_real, top.hc_pad, p->T * HW, st));
      }
    }
  }
  p->final_slot_h = tr ? p->T : (p->T & 1);
  p->final_slot_c = tr ? p->T : 0;
  LAUNCH(p, K_OTHER, st, launch_head_fwd(p->dtype, slot_ptr(p, top.Hs, p->final_slot_h, top.hc_pad), p->head_w, p->head_b, pred, HW, p->B,
                     top.hc_real, top.hc_pad, HW, st));  // model.py:274
  p->fwd_done = true;
  p->gates_valid = tr;
  p->bptt_done = false;
  p->tangent_kept = false;
  p->soa_params = false;
  return 0;
}

int nint_forward_ex(nint_plan* p, const void* x, int x_dtype, float* pred, float* seq, void* stream) {
  if (check_ready(p)) return 1;
  if (!x || !pred) return fail("nint_forward: null x / pred");
  if (seq && !p->cfg.return_sequence) return fail("seq output requires return_sequence in the plan");
  if (x_dtype != NINT_X_FP32 && x_dtype != NINT_X_BF16) return fail("unknown x dtype %d", x_dtype);
  if (x_dtype == NINT_X_BF16 && p->dtype != BF16) return fail("bf16 inputs need a bf16 plan (a tf32 plan would lose input precision)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  p->x_bank = false;
  LAUNCH(p, K_OTHER, st, launch_pack_input(p->dtype, x, x_dtype == NINT_X_BF16, p->X, p->B, p->T, p->cfg.in_channels, p->H, p->W, p->layer[0].cx_pad, p->ones_lane, st));
  return forward_steps(p, pred, seq, st);
}

int nint_forward(nint_plan* p, const float* x, float* pred, float* seq, void* stream) {
  return nint_forward_ex(p, x, NINT_X_FP32, pred, seq, stream);
}

int nint_forward_bank(nint_plan* p, const void* bank, long long n_frames, const int* win_start, float* pred, float* seq,
                      void* stream) {
  if (check_ready(p)) return 1;
  if (!bank || !win_start || !pred) return fail("nint_forward_bank: null bank / win_start / pred");
  if (n_frames < p->T) return fail("nint_forward_bank: %lld frames cannot hold a window of %d steps", n_frames, p->T);
  if (reinterpret_cast<uintptr_t>(bank) % 128) return fail("the frame bank must be 128-byte aligned");
  if (seq && !p->cfg.return_sequence) return fail("seq output requires return_sequence in the plan");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (bank != p->bank_ptr || n_frames != p->bank_frames) {
    if (encode_input_maps(p, const_cast<void*>(bank), n_frames, 1, &p->tmb_X, &p->tmbw_X, &p->tmbp_X)) return 1;
    p->bank_ptr = bank;
    p->bank_frames = n_frames;
    for (auto& a : p->layer[0].fwd_cache) a[1].valid = false;
  }
  p->x_bank = true;
  p->win_start = win_start;
  return forward_steps(p, pred, seq, st);
}

int nint_pack_frames(int dtype, const void* frames, int x_dtype, long long n_frames, int channels, int height, int width,
                     int c_pad, int ones_lane, void* bank, void* stream) {
  if (!frames || !bank) return fail("nint_pack_frames: null argument");
  if (dtype != BF16 && dtype != TF32) return fail("unknown dtype %d", dtype);
  if (x_dtype != NINT_X_FP32 && x_dtype != NINT_X_BF16) return fail("unknown x dtype %d", x_dtype);
  if (n_frames < 1 || channels < 1 || height < 1 || width < 1) return fail("nint_pack_frames: bad shape");
  if (c_pad < channels || c_pad % 16) return fail("nint_pack_frames: c_pad %d must be a multiple of 16 and >= %d", c_pad, channels);
  if (ones_lane >= 0 && (ones_lane < channels || ones_lane >= c_pad)) return fail("nint_pack_frames: ones lane %d outside the padding lanes", ones_lane);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAUNCH(nullptr, K_OTHER, st, launch_pack_frames(dtype, frames, x_dtype == NINT_X_BF16, bank, n_frames, channels, height, width, c_pad, ones_lane, st));
  return 0;
}

static int check_fuse_args(const float* levels3d, const float* emis2d, const float* mean, const float* std,
                           const float* statics, int n_static, long long frames, int levels, int height, int width,
                           int padded_height, int padded_width, int mode, const void* out) {
  if ((!levels3d && levels > 0) || !emis2d || !mean || !std || !out) return fail("nint_fuse_inputs: null argument");
  if (n_static < 0 || (n_static > 0 && !statics)) return fail("nint_fuse_inputs: %d static fields but no data", n_static);
  if (frames < 1 || levels < 0 || height < 1 || width < 1) return fail("nint_fuse_inputs: bad shape");
  if (mode != 0 && mode != 1) return fail("nint_fuse_inputs: mode must be 0 (reflect) or 1 (reference RNN dataset)");
  const int left = (padded_width - width) / 2, right = padded_width - width - left;
  const int top = (padded_height - height) / 2, bot = padded_height - height - top;
  if (padded_width < width || padded_height < height) return fail("nint_fuse_inputs: padded size smaller than the grid");
  if (left > width || right > width)   // dataset.py:80
    return fail("The requested padding size is larger than width size of the input image.");
  if (top + 1 > height || bot + 1 > height)   // dataset.py:98
    return fail("The requested padding size is larger than height size of the input image.");
  return 0;
}

int nint_fuse_inputs(const float* levels3d, const float* emis2d, const float* mean, const float* std,
                     const float* statics, int n_static, long long frames, int levels, int height, int width,
                     int padded_height, int padded_width, int mode, float* out, void* stream) {
  if (check_fuse_args(levels3d, emis2d, mean, std, statics, n_static, frames, levels, height, width, padded_height, padded_width, mode, out)) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAUNCH(nullptr, K_OTHER, st, launch_fuse_inputs(levels3d, emis2d, mean, std, statics, n_static, out, frames, levels, height, width, padded_height, padded_width, mode, st));
  return 0;
}

int nint_fuse_inputs_bank(const float* levels3d, const float* emis2d, const float* mean, const float* std,
                          const float* statics, int n_static, long long frames, int levels, int height, int width,
                          int padded_height, int padded_width, int mode, int dtype, int c_pad, int ones_lane,
                          void* bank, void* stream) {
  if (check_fuse_args(levels3d, emis2d, mean, std, statics, n_static, frames, levels, height, width, padded_height, padded_width, mode, bank)) return 1;
  if (dtype != BF16 && dtype != TF32) return fail("unknown dtype %d", dtype);
  const int C = levels + 1 + n_static;
  if (c_pad < C || c_pad % 16 || c_pad > 64) return fail("nint_fuse_inputs_bank: c_pad %d must be a multiple of 16 in [%d, 64]", c_pad, C);
  if (ones_lane >= 0 && (ones_lane < C || ones_lane >= c_pad)) return fail("nint_fuse_inputs_bank: ones lane %d outside the padding lanes", ones_lane);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAUNCH(nullptr, K_OTHER, st, launch_fuse_inputs_bank(dtype, levels3d, emis2d, mean, std, statics, n_static, bank, frames, levels, height, width, padded_height, padded_width, mode, c_pad, ones_lane, st));
  return 0;
}

int nint_fuse_inputs_adjoint(const float* dframes, const float* std, long long frames, int levels, int n_static,
                             int height, int width, int padded_height, int padded_width, int mode, float* d_levels3d,
                             float* d_emis2d, float* d_statics, void* stream) {
  // same conditions as the forward: dframes stands in for its inputs and its output, std for mean and std
  if (check_fuse_args(levels > 0 ? dframes : nullptr, dframes, dframes, std, d_statics, d_statics ? n_static : 0, frames,
                      levels, height, width, padded_height, padded_width, mode, dframes)) return 1;
  if (n_static < 0) return fail("nint_fuse_inputs: %d static fields", n_static);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAUNCH(nullptr, K_OTHER, st, launch_fuse_inputs_adjoint(dframes, std, frames, levels, n_static, height, width, padded_height, padded_width, mode,
                                                          levels > 0 ? d_levels3d : nullptr, d_emis2d, n_static > 0 ? d_statics : nullptr, st));
  return 0;
}

static int check_loss_args(const float* pred, const float* y, const float* loss, const float* stats, int batch, int height,
                           int width, int crop_y0, int crop_y1, int crop_x0, int crop_x1) {
  if (!pred || !y || !loss || !stats) return fail("nint_loss_mse_l1: null argument");
  if (batch < 1 || height < 1 || width < 1) return fail("nint_loss_mse_l1: bad shape");
  if (crop_y0 < 0 || crop_y1 > height || crop_y0 >= crop_y1 || crop_x0 < 0 || crop_x1 > width || crop_x0 >= crop_x1)
    return fail("nint_loss_mse_l1: crop [%d:%d, %d:%d] outside %dx%d", crop_y0, crop_y1, crop_x0, crop_x1, height, width);
  return 0;
}

int nint_loss_mse_l1(const float* pred, const float* y, int batch, int height, int width, int crop_y0, int crop_y1,
                     int crop_x0, int crop_x1, float* dpred, float* loss, float* stats, void* stream) {
  if (check_loss_args(pred, y, loss, stats, batch, height, width, crop_y0, crop_y1, crop_x0, crop_x1)) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAUNCH(nullptr, K_OTHER, st, launch_loss_mse_l1(pred, y, dpred, stats, loss, batch, height, width, crop_y0, crop_y1, crop_x0, crop_x1, nullptr, 0, 0, st));
  return 0;
}

int nint_loss_mse_l1_bank(const float* pred, const float* ybank, long long n_frames, const int* win_start, int y_offset, int batch,
                          int height, int width, int crop_y0, int crop_y1, int crop_x0, int crop_x1, float* dpred,
                          float* loss, float* stats, void* stream) {
  if (check_loss_args(pred, ybank, loss, stats, batch, height, width, crop_y0, crop_y1, crop_x0, crop_x1)) return 1;
  if (!win_start || n_frames < 1) return fail("nint_loss_mse_l1_bank: null win_start / empty target bank");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAUNCH(nullptr, K_OTHER, st, launch_loss_mse_l1(pred, ybank, dpred, stats, loss, batch, height, width, crop_y0, crop_y1, crop_x0, crop_x1, win_start, y_offset, n_frames, st));
  return 0;
}

int nint_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                   float beta1, float beta2, float eps, int step, float grad_scale, void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq) return fail("nint_adam_step: null argument");
  if (n < 0 || step < 1) return fail("nint_adam_step: n >= 0 and step >= 1 required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAUNCH(nullptr, K_OTHER, st, launch_adam(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, grad_scale, st));
  return 0;
}

int nint_adam_step_dev(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float* state,
                       float beta1, float beta2, float eps, float grad_scale, void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq || !state) return fail("nint_adam_step_dev: null argument");
  if (n < 0) return fail("nint_adam_step_dev: n >= 0 required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAUNCH(nullptr, K_OTHER, st, launch_adam_dev(params, grads, exp_avg, exp_avg_sq, n, state, beta1, beta2, eps, grad_scale, st));
  ++g_launches[K_OTHER];   // two kernels: the step tick and the update
  return 0;
}

int nint_dp_allreduce_adam(const void* const* peer_buffers, long long slot_offset_bytes, long long flags_offset_bytes,
                           int rank, int world, unsigned seq, float* params, float* exp_avg, float* exp_avg_sq,
                           long long n, float* state, float beta1, float beta2, float eps, float grad_scale, void* stream) {
  if (!peer_buffers || !params || !exp_avg || !exp_avg_sq || !state) return fail("nint_dp_allreduce_adam: null argument");
  if (world < 1 || world > 16 || rank < 0 || rank >= world) return fail("nint_dp_allreduce_adam: rank %d of %d (at most 16 ranks)", rank, world);
  if (n < 0 || seq == 0) return fail("nint_dp_allreduce_adam: n >= 0 and seq >= 1 required");
  if (slot_offset_bytes % 16 || flags_offset_bytes % 16) return fail("nint_dp_allreduce_adam: offsets must be 16-byte aligned");
  for (int r = 0; r < world; ++r)
    if (!peer_buffers[r]) return fail("nint_dp_allreduce_adam: no mapping of rank %d's buffer", r);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LAUNCH(nullptr, K_OTHER, st, launch_dp_allreduce_adam(peer_buffers, slot_offset_bytes, flags_offset_bytes, rank, world, seq, params,
                                                        exp_avg, exp_avg_sq, n, state, beta1, beta2, eps, grad_scale, st));
  return 0;
}

int nint_debug_read_trace(long long* host, int n, int clear) {
  if (!host || n < 0) return fail("nint_debug_read_trace: bad arguments");
  CK(cudaDeviceSynchronize());
  CK(read_trace(host, n));
  if (clear) CK(clear_trace());
  return 0;
}

int nint_debug_fail_record(unsigned long long* out5) {
  if (!out5) return fail("nint_debug_fail_record: null argument");
  cudaError_t e = fail_record(out5);
  if (e != cudaSuccess) return fail("nint_debug_fail_record: %s", cudaGetErrorString(e));
  return 0;
}

int nint_debug_raw_gates(nint_plan* p, const float* x, float* out, void* stream) {
  if (check_ready(p)) return 1;
  if (!x || !out) return fail("nint_debug_raw_gates: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  p->x_bank = false;
  LAUNCH(p, K_OTHER, st, launch_pack_input(p->dtype, x, 0, p->X, p->B, p->T, p->cfg.in_channels, p->H, p->W, p->layer[0].cx_pad, p->ones_lane, st));
  return cell_step(p, 0, 0, EPI_RAW, out, st);
}

static bool resid_on(const nint_plan* p) {
  return p->num_sms <= kResidCtas && static_cast<long long>(p->B) * p->T * p->H * p->W <= kResidMaxPixelSteps;
}

// step-independent launch parameters of layer l's dgrad + gate-backward kernel (has_next: with a dgates_{t+1} segment)
static int bwd_conv_params(nint_plan* p, int l, bool has_next, ConvGemmParams& g) {
  const int L = p->L;
  Layer& y = p->layer[l];
  Layer::CachedConv& cache = y.bwd_cache[has_next ? 1 : 0];
  if (cache.valid) {
    g = cache.g;
  } else {
    fill_common(p, y, g);
    g.n_tile = y.hc;
    g.n_blocks = 1;
    g.cluster = bwd_cluster(p, l);
    g.idesc = idesc_of(p->dtype, 128 * g.cluster, y.hc, 0, 0);
    int s = 0;
    if (has_next) {  // dh_t += dgates_{t+1} (*) flip(W_h)
      g.seg[s].tmap_act = y.tm_G; g.seg[s].wsel = 3;
      g.seg[s].ksize = y.k; g.seg[s].nchunks = 4 * y.hc / p->ce;
      ++s;
    }
    if (l < L - 1) {  // dh_t += dx of the layer above at the same t
      Layer& up = p->layer[l + 1];
      g.seg[s].tmap_act = up.tm_G; g.seg[s].wsel = 2;
      g.seg[s].ksize = up.k; g.seg[s].nchunks = 4 * up.hc / p->ce;
      ++s;
    }
    g.nseg = s;
    // epilogue I/O: gates_t -> dgates_t in place, c_{t-1}, running dc in place (c_t is recomputed)
    g.tm_c = y.tme_C; g.tm_h = y.tme_H; g.tm_g = y.tme_G; g.tm_dc = y.tme_dC;
    g.slot_c_in = g.slot_c_out = g.slot_h_out = -1;
    if (conv_halo_plan(EPI_BWD, p->dtype, g)) return fail("layer %d: the dgrad kernel's shared-memory plan does not fit (hidden %d, k %d)", l, y.hc, y.k);
    for (int i = 0; i < g.nseg; ++i) {
      Layer& owner = g.seg[i].wsel == 2 ? p->layer[l + 1] : y;   // wdx belongs to the layer above
      if (get_w_map(p, owner, g.seg[i].wsel, g.n_tile, g.n_tile / g.cluster, g.seg[i].ts, &g.seg[i].tmap_w)) return 1;
    }
    cache.g = g;
    cache.valid = true;
  }
  return 0;
}

// Time-fused BPTT launch (ConvGemmParams::n_steps) or one launch per step?  Fusing removes the pipeline drain and the
// tail imbalance of every launch; the fused kernel's steady state is a little slower (hand-off polling, storers waiting
// for write completion).  Measured on B200 with the last build of round 2 (same box, alternating runs): it pays while a
// launch is short -- a CTA pair walks few tile groups per step: reference recipe (3.8 rounds) -5 %, cfg 2 at B=8 (2.9
// rounds) -5.7 %, B=16 (5.8) -2.6 %, B=24 (8.8) -1 % -- and is neutral at 11.7 rounds (B=32: +0.2 %).
// NINT_FUSE_STEPS bit 1 forces it, 0 forbids it.
static int bwd_should_fuse(nint_plan* p, int l, bool* fuse) {
  *fuse = false;
  const int SB = p->sub_batch > 0 ? p->sub_batch : p->B;
  if (SB < p->B || p->T <= 2 || p->fuse_steps == 0) return 0;
  if (p->fuse_steps > 0) {
    *fuse = (p->fuse_steps & 2) != 0;
    return 0;
  }
  ConvGemmParams g;
  if (bwd_conv_params(p, l, true, g)) return 1;
  const int per_group = g.cluster * g.group;
  const double groups = (static_cast<double>(p->B) * p->tiles_x * p->tiles_y + per_group - 1) / per_group;
  const int clusters = p->num_sms / g.cluster;
  *fuse = clusters > 0 && groups / clusters <= 10.0;
  return 0;
}

// upstream gradient of the final state, per layer: dh_ext[l] ([B][H][W][hc] fp32) is added to layer l's dh at t = T-1,
// dc_given[l] says that layer's running dc already holds dL/dc_T
struct StateGrad {
  const float* dh_ext[NINT_MAX_LAYERS] = {};
  bool dc_given[NINT_MAX_LAYERS] = {};
};

// one fused dgrad + gate-backward launch of layer l at step t for images [b0, b0 + nb) (nb = 0: all); n_steps > 1: steps
// t, t-1, .. t-n_steps+1 as ONE time-fused launch (t < T-1: all of them have a dgates_{t+1} segment and a running dc)
static int bwd_step(nint_plan* p, int l, int t, const float* dpred, const float* dseq, const StateGrad& sg,
                    cudaStream_t st, int b0, int nb, int n_steps = 1) {
  const long long HW = static_cast<long long>(p->H) * p->W;
  const int L = p->L, T = p->T;
  Layer& y = p->layer[l];
  const bool has_next = t < T - 1;
  ConvGemmParams g;
  if (bwd_conv_params(p, l, has_next, g)) return 1;
  int s = 0;
  if (has_next) g.seg[s++].slot = t + 1;
  if (l < L - 1) g.seg[s++].slot = t;
  g.slot_g = t;
  g.slot_c_prev = (t == 0 && p->zero_init) ? -1 : t;
  g.has_dc_in = (t == T - 1) ? (sg.dc_given[l] ? 1 : 0) : 1;
  g.head_dpred = nullptr; g.head_w = nullptr; g.head_dpred_bstride = 0;
  if (l == L - 1) {
    if (dseq) {
      // per-step head gradient; dpred (last step) is folded in by the caller adding it to dseq[:, T-1]
      g.head_dpred = dseq + t * HW;
      g.head_dpred_bstride = T * HW;
      g.head_w = p->head_w;
    } else if (t == T - 1 && dpred) {
      g.head_dpred = dpred;
      g.head_dpred_bstride = HW;
      g.head_w = p->head_w;
    }
  }
  g.dh_ext = t == T - 1 ? sg.dh_ext[l] : nullptr;
  g.db_resid = resid_on(p) ? y.db_resid : nullptr;
  set_batch_range(p, g, b0, nb);
  g.n_steps = 1;
  g.c_prev_none_step = -1;
  if (n_steps > 1) {
    if (!has_next || nb > 0 || t - n_steps + 1 < 0) return fail("internal: bad time-fused backward launch");
    g.d_seg[0] = g.d_seg[1] = g.d_g = g.d_c_prev = -1;
    g.ring_bits = 0;
    g.slot_c_prev = t;                                   // the zero initial state is a per-step property here
    g.c_prev_none_step = (p->zero_init && t - n_steps + 1 == 0) ? n_steps - 1 : -1;
    g.head_dpred_sstride = -HW;                          // dseq + (t - s) * HW
    if (arm_fused(p, g, n_steps, 2, st)) return 1;
  }
  LAUNCH(p, K_BWD, st, launch_conv_halo(EPI_BWD, p->dtype, g, p->num_sms, st));
  if (p->prof.on && p->prof.used > 0) p->prof.weight[p->prof.used - 1] = n_steps;
  return 0;
}

static int bptt_loop(nint_plan* p, const float* dpred, const float* dseq, const StateGrad& sg, cudaStream_t st) {
  // ---- BPTT: reverse time, top layer first.  The dgrad conv of step t+1 (and of the layer
  // above at step t) accumulates dh_t in TMEM; its epilogue is the gate backward of step t and
  // overwrites the saved gates with dgates in place.
  const int SB = p->sub_batch > 0 ? p->sub_batch : p->B;
  for (int l = 0; l < p->L; ++l)
    if (p->layer[l].db_resid) CK(cudaMemsetAsync(p->layer[l].db_resid, 0, static_cast<size_t>(kResidCtas) * 4 * 4 * p->layer[l].hc * 4, st));
  bool any_fused = false;
  bool fuse_l[NINT_MAX_LAYERS];
  for (int l = 0; l < p->L; ++l) {
    if (bwd_should_fuse(p, l, &fuse_l[l])) return 1;
    any_fused = any_fused || fuse_l[l];
  }
  if (any_fused) {
    // layer-major schedule: top layer first; layer l reads the dgates of layer l+1 at the same t, all in place by then.
    // A fused layer runs its steps T-2 .. 0 as ONE persistent launch after its step T-1 (which has no dgates_{t+1}
    // segment); the others one launch per step
    for (int l = p->L - 1; l >= 0; --l) {
      if (bwd_step(p, l, p->T - 1, dpred, dseq, sg, st, 0, 0)) return 1;
      if (fuse_l[l]) {
        if (bwd_step(p, l, p->T - 2, dpred, dseq, sg, st, 0, 0, p->T - 1)) return 1;
      } else {
        for (int t = p->T - 2; t >= 0; --t)
          if (bwd_step(p, l, t, dpred, dseq, sg, st, 0, 0)) return 1;
      }
    }
  } else
  for (int b0 = 0; b0 < p->B; b0 += SB) {
    const int nb = b0 + SB <= p->B ? SB : p->B - b0;
    for (int t = p->T - 1; t >= 0; --t)
      for (int l = p->L - 1; l >= 0; --l)
        if (bwd_step(p, l, t, dpred, dseq, sg, st, b0, SB < p->B ? nb : 0)) return 1;
  }
  p->gates_valid = false;
  p->bptt_done = true;
  return 0;
}

int nint_backward_bptt_state(nint_plan* p, const float* dpred, const float* dseq, const float* const* dh_T,
                             const float* const* dc_T, float* grad_head_weight, float* grad_head_bias, void* stream) {
  if (check_ready(p)) return 1;
  if (!p->cfg.training) return fail("nint_backward needs a training plan");
  if (!p->fwd_done) return fail("nint_backward before nint_forward");
  if (!p->gates_valid)
    return fail("nint_backward: the activations saved by the last forward were already consumed by a backward (BPTT "
                "turns the saved gates into their gradients in place); run the forward again");
  bool state_in = false;
  for (int l = 0; l < p->L; ++l) state_in = state_in || (dh_T && dh_T[l]) || (dc_T && dc_T[l]);
  if (state_in && !p->state_grad)
    return fail("nint_backward: gradients of the final state need a training plan created with NINT_FLAG_STATE_GRAD");
  if (!dpred && !dseq && !state_in) return fail("nint_backward: no upstream gradient");
  if (dseq && !p->cfg.return_sequence) return fail("dseq requires return_sequence in the plan");
  if (dseq && dpred) return fail("pass either dpred or dseq (fold dpred into dseq[:, T-1])");
  p->bptt_done = false;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long HW = static_cast<long long>(p->H) * p->W;
  const int L = p->L, T = p->T;
  const Layer& top = p->layer[L - 1];
  // ---- final-state gradients: dL/dh_T joins layer l's dh at T-1 (next to the head term), dL/dc_T starts its running dc
  StateGrad sg;
  for (int l = 0; l < L && state_in; ++l) {
    Layer& y = p->layer[l];
    if (dh_T && dh_T[l]) {
      LAUNCH(p, K_OTHER, st, launch_nchw_to_nhwc_f32(dh_T[l], y.dh_ext, p->B, y.hc_real, p->H, p->W, y.hc, st));
      sg.dh_ext[l] = y.dh_ext;   // padding channels stay zero from nint_plan_bind
    }
    if (dc_T && dc_T[l]) {
      CK(cudaMemsetAsync(y.dC, 0, static_cast<size_t>(p->B) * HW * y.hc * 4, st));
      LAUNCH(p, K_OTHER, st, launch_nchw_to_nhwc_f32(dc_T[l], y.dC, p->B, y.hc_real, p->H, p->W, y.hc, st));
      sg.dc_given[l] = true;
    }
  }
  // ---- head gradients (model.py:274): dw = sum dpred * h_T, db = sum dpred
  if (grad_head_weight && grad_head_bias) {
    CK(cudaMemsetAsync(grad_head_weight, 0, top.hc_real * 4, st));
    CK(cudaMemsetAsync(grad_head_bias, 0, 4, st));
    if (dpred)
      LAUNCH(p, K_OTHER, st, launch_head_bwd(p->dtype, slot_ptr(p, top.Hs, T, top.hc_pad), dpred, HW, grad_head_weight, grad_head_bias, HW,
                         p->B, top.hc_real, top.hc_pad, p->head_part, st));
    if (dseq)
      for (int t = 0; t < T; ++t)
        LAUNCH(p, K_OTHER, st, launch_head_bwd(p->dtype, slot_ptr(p, top.Hs, t + 1, top.hc_pad), dseq + t * HW, T * HW, grad_head_weight,
                           grad_head_bias, HW, p->B, top.hc_real, top.hc_pad, p->head_part, st));
  }
  return bptt_loop(p, dpred, dseq, sg, st);
}

int nint_backward_bptt(nint_plan* p, const float* dpred, const float* dseq, float* grad_head_weight,
                       float* grad_head_bias, void* stream) {
  return nint_backward_bptt_state(p, dpred, dseq, nullptr, nullptr, grad_head_weight, grad_head_bias, stream);
}

// dL/dh_{-1} and dL/dc_{-1} of every layer: h_{-1} only enters layer l's gate convolution at t = 0 (the layer above
// reads h_t for t >= 0), so dh0 = dgates_0 (*) flip(W_h); the running dc after step 0 is dc_0 * f_0 = dc0
int nint_backward_initial_state(nint_plan* p, float* const* dh0, float* const* dc0, void* stream) {
  if (check_ready(p)) return 1;
  if (!p->cfg.training || !p->state_grad)
    return fail("nint_backward_initial_state needs a training plan created with NINT_FLAG_STATE_GRAD");
  if (!p->bptt_done) return fail("nint_backward_initial_state before nint_backward_bptt");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long HW = static_cast<long long>(p->H) * p->W;
  for (int l = 0; l < p->L; ++l) {
    Layer& y = p->layer[l];
    if (dh0 && dh0[l]) {
      if (dgrad_raw(p, l, 0, 3, y.hc, p->raw, st)) return 1;
      LAUNCH(p, K_OTHER, st, launch_unpack_raw(p->raw, dh0[l], p->B, y.hc_real, p->H, p->W, y.hc, y.hc_real * HW, st));
    }
    if (dc0 && dc0[l]) LAUNCH(p, K_OTHER, st, launch_nhwc_to_nchw_f32(y.dC, dc0[l], p->B, y.hc_real, p->H, p->W, y.hc, st));
  }
  return 0;
}

// ---- weight / bias gradient of one layer, batched over all T steps (needs the dgates nint_backward_bptt left)
int nint_backward_wgrad(nint_plan* p, int l, float* grad_weight_l, float* grad_bias_l, void* stream) {
  if (check_ready(p)) return 1;
  if (!p->cfg.training) return fail("nint_backward_wgrad needs a training plan");
  if (!p->bptt_done) return fail("nint_backward_wgrad before nint_backward_bptt");
  if (l < 0 || l >= p->L) return fail("layer %d out of range", l);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Layer& y = p->layer[l];
  const size_t slices = p->deterministic ? static_cast<size_t>(y.det_splits) : 1;
  CK(cudaMemsetAsync(y.dw_acc, 0, y.dw_acc_bytes * slices, st));
  CK(cudaMemsetAsync(y.db_acc, 0, 4 * y.hc * 4 * slices, st));
  const int bias_col = (l == 0) ? p->ones_lane : -1;
  for (size_t bi = 0; bi < y.wg_blocks.size(); ++bi) {
    WgradParams w;
    if (wgrad_params(p, l, bi, p->num_sms, w)) return 1;
    if (p->deterministic && wgrad_max_splits(w) > y.det_splits)
      return fail("deterministic wgrad: this device splits the reduction %d ways, the plan reserved %d slices", wgrad_max_splits(w), y.det_splits);
    LAUNCH(p, K_WGRAD, st, launch_wgrad(p->dtype, w, st));
  }
  if (grad_weight_l)
    LAUNCH(p, K_OTHER, st, launch_unpack_wgrad(y.dw_acc, y.db_acc, grad_weight_l, grad_bias_l, y.cin, y.hc_real, y.hc, y.k, y.ncols, y.cx_pad,
                                               bias_col, 0, p->deterministic ? y.det_splits : 0,
                                               resid_on(p) ? y.db_resid : nullptr, kResidCtas * 4, st));
  return 0;
}

int nint_backward(nint_plan* p, const float* dpred, const float* dseq, float* const* grad_weight,
                  float* const* grad_bias, float* grad_head_weight, float* grad_head_bias, void* stream) {
  if (!grad_weight || !grad_bias) return fail("nint_backward: null gradient tables");
  if (nint_backward_bptt(p, dpred, dseq, grad_head_weight, grad_head_bias, stream)) return 1;
  for (int l = 0; l < p->L; ++l)
    if (nint_backward_wgrad(p, l, grad_weight[l], grad_bias[l], stream)) return 1;
  return 0;
}

// dx_t = dgates_t (of layer 0) (*) flip(W_x), all t: x.grad of the reference's autograd
int nint_backward_input(nint_plan* p, float* dx, void* stream) {
  if (check_ready(p)) return 1;
  if (!p->cfg.training || !p->input_grad) return fail("nint_backward_input needs a training plan created with NINT_FLAG_INPUT_GRAD");
  if (!p->bptt_done) return fail("nint_backward_input before nint_backward_bptt");
  if (!dx) return fail("nint_backward_input: null dx");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Layer& y = p->layer[0];
  const long long HW = static_cast<long long>(p->H) * p->W;
  const int C = p->cfg.in_channels;
  for (int t = 0; t < p->T; ++t) {
    if (dgrad_raw(p, 0, t, 2, y.cin_rows, p->raw, st)) return 1;
    LAUNCH(p, K_OTHER, st, launch_unpack_raw(p->raw, dx + t * C * HW, p->B, C, p->H, p->W, y.cin_rows, static_cast<long long>(p->T) * C * HW, st));
  }
  return 0;
}

// the same dx_t, added into the frames of the bank the last forward read: dframes[win_start[b] + t] += dx[b][t], in
// increasing t, then increasing b (nint.h)
int nint_backward_input_bank(nint_plan* p, float* dframes, void* stream) {
  if (check_ready(p)) return 1;
  if (!p->cfg.training || !p->input_grad)
    return fail("nint_backward_input_bank needs a training plan created with NINT_FLAG_INPUT_GRAD");
  if (!p->bptt_done) return fail("nint_backward_input_bank before nint_backward_bptt");
  if (!p->x_bank) return fail("nint_backward_input_bank: the last forward did not read a frame bank (nint_forward_bank)");
  if (!dframes) return fail("nint_backward_input_bank: null dframes");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Layer& y = p->layer[0];
  for (int t = 0; t < p->T; ++t) {
    if (dgrad_raw(p, 0, t, 2, y.cin_rows, p->raw, st)) return 1;
    LAUNCH(p, K_OTHER, st, launch_accum_frames(p->raw, dframes, p->win_start, p->B, p->cfg.in_channels, p->H, p->W, y.cin_rows, t, p->bank_frames, st));
  }
  return 0;
}

// ---- tangent-linear forward (nint.h nint_forward_tangent): reads the gates, c and h history of the last forward and
// writes only the NINT_FLAG_TANGENT buffers, so the forward stays available to further tangents and to one backward
static int tangent_check(nint_plan* p, bool bank, const float* dseq) {
  if (check_ready(p)) return 1;
  if (!p->cfg.training || !p->tangent)
    return fail("nint_forward_tangent needs a training plan created with NINT_FLAG_TANGENT");
  if (!p->fwd_done) return fail("nint_forward_tangent before nint_forward");
  if (!p->gates_valid)
    return fail("nint_forward_tangent: the gates saved by the last forward were already consumed by a backward (BPTT "
                "turns them into their gradients in place); run the forward again");
  if (bank && !p->x_bank) return fail("nint_forward_tangent_bank: the last forward did not read a frame bank (nint_forward_bank)");
  if (!bank && p->x_bank) return fail("nint_forward_tangent: the last forward read a frame bank; use nint_forward_tangent_bank");
  if (dseq && !p->cfg.return_sequence) return fail("dseq output requires return_sequence in the plan");
  return 0;
}

// the parameter direction's term of layer l's tangent gate GEMM at step t: dW (*) [x_t, h_{t-1}] over the forward's own
// operands (its slots, bank windows and zero-state rule, as cell_step reads them) through the packed dW panels, added
// into the dump `raw` that the tangent GEMM W (*) [dx_t, dh_{t-1}] wrote (EPI_RAW_ACC); on layer 0 with the constant-1
// lane the GEMM also adds dbias
static int param_tangent_gemm(nint_plan* p, int l, int t, float* raw, cudaStream_t st) {
  Layer& y = p->layer[l];
  const bool bank = l == 0 && p->x_bank;
  const bool have_state = !(t == 0 && p->zero_init);
  ConvGemmParams g;
  if (fwd_conv_params(p, l, have_state, EPI_RAW_ACC, g)) return 1;
  g.seg[0].slot = l == 0 ? t : t + 1;
  g.seg[0].win_start = bank ? p->win_start : nullptr;
  g.seg[0].bank_frames = bank ? static_cast<int>(p->bank_frames) : 0;
  if (have_state) g.seg[1].slot = t;
  for (int i = 0; i < g.nseg; ++i) {
    g.seg[i].wsel += 4;
    if (get_w_map(p, y, g.seg[i].wsel, g.n_tile, g.n_tile / g.cluster, g.seg[i].ts, &g.seg[i].tmap_w)) return 1;
  }
  g.slot_c_in = g.slot_c_out = g.slot_h_out = g.slot_g = g.slot_c_prev = -1;
  g.raw_out = raw;
  LAUNCH(p, K_FWD, st, launch_conv_halo(EPI_RAW_ACC, p->dtype, g, p->num_sms, st));
  return 0;
}

// slot of dh_{s-1} in tH: a 2-slot ring, or the history of plans with both parameter-tangent and second-order flags
inline int th_slot(const nint_plan* p, int s) { return p->hist ? s : (s & 1); }

// the T x L tangent steps once the input tangent is in place (tX packed, or the tangent bank's map encoded)
static int tangent_steps(nint_plan* p, const float* const* dh0, const float* const* dc0, float* dpred, float* dseq,
                         float* const* dh_T, float* const* dc_T, cudaStream_t st) {
  const long long HW = static_cast<long long>(p->H) * p->W;
  const long long npix = p->B * HW;
  const Layer& top = p->layer[p->L - 1];
  bool any_param = p->dhead_set;
  for (int l = 0; l < p->L; ++l) any_param = any_param || p->layer[l].dw_set;
  bool dh_in[NINT_MAX_LAYERS];
  for (int l = 0; l < p->L; ++l) {
    Layer& y = p->layer[l];
    dh_in[l] = dh0 && dh0[l];
    if (dh_in[l]) LAUNCH(p, K_OTHER, st, launch_pack_state(p->dtype, dh0[l], y.tH, p->B, y.hc_real, p->H, p->W, y.hc_pad, st));
    else if (p->hist) CK(cudaMemsetAsync(y.tH, 0, act_bytes(p, 1, y.hc_pad), st));   // dh0 = 0 is read by the params call
    CK(cudaMemsetAsync(y.tC, 0, static_cast<size_t>(npix) * y.hc * 4, st));
    if (dc0 && dc0[l]) LAUNCH(p, K_OTHER, st, launch_nchw_to_nhwc_f32(dc0[l], y.tC, p->B, y.hc_real, p->H, p->W, y.hc, st));
  }
  for (int t = 0; t < p->T; ++t) {
    for (int l = 0; l < p->L; ++l) {
      Layer& y = p->layer[l];
      const bool bank = l == 0 && p->x_bank;
      const bool rec = t > 0 || dh_in[l];   // dh_{-1} = 0 contributes nothing: no recurrent K segment
      // the forward's gate GEMM (its packed weights, halved i/f/o columns, shared-memory plan) over the tangent
      // operands; EPI_RAW dumps the accumulators and adds no bias, and the tangent input's constant-1 lane is 0
      ConvGemmParams g;
      if (fwd_conv_params(p, l, rec, EPI_RAW, g)) return 1;
      g.seg[0].tmap_act = l == 0 ? (bank ? p->tmb_tX : p->tm_tX) : p->layer[l - 1].tm_tH_up;
      g.seg[0].slot = l == 0 ? t : th_slot(p, t + 1);
      g.seg[0].win_start = bank ? p->win_start : nullptr;
      g.seg[0].bank_frames = bank ? static_cast<int>(p->tbank_frames) : 0;
      if (rec) {
        g.seg[1].tmap_act = y.tm_tH;
        g.seg[1].slot = th_slot(p, t);
      }
      g.slot_c_in = g.slot_c_out = g.slot_h_out = g.slot_g = g.slot_c_prev = -1;
      // second-order plans keep every step's dump and dc for nint_backward_second_order
      float* raw = p->second_order ? y.tR + static_cast<size_t>(t) * npix * 4 * y.hc : p->traw;
      g.raw_out = raw;
      LAUNCH(p, K_FWD, st, launch_conv_halo(EPI_RAW, p->dtype, g, p->num_sms, st));
      if (y.dw_set && param_tangent_gemm(p, l, t, raw, st)) return 1;
      LAUNCH(p, K_OTHER, st, launch_tangent_cell(p->dtype, raw, slot_ptr(p, y.G, t, 4 * y.hc), cslot_ptr(p, y, t),
                                                 cslot_ptr(p, y, t + 1), tc_slot(p, y, t), tc_slot(p, y, t + 1),
                                                 slot_ptr(p, y.tH, th_slot(p, t + 1), y.hc_pad), npix, y.hc, y.hc_pad, st,
                                                 y.dbias_add ? y.tbias_q : nullptr));
    }
    if (dseq) {
      const void* dh = slot_ptr(p, top.tH, th_slot(p, t + 1), top.hc_pad);
      if (p->dhead_set)
        LAUNCH(p, K_OTHER, st, launch_head_tangent(p->dtype, slot_ptr(p, top.Hs, t + 1, top.hc_pad), dh, p->head_w,
                                                   p->thead_w, p->thead_b, dseq + t * HW, HW, p->B, top.hc_real,
                                                   top.hc_pad, p->T * HW, st));
      else
        LAUNCH(p, K_OTHER, st, launch_head_fwd(p->dtype, dh, p->head_w, p->tzero, dseq + t * HW, HW, p->B, top.hc_real,
                                               top.hc_pad, p->T * HW, st));
    }
  }
  if (dpred) {
    const void* dh = slot_ptr(p, top.tH, th_slot(p, p->T), top.hc_pad);
    if (p->dhead_set)
      LAUNCH(p, K_OTHER, st, launch_head_tangent(p->dtype, slot_ptr(p, top.Hs, p->T, top.hc_pad), dh, p->head_w, p->thead_w,
                                                 p->thead_b, dpred, HW, p->B, top.hc_real, top.hc_pad, HW, st));
    else
      LAUNCH(p, K_OTHER, st, launch_head_fwd(p->dtype, dh, p->head_w, p->tzero, dpred, HW, p->B, top.hc_real, top.hc_pad,
                                             HW, st));
  }
  for (int l = 0; l < p->L; ++l) {
    const Layer& y = p->layer[l];
    if (dh_T && dh_T[l])
      LAUNCH(p, K_OTHER, st, launch_unpack_state(p->dtype, slot_ptr(p, y.tH, th_slot(p, p->T), y.hc_pad), dh_T[l], p->B, y.hc_real,
                                                 p->H, p->W, y.hc_pad, st));
    if (dc_T && dc_T[l])
      LAUNCH(p, K_OTHER, st, launch_nhwc_to_nchw_f32(tc_slot(p, y, p->T), dc_T[l], p->B, y.hc_real, p->H, p->W, y.hc, st));
  }
  p->tangent_kept = p->second_order;
  p->param_in_tangent = any_param;
  p->soa_params = false;
  return 0;
}

int nint_forward_tangent(nint_plan* p, const void* dx, int dx_dtype, const float* const* dh0, const float* const* dc0,
                         float* dpred, float* dseq, float* const* dh_T, float* const* dc_T, void* stream) {
  if (tangent_check(p, false, dseq)) return 1;
  if (dx && dx_dtype != NINT_X_FP32 && dx_dtype != NINT_X_BF16) return fail("unknown dx dtype %d", dx_dtype);
  if (dx && dx_dtype == NINT_X_BF16 && p->dtype != BF16) return fail("bf16 tangents need a bf16 plan");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Layer& y = p->layer[0];
  if (dx)
    LAUNCH(p, K_OTHER, st, launch_pack_input(p->dtype, dx, dx_dtype == NINT_X_BF16, p->tX, p->B, p->T, p->cfg.in_channels,
                                             p->H, p->W, y.cx_pad, -1, st));
  else
    CK(cudaMemsetAsync(p->tX, 0, act_bytes(p, p->T, y.cx_pad), st));
  return tangent_steps(p, dh0, dc0, dpred, dseq, dh_T, dc_T, st);
}

int nint_forward_tangent_bank(nint_plan* p, const void* dbank, long long n_frames, const float* const* dh0,
                              const float* const* dc0, float* dpred, float* dseq, float* const* dh_T,
                              float* const* dc_T, void* stream) {
  if (tangent_check(p, true, dseq)) return 1;
  if (!dbank) return fail("nint_forward_tangent_bank: null dbank");
  if (n_frames != p->bank_frames)
    return fail("nint_forward_tangent_bank: %lld tangent frames for a bank of %lld", n_frames, p->bank_frames);
  if (reinterpret_cast<uintptr_t>(dbank) % 128) return fail("the tangent frame bank must be 128-byte aligned");
  if (dbank != p->tbank_ptr || n_frames != p->tbank_frames) {
    if (p->hist) {   // the params call's wgrad reads the tangent frames too
      if (encode_input_maps(p, const_cast<void*>(dbank), n_frames, 1, &p->tmb_tX, &p->tmbw_tX, &p->tmbp_tX)) return 1;
    } else if (encode_act_map(&p->tmb_tX, p->dtype, const_cast<void*>(dbank), p->layer[0].cx_pad, p->W, p->H,
                              static_cast<int>(n_frames), 1, p->ce, p->tile_w, p->tile_h, false, p->layer[0].k / 2)) return 1;
    p->tbank_ptr = dbank;
    p->tbank_frames = n_frames;
  }
  return tangent_steps(p, dh0, dc0, dpred, dseq, dh_T, dc_T, static_cast<cudaStream_t>(stream));
}

// ---- second-order adjoint (nint.h nint_backward_second_order): reads the forward's gates, c and h history and the
// tangent pass's per-step dumps and dc, writes only the NINT_FLAG_SECOND_ORDER buffers and the caller's outputs
static int soa_check(nint_plan* p, bool bank, const float* dpred, const float* dseq, const float* ddpred,
                     const float* ddseq) {
  if (check_ready(p)) return 1;
  if (!p->cfg.training || !p->second_order)
    return fail("nint_backward_second_order needs a training plan created with NINT_FLAG_SECOND_ORDER");
  if (!p->fwd_done) return fail("nint_backward_second_order before nint_forward");
  if (!p->gates_valid)
    return fail("nint_backward_second_order: the gates saved by the last forward were already consumed by a backward "
                "(BPTT turns them into their gradients in place); run the forward again");
  if (!p->tangent_kept)
    return fail("nint_backward_second_order before nint_forward_tangent of the last forward (or the parameter direction "
                "changed since)");
  if (bank && !p->x_bank)
    return fail("nint_backward_second_order_bank: the last forward did not read a frame bank (nint_forward_bank)");
  if (!bank && p->x_bank)
    return fail("nint_backward_second_order: the last forward read a frame bank; use nint_backward_second_order_bank");
  if ((dseq || ddseq) && !p->cfg.return_sequence) return fail("dseq / ddseq require return_sequence in the plan");
  if ((dseq && dpred) || (ddseq && ddpred)) return fail("pass either dpred or dseq (fold dpred into dseq[:, T-1])");
  return 0;
}

// EPI_RAW dgrad over the pass's dgates of both kinds (2B images: primal, then tangent) into p->sraw [2][npix][n_rows]:
// segment i reads layer owner[i]'s dgates through its packed dgrad operand wsel[i] (2: x part, 3: h part) at step slot
// slot[i] of the history (slot 0 of the single step on plans without it).  dW = true: the parameter direction's
// dW^T terms instead -- operands 6 / 7 (dW's dgrad panels) over the PRIMAL dgates only (B images), added into the
// tangent half of the dump (EPI_RAW_ACC); layers without a direction are left out
static int soa_dgrad(nint_plan* p, int l, int n_rows, int nseg, const int* owner, const int* wsel, const int* slot,
                     bool dW, cudaStream_t st) {
  Layer& y = p->layer[l];
  ConvGemmParams g;
  fill_common(p, y, g);
  g.B = dW ? p->B : 2 * p->B;
  g.n_tile = n_rows;
  g.n_blocks = 1;
  g.cluster = (n_rows % 32 == 0) ? p->cluster : 1;
  g.idesc = idesc_of(p->dtype, 128 * g.cluster, n_rows, 0, 0);
  int n = 0;
  for (int i = 0; i < nseg; ++i) {
    const Layer& o = p->layer[owner[i]];
    if (dW && !o.dw_set) continue;
    g.seg[n].tmap_act = o.tm_sA; g.seg[n].wsel = wsel[i] + (dW ? 4 : 0); g.seg[n].slot = p->hist ? slot[i] : 0;
    g.seg[n].ksize = o.k; g.seg[n].nchunks = 4 * o.hc / p->ce;
    ++n;
  }
  if (n == 0) return 0;
  g.nseg = n;
  g.tm_c = y.tme_C; g.tm_h = y.tme_H; g.tm_g = y.tme_G; g.tm_dc = y.tme_dC;
  g.slot_g = g.slot_c_in = g.slot_c_out = g.slot_h_out = g.slot_c_prev = -1;
  g.raw_out = dW ? p->sraw + static_cast<size_t>(p->B) * p->H * p->W * n_rows : p->sraw;
  const int epi = dW ? EPI_RAW_ACC : EPI_RAW;
  if (conv_halo_plan(epi, p->dtype, g))
    return fail("layer %d: the second-order dgrad's shared-memory plan does not fit (N %d, k %d)", l, n_rows, y.k);
  int k = 0;
  for (int i = 0; i < nseg; ++i) {
    if (dW && !p->layer[owner[i]].dw_set) continue;
    if (get_w_map(p, p->layer[owner[i]], g.seg[k].wsel, g.n_tile, g.n_tile / g.cluster, g.seg[k].ts, &g.seg[k].tmap_w)) return 1;
    ++k;
  }
  LAUNCH(p, K_OTHER, st, launch_conv_halo(epi, p->dtype, g, p->num_sms, st));
  return 0;
}

// the primal and tangent dgrad of (a, da), then, when the tangent pass had a parameter direction, its dW^T terms
static int soa_dgrad_all(nint_plan* p, int l, int n_rows, int nseg, const int* owner, const int* wsel, const int* slot,
                         cudaStream_t st) {
  if (soa_dgrad(p, l, n_rows, nseg, owner, wsel, slot, false, st)) return 1;
  return p->param_in_tangent ? soa_dgrad(p, l, n_rows, nseg, owner, wsel, slot, true, st) : 0;
}

// the reverse loop once the checks passed: per step t (descending) and layer l (top first) eta = one dgrad, then
// soa_cell_kernel; layer 0's x part goes to dx / ddx (explicit windows) or is added into dframes / ddframes (bank).
// Plans with both parameter flags also reduce the head's parameter gradient and H v terms into p->head_sums.
static int soa_steps(nint_plan* p, const float* dpred, const float* dseq, const float* ddpred, const float* ddseq,
                     float* dx, float* ddx, float* dframes, float* ddframes, float* const* dh0, float* const* dc0,
                     float* const* ddh0, float* const* ddc0, cudaStream_t st) {
  const long long HW = static_cast<long long>(p->H) * p->W;
  const long long npix = p->B * HW;
  const int L = p->L, T = p->T, C = p->cfg.in_channels;
  const Layer& y0 = p->layer[0];
  const Layer& top = p->layer[L - 1];
  const long long xs = static_cast<long long>(npix) * y0.cin_rows;   // tangent half of a dx dump
  for (int l = 0; l < L; ++l) CK(cudaMemsetAsync(p->layer[l].sK, 0, 2 * static_cast<size_t>(npix) * p->layer[l].hc * 4, st));
  float* hs = p->head_sums;   // {grad w [hc], grad b, hvp w [hc], hvp b, scratch}
  float* hpart = p->deterministic ? p->head_part : nullptr;
  if (p->hist) CK(cudaMemsetAsync(hs, 0, static_cast<size_t>(2 * (top.hc + 1) + 1) * 4, st));
  for (int t = T - 1; t >= 0; --t) {
    for (int l = L - 1; l >= 0; --l) {
      Layer& y = p->layer[l];
      int owner[2], wsel[2], slot[2], n = 0;
      if (t < T - 1) { owner[n] = l; wsel[n] = 3; slot[n++] = t + 1; }       // dh_t += da_{t+1} (*) flip(W_h)
      if (l < L - 1) { owner[n] = l + 1; wsel[n] = 2; slot[n++] = t; }       // dh_t += the layer above's x part at t
      if (n && soa_dgrad_all(p, l, y.hc, n, owner, wsel, slot, st)) return 1;
      const float *u = nullptr, *du = nullptr;
      long long ub = 0, dub = 0;
      if (l == L - 1) {
        u = dseq ? dseq + t * HW : (t == T - 1 ? dpred : nullptr);
        du = ddseq ? ddseq + t * HW : (t == T - 1 ? ddpred : nullptr);
        ub = dseq ? T * HW : HW;
        dub = ddseq ? T * HW : HW;
      }
      uint8_t* da = p->hist ? slot_ptr(p, y.sA, 2 * t, 4 * y.hc) : y.sA;
      LAUNCH(p, K_OTHER, st, launch_soa_cell(p->dtype, n ? p->sraw : nullptr, u, ub, du, dub, p->head_w,
                                             slot_ptr(p, y.G, t, 4 * y.hc), y.tR + static_cast<size_t>(t) * npix * 4 * y.hc,
                                             cslot_ptr(p, y, t), cslot_ptr(p, y, t + 1), tc_slot(p, y, t),
                                             tc_slot(p, y, t + 1), y.sK, da, npix, HW, y.hc, st,
                                             p->dhead_set ? p->thead_w : nullptr));
      // head parameters: grad w += u h_t, grad b += u; H v: w += du h_t + u dh_t, b += du
      if (p->hist && l == L - 1) {
        const uint8_t* h = slot_ptr(p, top.Hs, t + 1, top.hc_pad);
        const uint8_t* dh = slot_ptr(p, top.tH, t + 1, top.hc_pad);
        float *gw = hs, *gb = hs + top.hc, *hw = hs + top.hc + 1, *hb = hs + 2 * top.hc + 1;
        if (u) {
          LAUNCH(p, K_OTHER, st, launch_head_bwd(p->dtype, h, u, ub, gw, gb, HW, p->B, top.hc_real, top.hc_pad, hpart, st));
          // u dh_t reaches only the weight: its bias sum goes to a scratch slot
          LAUNCH(p, K_OTHER, st, launch_head_bwd(p->dtype, dh, u, ub, hw, hb + 1, HW, p->B, top.hc_real, top.hc_pad, hpart, st));
        }
        if (du) LAUNCH(p, K_OTHER, st, launch_head_bwd(p->dtype, h, du, dub, hw, hb, HW, p->B, top.hc_real, top.hc_pad, hpart, st));
      }
    }
    if (dx || ddx || dframes || ddframes) {
      const int owner = 0, wsel = 2;
      if (soa_dgrad_all(p, 0, y0.cin_rows, 1, &owner, &wsel, &t, st)) return 1;
      const long long xstride = static_cast<long long>(T) * C * HW;
      if (dx) LAUNCH(p, K_OTHER, st, launch_unpack_raw(p->sraw, dx + t * C * HW, p->B, C, p->H, p->W, y0.cin_rows, xstride, st));
      if (ddx) LAUNCH(p, K_OTHER, st, launch_unpack_raw(p->sraw + xs, ddx + t * C * HW, p->B, C, p->H, p->W, y0.cin_rows, xstride, st));
      if (dframes)
        LAUNCH(p, K_OTHER, st, launch_accum_frames(p->sraw, dframes, p->win_start, p->B, C, p->H, p->W, y0.cin_rows, t,
                                                   p->bank_frames, st));
      if (ddframes)
        LAUNCH(p, K_OTHER, st, launch_accum_frames(p->sraw + xs, ddframes, p->win_start, p->B, C, p->H, p->W, y0.cin_rows, t,
                                                   p->bank_frames, st));
    }
  }
  // initial state: h_{-1} enters only layer l's gate GEMM at t = 0, so dh0 = da_0 (*) flip(W_h); dc0 = kappa after t = 0
  for (int l = 0; l < L; ++l) {
    Layer& y = p->layer[l];
    const long long hs_ = static_cast<long long>(npix) * y.hc;
    const bool h = dh0 && dh0[l], dh = ddh0 && ddh0[l];
    if (h || dh) {
      const int wsel = 3, slot = 0;
      if (soa_dgrad_all(p, l, y.hc, 1, &l, &wsel, &slot, st)) return 1;
      const long long bs = static_cast<long long>(y.hc_real) * HW;
      if (h) LAUNCH(p, K_OTHER, st, launch_unpack_raw(p->sraw, dh0[l], p->B, y.hc_real, p->H, p->W, y.hc, bs, st));
      if (dh) LAUNCH(p, K_OTHER, st, launch_unpack_raw(p->sraw + hs_, ddh0[l], p->B, y.hc_real, p->H, p->W, y.hc, bs, st));
    }
    if (dc0 && dc0[l]) LAUNCH(p, K_OTHER, st, launch_nhwc_to_nchw_f32(y.sK, dc0[l], p->B, y.hc_real, p->H, p->W, y.hc, st));
    if (ddc0 && ddc0[l])
      LAUNCH(p, K_OTHER, st, launch_nhwc_to_nchw_f32(y.sK + hs_, ddc0[l], p->B, y.hc_real, p->H, p->W, y.hc, st));
  }
  p->soa_params = p->hist;
  return 0;
}

int nint_backward_second_order(nint_plan* p, const float* dpred, const float* dseq, const float* ddpred,
                               const float* ddseq, float* dx, float* ddx, float* const* dh0, float* const* dc0,
                               float* const* ddh0, float* const* ddc0, void* stream) {
  if (soa_check(p, false, dpred, dseq, ddpred, ddseq)) return 1;
  return soa_steps(p, dpred, dseq, ddpred, ddseq, dx, ddx, nullptr, nullptr, dh0, dc0, ddh0, ddc0,
                   static_cast<cudaStream_t>(stream));
}

int nint_backward_second_order_bank(nint_plan* p, const float* dpred, const float* dseq, const float* ddpred,
                                    const float* ddseq, float* dframes, float* ddframes, float* const* dh0,
                                    float* const* dc0, float* const* ddh0, float* const* ddc0, void* stream) {
  if (soa_check(p, true, dpred, dseq, ddpred, ddseq)) return 1;
  return soa_steps(p, dpred, dseq, ddpred, ddseq, nullptr, nullptr, dframes, ddframes, dh0, dc0, ddh0, ddc0,
                   static_cast<cudaStream_t>(stream));
}

// one wgrad reduction of the parameter outputs over all T steps of layer l into gw / gb (accumulate: add):
// kind 0 = wgrad(a, comb) (the gradient), 1 = wgrad(da, comb), 2 = wgrad(a, dcomb) -- the ordinary wgrad's launches
// with the pass's (a, da) history as the dgates operand and, for kind 2, the input tangent and dh history as the
// activations.  Kind 2 has no bias term: the caller passes gb = NULL (its bias column / sum is not read)
static int param_wgrad(nint_plan* p, int l, int kind, float* gw, float* gb, int accumulate, cudaStream_t st) {
  Layer& y = p->layer[l];
  const size_t slices = p->deterministic ? static_cast<size_t>(y.det_splits) : 1;
  CK(cudaMemsetAsync(y.dw_acc, 0, y.dw_acc_bytes * slices, st));
  CK(cudaMemsetAsync(y.db_acc, 0, 4 * y.hc * 4 * slices, st));
  const bool bank = l == 0 && p->x_bank;
  for (size_t bi = 0; bi < y.wg_blocks.size(); ++bi) {
    WgradParams w;
    if (wgrad_params(p, l, bi, p->num_sms, w)) return 1;
    const Layer::WgBlock& blk = y.wg_blocks[bi];
    const bool pv = w.pair && p->dtype == BF16;   // CTA-pair boxes, else the 32-channel wgrad boxes
    w.tmap_dg = pv ? y.tmp_sA[kind == 1 ? 1 : 0] : y.tmw_sA[kind == 1 ? 1 : 0];
    if (kind == 2) {
      if (l == 0) w.tmap_b[0] = bank ? (pv ? p->tmbp_tX : p->tmbw_tX) : (pv ? p->tmp_tX : p->tmw_tX);
      else w.tmap_b[0] = pv ? p->layer[l - 1].tmp_tH_up : p->layer[l - 1].tmw_tH_up;
      w.tmap_b[1] = pv ? y.tmp_tH : y.tmw_tH;
      if (blk.nch_x == 0) w.tmap_b[0] = w.tmap_b[1];
      if (blk.nch_h == 0) w.tmap_b[1] = w.tmap_b[0];
    }
    if (p->deterministic && wgrad_max_splits(w) > y.det_splits)
      return fail("deterministic wgrad: this device splits the reduction %d ways, the plan reserved %d slices", wgrad_max_splits(w), y.det_splits);
    LAUNCH(p, K_WGRAD, st, launch_wgrad(p->dtype, w, st));
  }
  LAUNCH(p, K_OTHER, st, launch_unpack_wgrad(y.dw_acc, y.db_acc, gw, gb, y.cin, y.hc_real, y.hc, y.k, y.ncols, y.cx_pad,
                                             l == 0 ? p->ones_lane : -1, accumulate, p->deterministic ? y.det_splits : 0,
                                             nullptr, 0, st));
  return 0;
}

int nint_backward_second_order_params(nint_plan* p, float* const* grad_weight, float* const* grad_bias,
                                      float* const* hvp_weight, float* const* hvp_bias, float* grad_head_weight,
                                      float* grad_head_bias, float* hvp_head_weight, float* hvp_head_bias, void* stream) {
  if (check_ready(p)) return 1;
  if (!p->cfg.training || !p->hist)
    return fail("nint_backward_second_order_params needs a training plan created with NINT_FLAG_SECOND_ORDER | "
                "NINT_FLAG_PARAM_TANGENT");
  if (!p->gates_valid)
    return fail("nint_backward_second_order_params: the gates saved by the last forward were already consumed by a "
                "backward; run the forward again");
  if (!p->soa_params)
    return fail("nint_backward_second_order_params before nint_backward_second_order[_bank] of the current forward, "
                "tangent pass and parameter direction");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int l = 0; l < p->L; ++l) {
    if (grad_weight && grad_weight[l] && param_wgrad(p, l, 0, grad_weight[l], grad_bias ? grad_bias[l] : nullptr, 0, st))
      return 1;
    if (hvp_weight && hvp_weight[l]) {   // term 1, then term 2 added: a fixed order (deterministic plans stay bit-exact)
      if (param_wgrad(p, l, 1, hvp_weight[l], hvp_bias ? hvp_bias[l] : nullptr, 0, st)) return 1;
      if (param_wgrad(p, l, 2, hvp_weight[l], nullptr, 1, st)) return 1;
    }
  }
  const Layer& top = p->layer[p->L - 1];
  const float* hs = p->head_sums;
  const size_t hb = static_cast<size_t>(top.hc_real) * 4;
  if (grad_head_weight) CK(cudaMemcpyAsync(grad_head_weight, hs, hb, cudaMemcpyDeviceToDevice, st));
  if (grad_head_bias) CK(cudaMemcpyAsync(grad_head_bias, hs + top.hc, 4, cudaMemcpyDeviceToDevice, st));
  if (hvp_head_weight) CK(cudaMemcpyAsync(hvp_head_weight, hs + top.hc + 1, hb, cudaMemcpyDeviceToDevice, st));
  if (hvp_head_bias) CK(cudaMemcpyAsync(hvp_head_bias, hs + 2 * top.hc + 1, 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

int nint_cell_forward(nint_plan* p, const float* x, const float* h, const float* c, float* h_out, float* c_out,
                      void* stream) {
  if (check_ready(p)) return 1;
  if (p->L != 1 || p->T != 1) return fail("nint_cell_forward needs a plan with one layer and seq_len 1");
  if (!x || !h || !c) return fail("nint_cell_forward: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (nint_plan_set_state(p, 0, h, c, stream)) return 1;
  p->x_bank = false;
  LAUNCH(p, K_OTHER, st, launch_pack_input(p->dtype, x, 0, p->X, p->B, 1, p->cfg.in_channels, p->H, p->W, p->layer[0].cx_pad, p->ones_lane, st));
  if (cell_step(p, 0, 0, EPI_FWD, nullptr, st)) return 1;
  const bool tr = p->cfg.training != 0;
  p->final_slot_h = tr ? 1 : 1;
  p->final_slot_c = tr ? 1 : 0;
  p->fwd_done = true;
  p->gates_valid = tr;
  p->bptt_done = false;
  return nint_plan_get_state(p, 0, h_out, c_out, stream);
}

int nint_cell_backward(nint_plan* p, const float* dh_out, const float* dc_out, float* dx, float* dh, float* dc,
                       float* grad_weight, float* grad_bias, void* stream) {
  if (check_ready(p)) return 1;
  if (p->L != 1 || p->T != 1 || !p->cfg.training || !p->input_grad)
    return fail("nint_cell_backward needs a one-layer, seq_len 1 training plan created with NINT_FLAG_INPUT_GRAD");
  if (!p->fwd_done || !p->gates_valid) return fail("nint_cell_backward: no forward to differentiate (or already consumed)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Layer& y = p->layer[0];
  const size_t npix = static_cast<size_t>(p->B) * p->H * p->W;
  if (dh_out) LAUNCH(p, K_OTHER, st, launch_nchw_to_nhwc_f32(dh_out, p->dh_ext, p->B, y.hc_real, p->H, p->W, y.hc, st));
  if (dc_out) {
    CK(cudaMemsetAsync(y.dC, 0, npix * y.hc * 4, st));
    LAUNCH(p, K_OTHER, st, launch_nchw_to_nhwc_f32(dc_out, y.dC, p->B, y.hc_real, p->H, p->W, y.hc, st));
  }
  StateGrad sg;
  sg.dh_ext[0] = dh_out ? p->dh_ext : nullptr;
  sg.dc_given[0] = dc_out != nullptr;
  if (bptt_loop(p, nullptr, nullptr, sg, st)) return 1;
  if (dc) LAUNCH(p, K_OTHER, st, launch_nhwc_to_nchw_f32(y.dC, dc, p->B, y.hc_real, p->H, p->W, y.hc, st));
  if (dh) {
    if (dgrad_raw(p, 0, 0, 3, y.hc, p->raw, st)) return 1;
    LAUNCH(p, K_OTHER, st, launch_unpack_raw(p->raw, dh, p->B, y.hc_real, p->H, p->W, y.hc, static_cast<long long>(y.hc_real) * p->H * p->W, st));
  }
  if (dx) {
    const int C = p->cfg.in_channels;
    if (dgrad_raw(p, 0, 0, 2, y.cin_rows, p->raw, st)) return 1;
    LAUNCH(p, K_OTHER, st, launch_unpack_raw(p->raw, dx, p->B, C, p->H, p->W, y.cin_rows, static_cast<long long>(C) * p->H * p->W, st));
  }
  if (grad_weight || grad_bias) {
    if (!grad_weight) return fail("nint_cell_backward: grad_bias without grad_weight");
    if (nint_backward_wgrad(p, 0, grad_weight, grad_bias, stream)) return 1;
  }
  return 0;
}

}  // extern "C"
