// Memory-bound layout / pointwise kernels of the ConvLSTM path (sm_100a): input and state
// repacking between the reference's NCHW fp32 tensors and the channels-last operand layout,
// weight packing into UMMA panels, the 1x1 output head (model.py:251,274) and its backward,
// and the unpacking of the wgrad accumulators into OIHW gradients.
#include <type_traits>

#include "nint_common.cuh"
#include "nint_kernels.h"

namespace nint {

__device__ __forceinline__ float round_for(float v, __nv_bfloat16*) { return v; }
__device__ __forceinline__ float round_for(float v, float*) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
template <typename E>
__device__ __forceinline__ E to_elem(float v);
template <>
__device__ __forceinline__ __nv_bfloat16 to_elem<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <>
__device__ __forceinline__ float to_elem<float>(float v) { return round_for(v, (float*)nullptr); }
__device__ __forceinline__ float from_elem(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float from_elem(float v) { return v; }

// ------------------------------------------------------------------------------------------
// NCHW-like fp32 source -> channels-last E.  One thread per pixel: reads are coalesced across
// the warp (consecutive pixels of one channel plane), writes are CP*sizeof(E) contiguous bytes
// per thread, i.e. a warp writes one contiguous span.  src image stride / dst image index are
// given by the caller through (src_img_stride, dst slot mapping).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float ldg_f(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldg_f(const __nv_bfloat16* p) {
  return __uint_as_float(static_cast<uint32_t>(__ldg(reinterpret_cast<const unsigned short*>(p))) << 16);
}
// raw (unconverted) loads, so a kernel can issue a whole batch of them before touching any result
template <typename S> struct RawOf;
template <> struct RawOf<float> { using type = float; };
template <> struct RawOf<__nv_bfloat16> { using type = unsigned short; };
__device__ __forceinline__ float ldg_raw(const float* p) { return __ldg(p); }
__device__ __forceinline__ unsigned short ldg_raw(const __nv_bfloat16* p) { return __ldg(reinterpret_cast<const unsigned short*>(p)); }
__device__ __forceinline__ float raw_to_f(float v) { return v; }
__device__ __forceinline__ float raw_to_f(unsigned short v) { return __uint_as_float(static_cast<uint32_t>(v) << 16); }

// S = source element type: fp32 (the reference's tensors) or bf16 (host-staged windows: half the PCIe bytes)
template <typename S, typename E, int CP>
__global__ void pack_cl_kernel(const S* __restrict__ src, E* __restrict__ dst, int C, long long HW,
                               int n_outer, int n_inner, long long src_outer_stride, long long src_inner_stride,
                               long long dst_outer_stride, long long dst_inner_stride, int ones_lane) {
  // image (o, i): src + o*src_outer_stride + i*src_inner_stride, [C][HW];  dst + o*dst_outer + i*dst_inner, [HW][CP]
  const long long total = static_cast<long long>(n_outer) * n_inner * HW;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long pix = idx % HW;
    const long long img = idx / HW;
    const int i = static_cast<int>(img % n_inner);
    const int o = static_cast<int>(img / n_inner);
    const S* s = src + o * src_outer_stride + i * src_inner_stride + pix;
    E* d = dst + o * dst_outer_stride + i * dst_inner_stride + pix * CP;
    // all loads first, into their own registers, conversions after: a load followed at once by its conversion makes the
    // compiler recycle one register for every channel and the loads serialise on it (measured: the bf16-source variant
    // ran at 1.3 TB/s against 5.5 TB/s for the fp32 one, whose loads already were independent)
    // (2-byte sources: the loads are made unconditional -- padding lanes re-read channel C-1, an L1 hit -- so that no
    // per-channel branch splits the basic block and the scheduler can hoist every load above the first conversion)
    typename RawOf<S>::type raw[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) {
      if constexpr (sizeof(S) == 2) raw[c] = ldg_raw(s + (c < C ? c : C - 1) * HW);
      else raw[c] = (c < C) ? ldg_raw(s + c * HW) : typename RawOf<S>::type(0);
    }
    float v[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) v[c] = (c < C) ? round_for(raw_to_f(raw[c]), (E*)nullptr) : (c == ones_lane ? 1.f : 0.f);
    store_elems<E, CP>(d, v);
  }
}

template <typename S, typename E>
static cudaError_t pack_cl(const S* src, E* dst, int C, int c_pad, long long HW, int n_outer, int n_inner,
                           long long so, long long si, long long dso, long long dsi, int ones_lane, cudaStream_t s) {
  const long long total = static_cast<long long>(n_outer) * n_inner * HW;
  const int threads = 256;
  long long blocks = (total + threads - 1) / threads;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks <= 0) return cudaSuccess;
  switch (c_pad) {
    case 16: pack_cl_kernel<S, E, 16><<<blocks, threads, 0, s>>>(src, dst, C, HW, n_outer, n_inner, so, si, dso, dsi, ones_lane); break;
    case 32: pack_cl_kernel<S, E, 32><<<blocks, threads, 0, s>>>(src, dst, C, HW, n_outer, n_inner, so, si, dso, dsi, ones_lane); break;
    case 48: pack_cl_kernel<S, E, 48><<<blocks, threads, 0, s>>>(src, dst, C, HW, n_outer, n_inner, so, si, dso, dsi, ones_lane); break;
    case 64: pack_cl_kernel<S, E, 64><<<blocks, threads, 0, s>>>(src, dst, C, HW, n_outer, n_inner, so, si, dso, dsi, ones_lane); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// generic (any channel count) variant: one thread per (pixel, 16-channel group)
template <typename S, typename E>
__global__ void pack_cl_wide_kernel(const S* __restrict__ src, E* __restrict__ dst, int C, int c_pad,
                                    long long HW, int n_outer, int n_inner, long long so, long long si,
                                    long long dso, long long dsi, int ones_lane) {
  const int groups = c_pad / 16;
  const long long total = static_cast<long long>(n_outer) * n_inner * groups * HW;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long pix = idx % HW;
    long long r = idx / HW;
    const int g = static_cast<int>(r % groups);
    r /= groups;
    const int i = static_cast<int>(r % n_inner);
    const int o = static_cast<int>(r / n_inner);
    const S* s = src + o * so + i * si + pix;
    E* d = dst + o * dso + i * dsi + pix * c_pad + g * 16;
    float v[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const int ch = g * 16 + c;
      v[c] = (ch < C) ? round_for(ldg_f(s + ch * HW), (E*)nullptr) : (ch == ones_lane ? 1.f : 0.f);
    }
    store_elems<E, 16>(d, v);
  }
}

template <typename S, typename E>
static cudaError_t pack_any(const S* src, E* dst, int C, int c_pad, long long HW, int n_outer, int n_inner,
                            long long so, long long si, long long dso, long long dsi, cudaStream_t s, int ones_lane = -1) {
  if (c_pad % 16) return cudaErrorInvalidValue;
  if (c_pad <= 64) return pack_cl<S, E>(src, dst, C, c_pad, HW, n_outer, n_inner, so, si, dso, dsi, ones_lane, s);
  const long long total = static_cast<long long>(n_outer) * n_inner * (c_pad / 16) * HW;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks <= 0) return cudaSuccess;
  pack_cl_wide_kernel<S, E><<<blocks, 256, 0, s>>>(src, dst, C, c_pad, HW, n_outer, n_inner, so, si, dso, dsi, ones_lane);
  return cudaGetLastError();
}

template <typename S>
static cudaError_t pack_dispatch(int dtype, const S* src, void* dst, int C, int c_pad, long long HW, int n_outer, int n_inner,
                                 long long so, long long si, long long dso, long long dsi, int ones_lane, cudaStream_t s) {
  if (dtype == NINT_BF16)
    return pack_any<S, __nv_bfloat16>(src, reinterpret_cast<__nv_bfloat16*>(dst), C, c_pad, HW, n_outer, n_inner, so, si, dso, dsi, s, ones_lane);
  return pack_any<S, float>(src, reinterpret_cast<float*>(dst), C, c_pad, HW, n_outer, n_inner, so, si, dso, dsi, s, ones_lane);
}

cudaError_t launch_pack_input(int dtype, const void* x, int x_bf16, void* X, int B, int T, int C, int H, int W, int c_pad,
                              int ones_lane, cudaStream_t s) {
  // x[b][t] (model.py:266) -> X[t][b]: outer = b, inner = t
  const long long HW = static_cast<long long>(H) * W;
  const long long so = static_cast<long long>(T) * C * HW, si = C * HW;
  const long long dso = HW * c_pad, dsi = static_cast<long long>(B) * HW * c_pad;
  if (x_bf16) return pack_dispatch(dtype, reinterpret_cast<const __nv_bfloat16*>(x), X, C, c_pad, HW, B, T, so, si, dso, dsi, ones_lane, s);
  return pack_dispatch(dtype, reinterpret_cast<const float*>(x), X, C, c_pad, HW, B, T, so, si, dso, dsi, ones_lane, s);
}

// frames [N][C][H][W] (fp32 or bf16) -> bank [N][H][W][c_pad] E: the HBM-resident frame bank of nint_forward_bank
cudaError_t launch_pack_frames(int dtype, const void* src, int src_bf16, void* bank, long long N, int C, int H, int W,
                               int c_pad, int ones_lane, cudaStream_t s) {
  const long long HW = static_cast<long long>(H) * W;
  if (N > 0x7fffffffLL) return cudaErrorInvalidValue;
  if (src_bf16) return pack_dispatch(dtype, reinterpret_cast<const __nv_bfloat16*>(src), bank, C, c_pad, HW, static_cast<int>(N), 1, C * HW, 0, HW * c_pad, 0, ones_lane, s);
  return pack_dispatch(dtype, reinterpret_cast<const float*>(src), bank, C, c_pad, HW, static_cast<int>(N), 1, C * HW, 0, HW * c_pad, 0, ones_lane, s);
}

cudaError_t launch_pack_state(int dtype, const float* src, void* dst, int B, int C, int H, int W, int c_pad,
                              cudaStream_t s) {
  const long long HW = static_cast<long long>(H) * W;
  return pack_dispatch(dtype, src, dst, C, c_pad, HW, B, 1, C * HW, 0, HW * c_pad, 0, -1, s);
}

// channels-last E / fp32 -> NCHW fp32: tile transpose through shared memory (32 pixels x 32 channels)
template <typename E>
__global__ void unpack_cl_kernel(const E* __restrict__ src, float* __restrict__ dst, int C, int c_pad, long long HW,
                                 long long dst_bstride) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const long long p0 = static_cast<long long>(blockIdx.x) * 32;
  const int c0 = blockIdx.y * 32;
  const E* s = src + static_cast<long long>(b) * HW * c_pad;
  float* d = dst + static_cast<long long>(b) * dst_bstride;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const long long p = p0 + r;
    const int c = c0 + threadIdx.x;
    tile[r][threadIdx.x] = (p < HW && c < C) ? from_elem(s[p * c_pad + c]) : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int c = c0 + r;
    const long long p = p0 + threadIdx.x;
    if (c < C && p < HW) d[c * HW + p] = tile[threadIdx.x][r];
  }
}

cudaError_t launch_unpack_state(int dtype, const void* src, float* dst, int B, int C, int H, int W, int c_pad,
                                cudaStream_t s) {
  const long long HW = static_cast<long long>(H) * W;
  dim3 grid(static_cast<unsigned>((HW + 31) / 32), (C + 31) / 32, B), block(32, 8);
  if (dtype == NINT_BF16)
    unpack_cl_kernel<__nv_bfloat16><<<grid, block, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), dst, C, c_pad, HW, C * HW);
  else
    unpack_cl_kernel<float><<<grid, block, 0, s>>>(reinterpret_cast<const float*>(src), dst, C, c_pad, HW, C * HW);
  return cudaGetLastError();
}
cudaError_t launch_unpack_raw(const float* raw, float* dst, int B, int C, int H, int W, int ncols, long long dst_bstride,
                              cudaStream_t s) {
  const long long HW = static_cast<long long>(H) * W;
  dim3 grid(static_cast<unsigned>((HW + 31) / 32), (C + 31) / 32, B), block(32, 8);
  unpack_cl_kernel<float><<<grid, block, 0, s>>>(raw, dst, C, ncols, HW, dst_bstride);
  return cudaGetLastError();
}

// EPI_RAW dump of step t [B][HW][ncols] added into the frames the windows read, dframes[win_start[b] + t][C][HW].  A
// block owns 32 pixels x 32 channels of the frame tensor and walks the samples in groups of kAccGroup: the group's dump
// tiles are staged through shared memory (loads coalesced along the channels-last rows), then every thread adds them
// into its (channel, pixel) elements (coalesced along the pixels).  A thread owns its elements for every b, so repeated
// window starts need no atomics: the samples of a group that hit the same frame are summed into one register in
// increasing b (the frame's first sample of the group holds it), and the frame is read and written once per group.
constexpr int kAccGroup = 8;
__global__ void __launch_bounds__(256) accum_frames_kernel(const float* __restrict__ raw, float* __restrict__ dframes,
                                                           const int* __restrict__ win_start, int B, int C, int ncols,
                                                           long long HW, int t, long long n_frames) {
  __shared__ float tile[kAccGroup][32][33];
  __shared__ long long s_frame[kAccGroup];   // -1: no sample, or a frame outside the bank (skipped)
  __shared__ int s_root[kAccGroup];          // first sample of the group with the same frame (-1: skipped)
  const long long p0 = static_cast<long long>(blockIdx.x) * 32;
  const int c0 = blockIdx.y * 32;
  const int tid = threadIdx.y * 32 + threadIdx.x;
  for (int b0 = 0; b0 < B; b0 += kAccGroup) {
    const int nb = B - b0 < kAccGroup ? B - b0 : kAccGroup;
    if (tid < kAccGroup) {
      long long f = -1;
      if (tid < nb) {
        f = static_cast<long long>(__ldg(win_start + b0 + tid)) + t;
        if (f < 0 || f >= n_frames) f = -1;
      }
      s_frame[tid] = f;
    }
    for (int g = 0; g < nb; ++g) {
      const float* s = raw + static_cast<long long>(b0 + g) * HW * ncols;
      for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const long long p = p0 + r;
        const int c = c0 + threadIdx.x;
        tile[g][r][threadIdx.x] = (p < HW && c < C) ? __ldg(s + p * ncols + c) : 0.f;
      }
    }
    __syncthreads();
    if (tid < kAccGroup) {
      const long long f = s_frame[tid];
      int root = -1;
      if (f >= 0) {
        root = tid;
        for (int h = 0; h < tid; ++h)
          if (s_frame[h] == f) { root = h; break; }
      }
      s_root[tid] = root;
    }
    __syncthreads();
    const long long p = p0 + threadIdx.x;
#pragma unroll
    for (int r0 = 0; r0 < 32; r0 += 8) {
      const int r = r0 + threadIdx.y;
      const int c = c0 + r;
      if (c < C && p < HW) {
        float acc[kAccGroup];
#pragma unroll
        for (int g = 0; g < kAccGroup; ++g)
          acc[g] = s_root[g] == g ? dframes[(s_frame[g] * C + c) * HW + p] : 0.f;
#pragma unroll
        for (int g = 0; g < kAccGroup; ++g) {
          const float v = tile[g][threadIdx.x][r];
          const int root = s_root[g];
#pragma unroll
          for (int h = 0; h <= g; ++h)
            if (root == h) acc[h] += v;
        }
#pragma unroll
        for (int g = 0; g < kAccGroup; ++g)
          if (s_root[g] == g) dframes[(s_frame[g] * C + c) * HW + p] = acc[g];
      }
    }
    __syncthreads();
  }
}

cudaError_t launch_accum_frames(const float* raw, float* dframes, const int* win_start, int B, int C, int H, int W,
                                int ncols, int t, long long n_frames, cudaStream_t s) {
  const long long HW = static_cast<long long>(H) * W;
  dim3 grid(static_cast<unsigned>((HW + 31) / 32), (C + 31) / 32), block(32, 8);
  accum_frames_kernel<<<grid, block, 0, s>>>(raw, dframes, win_start, B, C, ncols, HW, t, n_frames);
  return cudaGetLastError();
}

__global__ void nchw_to_nhwc_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int c_pad, long long HW) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const long long p0 = static_cast<long long>(blockIdx.x) * 32;
  const int c0 = blockIdx.y * 32;
  const float* s = src + static_cast<long long>(b) * C * HW;
  float* d = dst + static_cast<long long>(b) * c_pad * HW;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int c = c0 + r;
    const long long p = p0 + threadIdx.x;
    tile[r][threadIdx.x] = (c < C && p < HW) ? s[c * HW + p] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const long long p = p0 + r;
    const int c = c0 + threadIdx.x;
    if (p < HW && c < C) d[p * c_pad + c] = tile[threadIdx.x][r];
  }
}
// c_pad >= C channels per pixel in the NHWC tensor (padding lanes are left untouched)
cudaError_t launch_nchw_to_nhwc_f32(const float* src, float* dst, int B, int C, int H, int W, int c_pad, cudaStream_t s) {
  const long long HW = static_cast<long long>(H) * W;
  dim3 grid(static_cast<unsigned>((HW + 31) / 32), (C + 31) / 32, B), block(32, 8);
  nchw_to_nhwc_f32_kernel<<<grid, block, 0, s>>>(src, dst, C, c_pad, HW);
  return cudaGetLastError();
}
cudaError_t launch_nhwc_to_nchw_f32(const float* src, float* dst, int B, int C, int H, int W, int c_pad, cudaStream_t s) {
  return launch_unpack_state(NINT_TF32, src, dst, B, C, H, W, c_pad, s);
}

// ------------------------------------------------------------------------------------------
// Tangent-linear cell step (nint_forward_tangent), the linearisation of the forward epilogue (model.py:221-229) at the
// saved gates:  da = the tangent GEMM's raw dump (i, f, o columns hold da/2: the packed forward weights are halved),
//   di = i(1-i) da_i   df = f(1-f) da_f   dg = (1-g^2) da_g   do = o(1-o) da_o
//   dc_t = f dc_{t-1} + c_{t-1} df + g di + i dg        dh_t = tanh(c_t) do + o (1 - tanh^2(c_t)) dc_t
// One thread per (pixel, 8 hidden channels): its raw / gate columns are four 8-wide runs of the q-order row
// (grp*64 + gate*16 + half*8), c and dc eight consecutive fp32; consecutive threads walk a pixel's channel groups, so a
// warp reads contiguous spans.  Every load of the thread is issued before the first use.  Padded hidden channels
// (zero weights) get raw = 0 and c = 0, so their dc and dh stay exactly 0.  dc_in / dc_out: the same buffer (updated in
// place) or, on NINT_FLAG_SECOND_ORDER plans, consecutive slots of the per-step dc history the second-order pass reads.
// ------------------------------------------------------------------------------------------
// BIAS: add the parameter tangent's q-order bias dbias_q [4*hc] (i/f/o halved like raw) to raw first, and store the
// sum back into raw, so the dump holds the whole tangent pre-activation (the second-order pass linearises at it)
template <typename E, bool BIAS>
__device__ __forceinline__ void tangent_cell_body(float* __restrict__ raw, const E* __restrict__ gates,
                                                  const float* __restrict__ c_prev, const float* __restrict__ c_cur,
                                                  const float* dc_in, float* dc_out, E* __restrict__ dh_out, long long npix,
                                                  int hc, int hc_pad, const float* __restrict__ dbias_q) {
  constexpr bool FAST = std::is_same<E, __nv_bfloat16>::value;   // the forward's activation variant (nint_common.cuh)
  const int groups = hc / 8;
  const long long total = npix * groups;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long pix = i / groups;
    const int c0 = static_cast<int>(i - pix * groups) * 8;
    const int q0 = (c0 >> 4) * 64 + (c0 & 8);
    const float* rp = raw + pix * 4 * hc + q0;
    const E* gp = gates + pix * 4 * hc + q0;
    const long long ci = pix * hc + c0;
    float a[4][8], g[4][8], cp[8], cc[8], d[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) load_elems<float, 8>(rp + k * 16, a[k]);
#pragma unroll
    for (int k = 0; k < 4; ++k) load_elems<E, 8>(gp + k * 16, g[k]);
    load_elems<float, 8>(c_prev + ci, cp);
    load_elems<float, 8>(c_cur + ci, cc);
    load_elems<float, 8>(dc_in + ci, d);
    if constexpr (BIAS) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float b[8];
        load_elems<float, 8>(dbias_q + q0 + k * 16, b);
#pragma unroll
        for (int j = 0; j < 8; ++j) a[k][j] += b[j];
        store_elems<float, 8>(raw + pix * 4 * hc + q0 + k * 16, a[k]);
      }
    }
    float h[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float i_ = g[0][j], f_ = g[1][j], g_ = g[2][j], o_ = g[3][j];
      const float di = fmaf(-i_, i_, i_) * (2.f * a[0][j]);
      const float df = fmaf(-f_, f_, f_) * (2.f * a[1][j]);
      const float dg = fmaf(-g_, g_, 1.f) * a[2][j];
      const float d_o = fmaf(-o_, o_, o_) * (2.f * a[3][j]);
      const float dcv = fmaf(f_, d[j], fmaf(cp[j], df, fmaf(g_, di, i_ * dg)));
      const float tc = act_tanh<FAST>(cc[j]);
      d[j] = dcv;
      // dh_t is the next GEMM's operand: tf32 rounds to nearest here (the MMA would truncate), bf16 as it is stored
      h[j] = round_for(fmaf(tc, d_o, o_ * fmaf(-tc, tc, 1.f) * dcv), static_cast<E*>(nullptr));
    }
    store_elems<float, 8>(dc_out + ci, d);
    store_elems<E, 8>(dh_out + pix * hc_pad + c0, h);
  }
}

template <typename E>
__global__ void __launch_bounds__(256) tangent_cell_kernel(const float* __restrict__ raw, const E* __restrict__ gates,
                                                           const float* __restrict__ c_prev, const float* __restrict__ c_cur,
                                                           const float* dc_in, float* dc_out, E* __restrict__ dh_out,
                                                           long long npix, int hc, int hc_pad) {
  tangent_cell_body<E, false>(const_cast<float*>(raw), gates, c_prev, c_cur, dc_in, dc_out, dh_out, npix, hc, hc_pad, nullptr);
}

// the same with a parameter tangent's bias (layers whose bias is not folded into the GEMM through the constant-1 lane)
template <typename E>
__global__ void __launch_bounds__(256) tangent_cell_bias_kernel(float* __restrict__ raw, const E* __restrict__ gates,
                                                                const float* __restrict__ c_prev,
                                                                const float* __restrict__ c_cur, const float* dc_in,
                                                                float* dc_out, E* __restrict__ dh_out, long long npix,
                                                                int hc, int hc_pad, const float* __restrict__ dbias_q) {
  tangent_cell_body<E, true>(raw, gates, c_prev, c_cur, dc_in, dc_out, dh_out, npix, hc, hc_pad, dbias_q);
}

template <typename E>
static void launch_tangent_cell_e(long long blocks, float* raw, const void* gates, const float* c_prev,
                                  const float* c_cur, const float* dc_in, float* dc_out, void* dh_out, long long npix,
                                  int hc, int hc_pad, cudaStream_t s, const float* dbias_q) {
  const E* g = reinterpret_cast<const E*>(gates);
  E* dh = reinterpret_cast<E*>(dh_out);
  if (dbias_q)
    tangent_cell_bias_kernel<E><<<blocks, 256, 0, s>>>(raw, g, c_prev, c_cur, dc_in, dc_out, dh, npix, hc, hc_pad, dbias_q);
  else
    tangent_cell_kernel<E><<<blocks, 256, 0, s>>>(raw, g, c_prev, c_cur, dc_in, dc_out, dh, npix, hc, hc_pad);
}

cudaError_t launch_tangent_cell(int dtype, float* raw, const void* gates, const float* c_prev, const float* c_cur,
                                const float* dc_in, float* dc_out, void* dh_out, long long npix, int hc, int hc_pad,
                                cudaStream_t s, const float* dbias_q) {
  const long long total = npix * (hc / 8);
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks <= 0) return cudaSuccess;
  if (dtype == NINT_BF16)
    launch_tangent_cell_e<__nv_bfloat16>(blocks, raw, gates, c_prev, c_cur, dc_in, dc_out, dh_out, npix, hc, hc_pad, s, dbias_q);
  else
    launch_tangent_cell_e<float>(blocks, raw, gates, c_prev, c_cur, dc_in, dc_out, dh_out, npix, hc, hc_pad, s, dbias_q);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Second-order adjoint cell step (nint_backward_second_order): the cell's adjoint (the fused backward's epilogue,
// nint_epilogue.cuh) and its linearisation at the saved gates i, f, g, o, c_{t-1} = cp, c_t = c, tau = tanh(c) and the
// tangent pass's da (raw, i/f/o halved), dc_{t-1} = dcp, dc_t = dc:
//   eta = dgrad h part + u w_head              deta = its tangent + du w_head
//   di = i(1-i) da_i  df = f(1-f) da_f  dg = (1-g^2) da_g  do = o(1-o) da_o  dtau = (1-tau^2) dc
//   kt  = k + eta o (1-tau^2)                  dkt  = dk + deta o (1-tau^2) + eta do (1-tau^2) - 2 eta o tau dtau
//   ai  = kt g i(1-i)                          dai  = dkt g i(1-i) + kt dg i(1-i) + kt g (1-2i) di
//   af  = kt cp f(1-f)                         daf  = dkt cp f(1-f) + kt dcp f(1-f) + kt cp (1-2f) df
//   ag  = kt i (1-g^2)                         dag  = dkt i (1-g^2) + kt di (1-g^2) - 2 kt i g dg
//   ao  = eta tau o(1-o)                       dao  = deta tau o(1-o) + eta dtau o(1-o) + eta tau (1-2o) do
//   k <- kt f                                  dk  <- dkt f + kt df
// ai .. ao and their tangents are stored like the fused backward stores dgates over G (q-order, unscaled, rounded to
// the operand format: the packed dgrad panels apply unchanged).  Thread layout and load order as tangent_cell_kernel;
// padded hidden channels have zero raw, c, eta and head weight, so their outputs stay exactly 0.
// ------------------------------------------------------------------------------------------
// DHW: the head weight has a tangent too (parameter direction): deta also gains u dhead_w
template <typename E, bool DHW>
__device__ __forceinline__ void soa_cell_body(const float* __restrict__ eta, const float* __restrict__ u,
                                              long long u_bstride, const float* __restrict__ du, long long du_bstride,
                                              const float* __restrict__ head_w, const E* __restrict__ gates,
                                              const float* __restrict__ traw, const float* __restrict__ c_prev,
                                              const float* __restrict__ c_cur, const float* __restrict__ dc_prev,
                                              const float* __restrict__ dc_cur, float* __restrict__ kappa,
                                              E* __restrict__ da_out, long long npix, long long HW, int hc,
                                              const float* __restrict__ dhead_w) {
  constexpr bool FAST = std::is_same<E, __nv_bfloat16>::value;
  const int groups = hc / 8;
  const long long total = npix * groups;
  const long long nk = npix * hc;   // offset of the tangent half of eta / kappa
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long pix = i / groups;
    const int c0 = static_cast<int>(i - pix * groups) * 8;
    const int q0 = (c0 >> 4) * 64 + (c0 & 8);
    const long long gi = pix * 4 * hc + q0;
    const long long ci = pix * hc + c0;
    float a[4][8], g[4][8], cp[8], cc[8], dcp[8], dcc[8], e[8], de[8], k[8], dk[8], w[8], dw[8];
    float uv = 0.f, duv = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) load_elems<float, 8>(traw + gi + q * 16, a[q]);
#pragma unroll
    for (int q = 0; q < 4; ++q) load_elems<E, 8>(gates + gi + q * 16, g[q]);
    load_elems<float, 8>(c_prev + ci, cp);
    load_elems<float, 8>(c_cur + ci, cc);
    load_elems<float, 8>(dc_prev + ci, dcp);
    load_elems<float, 8>(dc_cur + ci, dcc);
    load_elems<float, 8>(kappa + ci, k);
    load_elems<float, 8>(kappa + nk + ci, dk);
    if (eta) {
      load_elems<float, 8>(eta + ci, e);
      load_elems<float, 8>(eta + nk + ci, de);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) e[j] = de[j] = 0.f;
    }
    if (u || du) {
      const long long b = pix / HW, r = pix - b * HW;
      if (u) uv = __ldg(u + b * u_bstride + r);
      if (du) duv = __ldg(du + b * du_bstride + r);
      load_elems<float, 8>(head_w + c0, w);
      if constexpr (DHW) load_elems<float, 8>(dhead_w + c0, dw);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) w[j] = dw[j] = 0.f;
    }
    float o0[4][8], o1[4][8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float i_ = g[0][j], f_ = g[1][j], g_ = g[2][j], o_ = g[3][j];
      const float si = fmaf(-i_, i_, i_), sf = fmaf(-f_, f_, f_), so = fmaf(-o_, o_, o_), tg = fmaf(-g_, g_, 1.f);
      const float di = si * (2.f * a[0][j]), df = sf * (2.f * a[1][j]), dg = tg * a[2][j], d_o = so * (2.f * a[3][j]);
      const float tau = act_tanh<FAST>(cc[j]);
      const float tt = fmaf(-tau, tau, 1.f);
      const float dtau = tt * dcc[j];
      const float et = fmaf(uv, w[j], e[j]);
      float det = fmaf(duv, w[j], de[j]);
      if constexpr (DHW) det = fmaf(uv, dw[j], det);
      const float kt = fmaf(et * o_, tt, k[j]);
      const float dkt = fmaf(det * o_, tt, fmaf(et * d_o, tt, fmaf(-2.f * et * o_, tau * dtau, dk[j])));
      o0[0][j] = kt * g_ * si;
      o1[0][j] = fmaf(dkt * g_, si, fmaf(kt * dg, si, kt * g_ * fmaf(-2.f, i_, 1.f) * di));
      o0[1][j] = kt * cp[j] * sf;
      o1[1][j] = fmaf(dkt * cp[j], sf, fmaf(kt * dcp[j], sf, kt * cp[j] * fmaf(-2.f, f_, 1.f) * df));
      o0[2][j] = kt * i_ * tg;
      o1[2][j] = fmaf(dkt * i_, tg, fmaf(kt * di, tg, -2.f * kt * i_ * g_ * dg));
      o0[3][j] = et * tau * so;
      o1[3][j] = fmaf(det * tau, so, fmaf(et * dtau, so, et * tau * fmaf(-2.f, o_, 1.f) * d_o));
      k[j] = kt * f_;
      dk[j] = fmaf(dkt, f_, kt * df);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        // dgates are the next dgrad's operands: tf32 rounds to nearest here (the MMA would truncate), bf16 as stored
        o0[q][j] = round_for(o0[q][j], static_cast<E*>(nullptr));
        o1[q][j] = round_for(o1[q][j], static_cast<E*>(nullptr));
      }
    }
    store_elems<float, 8>(kappa + ci, k);
    store_elems<float, 8>(kappa + nk + ci, dk);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      store_elems<E, 8>(da_out + gi + q * 16, o0[q]);
      store_elems<E, 8>(da_out + npix * 4 * hc + gi + q * 16, o1[q]);
    }
  }
}

template <typename E>
__global__ void __launch_bounds__(256) soa_cell_kernel(const float* __restrict__ eta, const float* __restrict__ u,
                                                       long long u_bstride, const float* __restrict__ du,
                                                       long long du_bstride, const float* __restrict__ head_w,
                                                       const E* __restrict__ gates, const float* __restrict__ traw,
                                                       const float* __restrict__ c_prev, const float* __restrict__ c_cur,
                                                       const float* __restrict__ dc_prev, const float* __restrict__ dc_cur,
                                                       float* __restrict__ kappa, E* __restrict__ da_out, long long npix,
                                                       long long HW, int hc) {
  soa_cell_body<E, false>(eta, u, u_bstride, du, du_bstride, head_w, gates, traw, c_prev, c_cur, dc_prev, dc_cur, kappa,
                          da_out, npix, HW, hc, nullptr);
}

// the same with the head weight's tangent of a parameter direction
template <typename E>
__global__ void __launch_bounds__(256) soa_cell_dhead_kernel(const float* __restrict__ eta, const float* __restrict__ u,
                                                             long long u_bstride, const float* __restrict__ du,
                                                             long long du_bstride, const float* __restrict__ head_w,
                                                             const E* __restrict__ gates, const float* __restrict__ traw,
                                                             const float* __restrict__ c_prev,
                                                             const float* __restrict__ c_cur,
                                                             const float* __restrict__ dc_prev,
                                                             const float* __restrict__ dc_cur, float* __restrict__ kappa,
                                                             E* __restrict__ da_out, long long npix, long long HW, int hc,
                                                             const float* __restrict__ dhead_w) {
  soa_cell_body<E, true>(eta, u, u_bstride, du, du_bstride, head_w, gates, traw, c_prev, c_cur, dc_prev, dc_cur, kappa,
                         da_out, npix, HW, hc, dhead_w);
}

template <typename E>
static void launch_soa_cell_e(long long blocks, const float* eta, const float* u, long long u_bstride, const float* du,
                              long long du_bstride, const float* head_w, const void* gates, const float* traw,
                              const float* c_prev, const float* c_cur, const float* dc_prev, const float* dc_cur,
                              float* kappa, void* da_out, long long npix, long long HW, int hc, cudaStream_t s,
                              const float* dhead_w) {
  const E* g = reinterpret_cast<const E*>(gates);
  E* da = reinterpret_cast<E*>(da_out);
  if (dhead_w)
    soa_cell_dhead_kernel<E><<<blocks, 256, 0, s>>>(eta, u, u_bstride, du, du_bstride, head_w, g, traw, c_prev, c_cur,
                                                    dc_prev, dc_cur, kappa, da, npix, HW, hc, dhead_w);
  else
    soa_cell_kernel<E><<<blocks, 256, 0, s>>>(eta, u, u_bstride, du, du_bstride, head_w, g, traw, c_prev, c_cur, dc_prev,
                                              dc_cur, kappa, da, npix, HW, hc);
}

cudaError_t launch_soa_cell(int dtype, const float* eta, const float* u, long long u_bstride, const float* du,
                            long long du_bstride, const float* head_w, const void* gates, const float* traw,
                            const float* c_prev, const float* c_cur, const float* dc_prev, const float* dc_cur,
                            float* kappa, void* da_out, long long npix, long long HW, int hc, cudaStream_t s,
                            const float* dhead_w) {
  const long long total = npix * (hc / 8);
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks <= 0) return cudaSuccess;
  if (dtype == NINT_BF16)
    launch_soa_cell_e<__nv_bfloat16>(blocks, eta, u, u_bstride, du, du_bstride, head_w, gates, traw, c_prev, c_cur, dc_prev,
                                     dc_cur, kappa, da_out, npix, HW, hc, s, dhead_w);
  else
    launch_soa_cell_e<float>(blocks, eta, u, u_bstride, du, du_bstride, head_w, gates, traw, c_prev, c_cur, dc_prev,
                             dc_cur, kappa, da_out, npix, HW, hc, s, dhead_w);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// weight packing.  Reference layout: W[n][c][dy][dx], n = gate*hc + channel, c over cat(x, h)
// (model.py:207-211,219).  Packed panel row index = ((nb*nchunks + chunk)*taps + tap)*n_tile + col,
// each row holds one chunk (CE elements) of K.
// ------------------------------------------------------------------------------------------
// gate / hidden channel of kernel column q (q-order, nint_kernels.h)
__device__ __forceinline__ int q_gate(int q) { return (q >> 4) & 3; }
__device__ __forceinline__ int q_chan(int q) { return (q >> 6) * 16 + (q & 15); }

// hc = the layer's (padded) hidden size the kernels run with, hc_real <= hc the reference's: weights and biases of the
// padding channels are zero, so their gates are (0.5, 0.5, 0, 0.5) and their c and h stay exactly 0 (model.py:223-229)
template <typename E>
__global__ void pack_w_fwd_kernel(const float* __restrict__ w, const float* __restrict__ bias, E* __restrict__ wx,
                                  E* __restrict__ wh, float* __restrict__ bias_q, int cin, int hc_real, int hc, int hcb,
                                  int k, int cx_pad, int hc_pad, int bias_lane) {
  constexpr int CE = ElemTraits<E>::kPerChunk;
  const int n_blocks = hc / hcb, n_tile = 4 * hcb, taps = k * k;
  const int ctot = cin + hc_real;
  const int chx = cx_pad / CE, chh = hc_pad / CE;
  const long long nx = static_cast<long long>(n_blocks) * taps * chx * n_tile * CE;
  const long long nh = static_cast<long long>(n_blocks) * taps * chh * n_tile * CE;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < nx + nh;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const bool is_h = idx >= nx;
    long long r = is_h ? idx - nx : idx;
    const int nch = is_h ? chh : chx;
    const int e = static_cast<int>(r % CE); r /= CE;
    const int col = static_cast<int>(r % n_tile); r /= n_tile;
    const int tap = static_cast<int>(r % taps); r /= taps;
    const int ch = static_cast<int>(r % nch);
    const int nb = static_cast<int>(r / nch);
    const int q = nb * n_tile + col;
    const int oc = q_chan(q);
    const int cl = ch * CE + e;
    const int climit = is_h ? hc_real : cin;
    float v = 0.f;
    if (cl < climit && oc < hc_real)
      v = w[(static_cast<long long>(q_gate(q) * hc_real + oc) * ctot + (is_h ? cin + cl : cl)) * taps + tap];
    // bias folded into the GEMM: the input carries 1.0 in padding lane `bias_lane`, so the centre tap's weight for that
    // lane IS the bias (the epilogue then adds nothing); off the centre the lane keeps a zero weight
    if (!is_h && cl == bias_lane && tap == taps / 2 && oc < hc_real && bias) v = bias[q_gate(q) * hc_real + oc];
    // sigmoid gates (i, f, o) are fed HALVED pre-activations (act_sigmoid_halved): exact, 0.5 is a power of two
    if (q_gate(q) != 2) v *= 0.5f;
    (is_h ? wh : wx)[is_h ? idx - nx : idx] = to_elem<E>(v);
  }
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < 4 * hc; q += gridDim.x * blockDim.x)
    bias_q[q] = (bias && q_chan(q) < hc_real) ? bias[q_gate(q) * hc_real + q_chan(q)] * (q_gate(q) != 2 ? 0.5f : 1.f) : 0.f;
}

// dgrad operands: K = q (4*hc), N = input channel, taps flipped (transposed convolution):
//   wd[chunk][tap'][col][e] = W[n(q = chunk*CE + e)][c(col)][k-1-dy'][k-1-dx']
// wdx has cin_rows >= cin rows of N (rows >= cin are zero: the padded width of the tensor the gradient flows into),
// wdh has hc rows (rows >= hc_real zero)
template <typename E>
__global__ void pack_w_bwd_kernel(const float* __restrict__ w, E* __restrict__ wdx, E* __restrict__ wdh, int cin,
                                  int cin_rows, int hc_real, int hc, int k) {
  constexpr int CE = ElemTraits<E>::kPerChunk;
  const int taps = k * k, ctot = cin + hc_real, nch = 4 * hc / CE;
  const long long nx = wdx ? static_cast<long long>(taps) * nch * cin_rows * CE : 0;
  const long long nh = static_cast<long long>(taps) * nch * hc * CE;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < nx + nh;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const bool is_h = idx >= nx;
    long long r = is_h ? idx - nx : idx;
    const int ncol = is_h ? hc : cin_rows;
    const int e = static_cast<int>(r % CE); r /= CE;
    const int col = static_cast<int>(r % ncol); r /= ncol;
    const int tap = static_cast<int>(r % taps);
    const int ch = static_cast<int>(r / taps);
    const int q = ch * CE + e;
    const int oc = q_chan(q);
    float v = 0.f;
    if (oc < hc_real && col < (is_h ? hc_real : cin)) {
      const int c = is_h ? cin + col : col;
      v = w[(static_cast<long long>(q_gate(q) * hc_real + oc) * ctot + c) * taps + (taps - 1 - tap)];
    }
    (is_h ? wdh : wdx)[is_h ? idx - nx : idx] = to_elem<E>(v);
  }
}

cudaError_t launch_pack_weights_fwd(int dtype, const float* w, const float* bias, void* wx, void* wh, float* bias_q,
                                    int cin, int hc_real, int hc, int hcb, int k, int cx_pad, int hc_pad, int bias_lane,
                                    cudaStream_t s) {
  if (dtype == NINT_BF16)
    pack_w_fwd_kernel<__nv_bfloat16><<<296, 256, 0, s>>>(w, bias, reinterpret_cast<__nv_bfloat16*>(wx),
                                                         reinterpret_cast<__nv_bfloat16*>(wh), bias_q, cin, hc_real, hc, hcb,
                                                         k, cx_pad, hc_pad, bias_lane);
  else
    pack_w_fwd_kernel<float><<<296, 256, 0, s>>>(w, bias, reinterpret_cast<float*>(wx), reinterpret_cast<float*>(wh),
                                                 bias_q, cin, hc_real, hc, hcb, k, cx_pad, hc_pad, bias_lane);
  return cudaGetLastError();
}
cudaError_t launch_pack_weights_bwd(int dtype, const float* w, void* wdx, void* wdh, int cin, int cin_rows, int hc_real,
                                    int hc, int k, cudaStream_t s) {
  if (dtype == NINT_BF16)
    pack_w_bwd_kernel<__nv_bfloat16><<<296, 256, 0, s>>>(w, reinterpret_cast<__nv_bfloat16*>(wdx),
                                                         reinterpret_cast<__nv_bfloat16*>(wdh), cin, cin_rows, hc_real, hc, k);
  else
    pack_w_bwd_kernel<float><<<296, 256, 0, s>>>(w, reinterpret_cast<float*>(wdx), reinterpret_cast<float*>(wdh), cin,
                                                 cin_rows, hc_real, hc, k);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// 1x1 head: pred[b][pix] = bias + sum_c h[b][pix][c] * w[c]    (model.py:274)
// One thread per pixel, 16-byte loads; a pixel's channel vector (<= 512 B) stays in L1 between the thread's consecutive
// loads, so DRAM traffic is the algorithmic hc_pad*sizeof(E) per pixel, and a thread keeps hc_pad*sizeof(E)/16 loads in
// flight.  Measured under ncu at cfg 2 (53 MB): 20 us; a warp-cooperative version with fully coalesced 512-byte
// requests but one load in flight per lane took 26 us, the same with four in flight per lane 49 us (95 registers).
// ------------------------------------------------------------------------------------------
template <typename E>
__global__ void head_fwd_kernel(const E* __restrict__ h, const float* __restrict__ w, const float* __restrict__ bias,
                                float* __restrict__ out, long long npix, int B, int hc, int hc_pad,
                                long long out_bstride) {
  extern __shared__ float s_w[];
  for (int i = threadIdx.x; i < hc_pad; i += blockDim.x) s_w[i] = i < hc ? w[i] : 0.f;
  __syncthreads();
  constexpr int V = 16 / sizeof(E);
  const long long total = static_cast<long long>(B) * npix;
  const float b0 = bias[0];
  for (long long gp = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; gp < total;
       gp += static_cast<long long>(gridDim.x) * blockDim.x) {
    const E* hp = h + gp * hc_pad;
    float acc = b0;
    for (int c0 = 0; c0 < hc_pad; c0 += V) {
      float f[V];
      load_elems<E, V>(hp + c0, f);
#pragma unroll
      for (int j = 0; j < V; ++j) acc = fmaf(f[j], s_w[c0 + j], acc);
    }
    const long long b = gp / npix;
    out[b * out_bstride + (gp - b * npix)] = acc;
  }
}

cudaError_t launch_head_fwd(int dtype, const void* h, const float* w, const float* b, float* out, long long npix,
                            int B, int hc, int hc_pad, long long out_bstride, cudaStream_t s) {
  const long long total = static_cast<long long>(B) * npix;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks <= 0) return cudaSuccess;
  if (dtype == NINT_BF16)
    head_fwd_kernel<__nv_bfloat16><<<blocks, 256, hc_pad * 4, s>>>(reinterpret_cast<const __nv_bfloat16*>(h), w, b, out,
                                                                  npix, B, hc, hc_pad, out_bstride);
  else
    head_fwd_kernel<float><<<blocks, 256, hc_pad * 4, s>>>(reinterpret_cast<const float*>(h), w, b, out, npix, B, hc,
                                                          hc_pad, out_bstride);
  return cudaGetLastError();
}

// Head tangent with a parameter direction: out = db + sum_c dh[pix][c] w[c] + h[pix][c] dw[c].  Same thread layout as
// head_fwd_kernel, reading the primal and the tangent h of a pixel in the same pass.
template <typename E>
__global__ void head_tangent_kernel(const E* __restrict__ h, const E* __restrict__ dh, const float* __restrict__ w,
                                    const float* __restrict__ dw, const float* __restrict__ db, float* __restrict__ out,
                                    long long npix, int B, int hc, int hc_pad, long long out_bstride) {
  extern __shared__ float s_w[];   // [hc_pad] w, then [hc_pad] dw
  for (int i = threadIdx.x; i < hc_pad; i += blockDim.x) {
    s_w[i] = i < hc ? w[i] : 0.f;
    s_w[hc_pad + i] = i < hc ? dw[i] : 0.f;
  }
  __syncthreads();
  constexpr int V = 16 / sizeof(E);
  const long long total = static_cast<long long>(B) * npix;
  const float b0 = db[0];
  for (long long gp = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; gp < total;
       gp += static_cast<long long>(gridDim.x) * blockDim.x) {
    const E* hp = h + gp * hc_pad;
    const E* dp = dh + gp * hc_pad;
    float acc = b0;
    for (int c0 = 0; c0 < hc_pad; c0 += V) {
      float f[V], d[V];
      load_elems<E, V>(dp + c0, d);
      load_elems<E, V>(hp + c0, f);
#pragma unroll
      for (int j = 0; j < V; ++j) acc = fmaf(f[j], s_w[hc_pad + c0 + j], fmaf(d[j], s_w[c0 + j], acc));
    }
    const long long b = gp / npix;
    out[b * out_bstride + (gp - b * npix)] = acc;
  }
}

cudaError_t launch_head_tangent(int dtype, const void* h, const void* dh, const float* w, const float* dw, const float* db,
                                float* out, long long npix, int B, int hc, int hc_pad, long long out_bstride,
                                cudaStream_t s) {
  const long long total = static_cast<long long>(B) * npix;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks <= 0) return cudaSuccess;
  if (dtype == NINT_BF16)
    head_tangent_kernel<__nv_bfloat16><<<blocks, 256, 2 * hc_pad * 4, s>>>(
        reinterpret_cast<const __nv_bfloat16*>(h), reinterpret_cast<const __nv_bfloat16*>(dh), w, dw, db, out, npix, B, hc,
        hc_pad, out_bstride);
  else
    head_tangent_kernel<float><<<blocks, 256, 2 * hc_pad * 4, s>>>(reinterpret_cast<const float*>(h),
                                                                  reinterpret_cast<const float*>(dh), w, dw, db, out,
                                                                  npix, B, hc, hc_pad, out_bstride);
  return cudaGetLastError();
}

static int head_lanes_per_pixel(int dtype, int hc_pad) {
  const int cpp = hc_pad / (dtype == NINT_BF16 ? 8 : 4);
  int lp = 1;
  while (lp * 2 <= cpp && lp < 32) lp *= 2;     // largest power of two <= min(cpp, 32) (cpp is 4 * k: lp >= 4)
  return lp;
}

// head backward: dw[c] = sum_pix dpred[pix] * h[pix][c], db = sum dpred   (dh is fused into the gate-backward
// epilogue).  Same access pattern as the forward: LP lanes share a pixel and each lane keeps the partial sums of its
// own 16-byte channel slices in registers across all its pixels; one shuffle + shared-memory reduction per block at
// the end, then either fp32 atomics (default) or a per-block partial row reduced in a fixed order by the caller's
// second launch (deterministic mode: `part` != null, [gridDim.x * gridDim.y][hc_pad + 1]).
template <typename E>
__global__ void __launch_bounds__(256) head_bwd_kernel(const E* __restrict__ h, const float* __restrict__ dpred,
                                                       long long dpred_bstride, float* __restrict__ dw,
                                                       float* __restrict__ db, long long npix, int hc, int hc_pad, int lp,
                                                       float* __restrict__ part) {
  constexpr int V = 16 / sizeof(E);
  constexpr int KMAX = 2;                       // chunk slots per lane: cpp / lp <= 2 (hc_pad <= 256)
  const int cpp = hc_pad / V;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & (lp - 1), ppw = 32 / lp;
  const int b = blockIdx.y;
  const float* dp = dpred + b * dpred_bstride;
  const E* hb = h + static_cast<long long>(b) * npix * hc_pad;
  float acc[KMAX][V];
#pragma unroll
  for (int k = 0; k < KMAX; ++k)
#pragma unroll
    for (int j = 0; j < V; ++j) acc[k][j] = 0.f;
  float accb = 0.f;
  const long long wstride = static_cast<long long>(gridDim.x) * (blockDim.x >> 5) * ppw;
  for (long long p0 = (static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + warp) * ppw; p0 < npix; p0 += wstride) {
    const long long px = p0 + lane / lp;
    if (px < npix) {
      const float d = __ldg(dp + px);
      const E* row = hb + px * hc_pad;
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        const int ck = sub + k * lp;
        if (ck < cpp) {
          float f[V];
          load_elems<E, V>(row + ck * V, f);
#pragma unroll
          for (int j = 0; j < V; ++j) acc[k][j] = fmaf(d, f[j], acc[k][j]);
        }
      }
      if (sub == 0) accb += d;
    }
  }
  // lanes with the same `sub` hold partial sums of the same channels: fold them (offsets lp, 2*lp, ...)
  for (int o = lp; o < 32; o <<= 1) {
#pragma unroll
    for (int k = 0; k < KMAX; ++k)
#pragma unroll
      for (int j = 0; j < V; ++j) acc[k][j] += __shfl_xor_sync(0xffffffffu, acc[k][j], o);
    accb += __shfl_xor_sync(0xffffffffu, accb, o);
  }
  __shared__ float red[8][256 + 1];
  if (lane < lp) {
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
      const int ck = sub + k * lp;
      if (ck < cpp) {
#pragma unroll
        for (int j = 0; j < V; ++j) red[warp][ck * V + j] = acc[k][j];
      }
    }
    if (lane == 0) red[warp][256] = accb;
  }
  __syncthreads();
  const int blk = blockIdx.y * gridDim.x + blockIdx.x;
  for (int c = threadIdx.x; c <= hc; c += blockDim.x) {
    const int col = c < hc ? c : 256;            // c == hc: the bias column
    float sum = 0.f;
    for (int wv = 0; wv < 8; ++wv) sum += red[wv][col];
    if (part) part[static_cast<long long>(blk) * (hc + 1) + c] = sum;
    else atomicAdd(c < hc ? dw + c : db, sum);
  }
}
// deterministic mode: fixed-order sum of the per-block partial rows; accumulates into dw / db
__global__ void head_bwd_reduce_kernel(const float* __restrict__ part, int nblocks, int hc, float* __restrict__ dw,
                                       float* __restrict__ db) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c <= hc; c += gridDim.x * blockDim.x) {
    float sum = 0.f;
    for (int i = 0; i < nblocks; ++i) sum += part[static_cast<long long>(i) * (hc + 1) + c];
    if (c < hc) dw[c] += sum; else db[0] += sum;
  }
}

int head_bwd_blocks(int B) {
  int gx = (148 * 4 + B - 1) / B;
  return (gx < 1 ? 1 : gx) * B;
}
cudaError_t launch_head_bwd(int dtype, const void* h, const float* dpred, long long dpred_bstride, float* dw, float* db,
                            long long npix, int B, int hc, int hc_pad, float* part, cudaStream_t s) {
  if (hc_pad > 256) return cudaErrorInvalidValue;
  const int lp = head_lanes_per_pixel(dtype, hc_pad);
  const dim3 grid(head_bwd_blocks(B) / B, B);
  if (dtype == NINT_BF16)
    head_bwd_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(h), dpred, dpred_bstride,
                                                       dw, db, npix, hc, hc_pad, lp, part);
  else
    head_bwd_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(h), dpred, dpred_bstride, dw, db, npix,
                                               hc, hc_pad, lp, part);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || !part) return e;
  head_bwd_reduce_kernel<<<1, 256, 0, s>>>(part, grid.x * grid.y, hc, dw, db);
  return cudaGetLastError();
}

// dw_acc [taps][4hc (q)][ncols] -> grad W[n][c][dy][dx];  col(c) = c (x part) or cx_pad + (c - cin) (h part).
// nparts > 0 (deterministic mode): dw_acc / db_acc hold `nparts` partial-sum slices one after the other, summed here in a
// fixed order.
__global__ void unpack_wgrad_kernel(const float* __restrict__ dw_acc, const float* __restrict__ db_acc,
                                    float* __restrict__ gw, float* __restrict__ gb, int cin, int hc_real, int hc, int k,
                                    int ncols, int cx_pad, int bias_col, int accumulate, int nparts,
                                    const float* __restrict__ db_resid, int resid_slots) {
  const int taps = k * k, ctot = cin + hc_real, hc4 = 4 * hc;
  const long long total = static_cast<long long>(hc4) * ctot * taps;
  const long long slice = static_cast<long long>(taps) * hc4 * ncols;
  const int np = nparts > 0 ? nparts : 1;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    // read-coalesced order: (tap, q, c)
    const int c = static_cast<int>(idx % ctot);
    long long r = idx / ctot;
    const int q = static_cast<int>(r % hc4);
    const int tap = static_cast<int>(r / hc4);
    if (q_chan(q) >= hc_real) continue;   // padding channel of the hidden size: no such row in the reference's weight
    const int col = c < cin ? c : cx_pad + (c - cin);
    const float* src = dw_acc + (static_cast<long long>(tap) * hc4 + q) * ncols + col;
    float v = 0.f;
    for (int s = 0; s < np; ++s) v += src[s * slice];
    float* dst = gw + (static_cast<long long>(q_gate(q) * hc_real + q_chan(q)) * ctot + c) * taps + tap;
    *dst = accumulate ? *dst + v : v;
  }
  if (gb) {
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < hc4; q += gridDim.x * blockDim.x) {
      if (q_chan(q) >= hc_real) continue;
      float* dst = gb + q_gate(q) * hc_real + q_chan(q);
      // bias_col: x carried 1.0 in that channel, so the centre tap's column is sum_pixels dgates = db
      float v = 0.f;
      for (int s = 0; s < np; ++s)
        v += bias_col >= 0 ? dw_acc[s * slice + (static_cast<long long>(taps / 2) * hc4 + q) * ncols + bias_col]
                           : db_acc[static_cast<long long>(s) * hc4 + q];
      // tf32 mode: plus what rounding the stored dgates to tf32 took away from the sum (fixed-order over the slots)
      float r = 0.f;
      for (int i = 0; i < resid_slots; ++i) r += db_resid[static_cast<long long>(i) * hc4 + q];
      v += r;
      *dst = accumulate ? *dst + v : v;
    }
  }
}
cudaError_t launch_unpack_wgrad(const float* dw_acc, const float* db_acc, float* gw, float* gb, int cin, int hc_real,
                                int hc, int k, int ncols, int cx_pad, int bias_col, int accumulate, int nparts,
                                const float* db_resid, int resid_slots, cudaStream_t s) {
  unpack_wgrad_kernel<<<296, 256, 0, s>>>(dw_acc, db_acc, gw, gb, cin, hc_real, hc, k, ncols, cx_pad, bias_col, accumulate,
                                          nparts, db_resid, db_resid ? resid_slots : 0);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// preprocessing fusion (north-star item 4; dataset.py:520-537 stack + z-score, dataset.py:67-98 halo): stack the
// first L levels of a 3-D forcing [N,L,H,W] with a 2-D emission field [N,H,W] as channel L, z-score per channel,
// append S pre-normalised static attribute fields [S,H,W] (dataset.py:100-122,532-533: the same for every frame),
// cyclic halo in longitude, reflect halo in latitude.  mode 1 reproduces the shipped RNN dataset's quirk (np.fliplr on
// a (T,C,rows,W) slab flips CHANNELS: halo rows keep their order, channel order is reversed; dataset.py:96).
//
// One kernel, two output layouts:
//   PLANAR = false  the frame bank [N][Hp][Wp][CP] of E (bf16, or fp32 holding tf32-rounded values): the model's own
//                   operand layout -- channels-last, zero padding lanes, the constant-1 lane the bias gradient rides on
//                   -- that nint_forward_bank's TMA descriptors read.  No fp32 NCHW intermediate, no second packing pass.
//   PLANAR = true   [N][C][Hp][Wp] fp32: the reference dataset's tensor layout (nint_fuse_inputs).
// One thread per output pixel.  For a fixed channel the warp's loads are 32 consecutive longitudes of one source row
// (coalesced; the cyclic wrap splits at most one request).  What it took to get off the instruction-issue limit
// (measured on B200, 797 MB per call: 698 us -> see profiles/): every load of the pixel is issued before the first
// use, unconditionally (padding lanes re-read channel C-1, an L1 hit: no per-channel branch splits the basic block), and
// the z-score's IEEE division by the per-channel constant is Markstein's sequence on a precomputed RN(1/std) -- q0 =
// RN(a*r), e = a - std*q0 (exact, fma), q = RN(q0 + e*r), the correctly rounded quotient whenever no intermediate leaves
// the normal range -- three dependent FMA-class instructions instead of the ~10 of a general division; out-of-range
// operands take the true division.  Results stay bit-identical to the numpy float32 pipeline.
// ------------------------------------------------------------------------------------------
// z-score with the exact quotient: q0 = a*r; two Newton corrections on the exact (fma) residual.  The first makes q1
// a faithful approximation of a/sd, Markstein's theorem then makes RN(q1 + e1*r) THE correctly rounded quotient.
__device__ __forceinline__ float zscore_exact(float a, float sd, float rcp) {
  const float q0 = a * rcp;
  const float q1 = fmaf(fmaf(-sd, q0, a), rcp, q0);
  return fmaf(fmaf(-sd, q1, a), rcp, q1);
}

struct FuseChan {            // per source channel, built once per block in shared memory
  const float* src;          // frame 0, pixel 0 of the channel's field
  long long frame_stride;    // elements between frames (0 for the static attributes)
};

template <typename E, int CP, bool PLANAR>
__global__ void __launch_bounds__(256) fuse_kernel(const float* __restrict__ lev, const float* __restrict__ emis,
                                                   const float* __restrict__ mean, const float* __restrict__ stdv,
                                                   const float* __restrict__ statics, int S, E* __restrict__ out,
                                                   long long N, int L, int H, int W, int Hp, int Wp, int mode,
                                                   int ones_lane) {
  const int C = L + 1 + S;
  const int HWp = Hp * Wp;
  const long long HW = static_cast<long long>(H) * W;
  __shared__ FuseChan s_ch[CP];
  __shared__ float4 s_k[CP];                  // {mean, std, RN(1/std), range-check poison}; static attributes: {0, 1, 1, 0}
  __shared__ const float* s_base[CP];         // s_ch[c].src advanced to the block's current frame
  for (int c = threadIdx.x; c < CP; c += blockDim.x) {
    FuseChan k;
    const int cc = c < C ? c : C - 1;         // padding lanes alias the last channel (their loads are discarded)
    if (cc < L) { k.src = lev + cc * HW; k.frame_stride = L * HW; }
    else if (cc == L) { k.src = emis; k.frame_stride = HW; }
    else { k.src = statics + (cc - L - 1) * HW; k.frame_stride = 0; }
    s_ch[c] = k;
    const bool zs = cc <= L;
    const float sd = zs ? stdv[cc] : 1.f, rcp = 1.0f / sd;
    // constants whose reciprocal leaves [2^-40, 2^40] (or is not finite) poison the range check: general division
    const bool usual = fabsf(rcp) > 9.1e-13f && fabsf(rcp) < 1.1e12f;
    s_k[c] = make_float4(zs ? mean[cc] : 0.f, sd, rcp, usual ? 0.f : -INFINITY);
  }
  const int left = (Wp - W) / 2, top = (Hp - H) / 2, bot = Hp - H - top;
  const int chunks = (HWp + 255) / 256;       // 256-pixel chunks of one output frame
  const long long items = N * chunks;
  for (long long item = blockIdx.x; item < items; item += gridDim.x) {
    const long long n = item / chunks;        // block-uniform: the frame's base pointers are computed once per chunk
    const int chunk = static_cast<int>(item - n * chunks);
    __syncthreads();
    if (threadIdx.x < CP) s_base[threadIdx.x] = s_ch[threadIdx.x].src + n * s_ch[threadIdx.x].frame_stride;
    __syncthreads();
    const int p = chunk * 256 + static_cast<int>(threadIdx.x);
    if (p >= HWp) continue;
    const int yp = p / Wp, xp = p - yp * Wp;
    int xs = xp - left;                       // cyclic longitude (dataset.py:67-80)
    if (xs < 0) xs += W;
    if (xs >= W) xs -= W;
    int ys = yp - top;
    bool flip = false;                        // mode 1: halo rows carry the channels in reverse order (dataset.py:96)
    if (ys < 0) {                             // upper halo: rows 1..top (dataset.py:82-98)
      if (mode == 0) ys = top - yp; else { ys = 1 + yp; flip = true; }
    } else if (ys >= H) {                     // lower halo: rows H-bot-1..H-2
      const int j = ys - H;
      if (mode == 0) ys = H - 2 - j; else { ys = H - bot - 1 + j; flip = true; }
    }
    const int pix = ys * W + xs;
    // pass 1: loads only, in groups of eight channels (a group past the last channel is skipped; inside a group the
    // padding lanes re-read channel 0 or C-1, an L1 hit): nothing here depends on a loaded value.  pass 2: z-score.
    // Static attributes carry the constants {0, 1, 1}: the same arithmetic returns them unchanged.
    // The exactness argument (Markstein) needs a = v - mean and every intermediate in the normal range: with the
    // per-channel constants vetted once per block (s_k.w) that holds whenever 2^-60 <= |a| <= 2^60, so the only
    // per-element bookkeeping is min / max of |a|; a pixel that fails (zeros included) is redone with the division.
    float v[CP];
    float lo = 3.0e38f, hi = 0.f;
    auto body = [&](auto flip_tag) {
      constexpr bool FLIP = decltype(flip_tag)::value;
#pragma unroll
      for (int c0 = 0; c0 < CP; c0 += 8) {
        if (c0 < C) {
#pragma unroll
          for (int c = c0; c < c0 + 8; ++c) {
            const int cs = FLIP ? (c < C ? C - 1 - c : 0) : c;
            v[c] = __ldg(s_base[cs] + pix);
          }
        } else {
#pragma unroll
          for (int c = c0; c < c0 + 8; ++c) v[c] = 0.f;
        }
      }
#pragma unroll
      for (int c = 0; c < CP; ++c) {
        if (c < C) {
          const float4 k = s_k[FLIP ? C - 1 - c : c];
          const float a = v[c] - k.x;           // IEEE subtract as in numpy
          lo = fminf(lo, fabsf(a) + k.w);       // k.w = 0, or -inf (poison) when the channel's constants are unusual
          hi = fmaxf(hi, fabsf(a));
          v[c] = zscore_exact(a, k.y, k.z);
        } else {
          v[c] = (c == ones_lane) ? 1.f : 0.f;
        }
      }
    };
    if (flip) body(std::true_type{}); else body(std::false_type{});
    if (!(lo > 8.7e-19f && hi < 1.1e18f)) {     // 2^-60 .. 2^60
#pragma unroll
      for (int c = 0; c < CP; ++c) {
        if (c < C) {
          const int cs = flip ? C - 1 - c : c;
          const float4 k = s_k[cs];
          v[c] = (__ldg(s_base[cs] + pix) - k.x) / k.y;
        }
      }
    }
    if constexpr (PLANAR) {
      float* o = reinterpret_cast<float*>(out) + (n * C * Hp + yp) * Wp + xp;
#pragma unroll
      for (int c = 0; c < CP; ++c)
        if (c < C) o[static_cast<long long>(c) * HWp] = v[c];
    } else {
      float r[CP];
#pragma unroll
      for (int c = 0; c < CP; ++c) r[c] = round_for(v[c], (E*)nullptr);
      store_elems<E, CP>(out + (n * HWp + p) * CP, r);
    }
  }
}

template <typename E, bool PLANAR>
static cudaError_t fuse_launch(const float* lev, const float* emis, const float* mean, const float* stdv, const float* statics,
                               int S, E* out, long long N, int L, int H, int W, int Hp, int Wp, int mode, int c_pad,
                               int ones_lane, cudaStream_t s) {
  if (static_cast<long long>(Hp) * Wp > 0x7fffff00LL || static_cast<long long>(H) * W > 0x7fffff00LL) return cudaErrorInvalidValue;
  long long blocks = N * ((static_cast<long long>(Hp) * Wp + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks <= 0) return cudaSuccess;
  switch (c_pad) {
    case 16: fuse_kernel<E, 16, PLANAR><<<blocks, 256, 0, s>>>(lev, emis, mean, stdv, statics, S, out, N, L, H, W, Hp, Wp, mode, ones_lane); break;
    case 32: fuse_kernel<E, 32, PLANAR><<<blocks, 256, 0, s>>>(lev, emis, mean, stdv, statics, S, out, N, L, H, W, Hp, Wp, mode, ones_lane); break;
    case 48: fuse_kernel<E, 48, PLANAR><<<blocks, 256, 0, s>>>(lev, emis, mean, stdv, statics, S, out, N, L, H, W, Hp, Wp, mode, ones_lane); break;
    case 64: fuse_kernel<E, 64, PLANAR><<<blocks, 256, 0, s>>>(lev, emis, mean, stdv, statics, S, out, N, L, H, W, Hp, Wp, mode, ones_lane); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// planar fp32 output for up to 64 channels; more channels (never the case for this model) take 64 at a time
cudaError_t launch_fuse_inputs(const float* lev, const float* emis, const float* mean, const float* stdv,
                               const float* statics, int S, float* out, long long N, int L, int H, int W, int Hp, int Wp,
                               int mode, cudaStream_t s) {
  const int C = L + 1 + S;
  if (C > 64) return cudaErrorInvalidValue;
  return fuse_launch<float, true>(lev, emis, mean, stdv, statics, S, out, N, L, H, W, Hp, Wp, mode, (C + 15) / 16 * 16, -1, s);
}

template <typename E>
static cudaError_t fuse_bank(const float* lev, const float* emis, const float* mean, const float* stdv, const float* statics,
                             int S, E* out, long long N, int L, int H, int W, int Hp, int Wp, int mode, int c_pad,
                             int ones_lane, cudaStream_t s) {
  return fuse_launch<E, false>(lev, emis, mean, stdv, statics, S, out, N, L, H, W, Hp, Wp, mode, c_pad, ones_lane, s);
}
cudaError_t launch_fuse_inputs_bank(int dtype, const float* lev, const float* emis, const float* mean, const float* stdv,
                                    const float* statics, int S, void* out, long long N, int L, int H, int W, int Hp, int Wp,
                                    int mode, int c_pad, int ones_lane, cudaStream_t s) {
  if (dtype == NINT_BF16)
    return fuse_bank<__nv_bfloat16>(lev, emis, mean, stdv, statics, S, reinterpret_cast<__nv_bfloat16*>(out), N, L, H, W, Hp, Wp, mode, c_pad, ones_lane, s);
  return fuse_bank<float>(lev, emis, mean, stdv, statics, S, reinterpret_cast<float*>(out), N, L, H, W, Hp, Wp, mode, c_pad, ones_lane, s);
}

// ------------------------------------------------------------------------------------------
// Adjoint of the fusion (PLANAR layout): every source element gathers the padded positions fuse_kernel copied it to
// -- at most three rows (the upper halo row, the interior row, the lower halo row; in mode 1 the halo rows hold the
// element in channel C-1-c) times at most three columns (the interior column and its cyclic copies left and right) --
// and sums them in fp32 in increasing padded row, then padded column; z-scored channels then take one IEEE division by
// std (autograd of (v - mean) / std).  No atomics, nothing depends on the launch shape.
// Threads: one per (static channel, source pixel), running over the frames in order (one fp32 sum in frame, row,
// column order: d_statics is summed over every frame), then one per (frame, z-scored channel, source pixel).  The
// static threads come first so that their long loops start first.  A warp's threads are consecutive longitudes of one
// source row: every gathered load is a coalesced run (the cyclic wrap splits at most one).
// ------------------------------------------------------------------------------------------
struct AdjTaps {        // slots in increasing padded order: upper halo / interior / lower halo row; left / interior / right column
  long long row[3];     // element offset of the preimage row in its frame: (channel * Hp + yp) * Wp
  int col[3];
  bool row_ok[3], col_ok[3];
};

__device__ __forceinline__ AdjTaps adj_taps(int c, int C, int ys, int xs, int H, int W, int Hp, int Wp, int top, int bot,
                                           int left, int mode) {
  AdjTaps a;
  const int cf = mode == 0 ? c : C - 1 - c;   // channel of the element in the halo rows
  const int j = mode == 0 ? H - 2 - ys : ys - (H - bot - 1);
  a.row_ok[0] = ys >= 1 && ys <= top;         // upper halo: reflected row top - ys, or (mode 1) row ys - 1
  a.row[0] = (static_cast<long long>(cf) * Hp + (mode == 0 ? top - ys : ys - 1)) * Wp;
  a.row_ok[1] = true;
  a.row[1] = (static_cast<long long>(c) * Hp + top + ys) * Wp;
  a.row_ok[2] = j >= 0 && j < bot;            // lower halo: row top + H + j
  a.row[2] = (static_cast<long long>(cf) * Hp + top + H + j) * Wp;
  a.col_ok[0] = xs + left - W >= 0;
  a.col[0] = xs + left - W;
  a.col_ok[1] = true;
  a.col[1] = xs + left;
  a.col_ok[2] = xs + left + W < Wp;
  a.col[2] = xs + left + W;
  return a;
}

// adds the element's preimages in frame `f` (pointer to the frame) to acc, in padded row then column order; every load
// is issued before the first add
__device__ __forceinline__ float adj_gather(const float* __restrict__ f, const AdjTaps& a, float acc) {
  float v[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) v[i * 3 + k] = (a.row_ok[i] && a.col_ok[k]) ? __ldg(f + a.row[i] + a.col[k]) : 0.f;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k)
      if (a.row_ok[i] && a.col_ok[k]) acc += v[i * 3 + k];
  return acc;
}

__global__ void __launch_bounds__(256, 4) fuse_adjoint_kernel(const float* __restrict__ dframes, const float* __restrict__ stdv,
                                                           long long N, int L, int S, int H, int W, int Hp, int Wp,
                                                           int mode, float* __restrict__ d_lev,
                                                           float* __restrict__ d_emis, float* __restrict__ d_statics) {
  const int C = L + 1 + S;
  const long long HW = static_cast<long long>(H) * W;
  const long long frame = static_cast<long long>(C) * Hp * Wp;
  const int left = (Wp - W) / 2, top = (Hp - H) / 2, bot = Hp - H - top;
  const long long n_static = d_statics ? S * HW : 0;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx < n_static) {
    const int s = static_cast<int>(idx / HW);
    const int pix = static_cast<int>(idx - s * HW);
    const int ys = pix / W, xs = pix - ys * W;
    const AdjTaps a = adj_taps(L + 1 + s, C, ys, xs, H, W, Hp, Wp, top, bot, left, mode);
    float acc = 0.f;
#pragma unroll 2
    for (long long n = 0; n < N; ++n) acc = adj_gather(dframes + n * frame, a, acc);
    d_statics[idx] = acc;       // the fusion does not z-score the static attributes
    return;
  }
  const long long z = idx - n_static;
  if (z >= N * (L + 1) * HW) return;
  const long long pix = z % HW;
  const long long nc = z / HW;
  const int c = static_cast<int>(nc % (L + 1));
  const long long n = nc / (L + 1);
  float* out = c < L ? d_lev : d_emis;
  if (!out) return;
  const int ys = static_cast<int>(pix / W), xs = static_cast<int>(pix - static_cast<long long>(ys) * W);
  const AdjTaps a = adj_taps(c, C, ys, xs, H, W, Hp, Wp, top, bot, left, mode);
  const float g = __fdiv_rn(adj_gather(dframes + n * frame, a, 0.f), __ldg(stdv + c));
  if (c < L) d_lev[(n * L + c) * HW + pix] = g;
  else d_emis[n * HW + pix] = g;
}

cudaError_t launch_fuse_inputs_adjoint(const float* dframes, const float* stdv, long long N, int L, int S, int H, int W,
                                       int Hp, int Wp, int mode, float* d_lev, float* d_emis, float* d_statics,
                                       cudaStream_t s) {
  const long long HW = static_cast<long long>(H) * W;
  const long long items = (d_statics ? S * HW : 0) + ((d_lev || d_emis) ? N * (L + 1) * HW : 0);
  const long long blocks = (items + 255) / 256;
  if (blocks <= 0) return cudaSuccess;
  if (blocks > 0x7fffffffLL) return cudaErrorInvalidValue;
  fuse_adjoint_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(dframes, stdv, N, L, S, H, W, Hp, Wp, mode, d_lev,
                                                                   d_emis, d_statics);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// training loss (train.py:74-75,102,105): MSELoss(y, p) + L1Loss(y, p), both 'mean', on the cropped prediction
// pred[:, 0, y0:y1, x0:x1]; forward value and d loss / d pred in one pass.  stats = {sum (p-y)^2, sum |p-y|,
// sum y, sum y^2, blocks done}: the last block to finish turns them into the scalar loss (the two extra sums
// are what an on-device R^2, train.py:114, needs).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) loss_mse_l1_kernel(const float* __restrict__ pred, const float* __restrict__ y,
                                                          float* __restrict__ dpred, float* __restrict__ stats,
                                                          float* __restrict__ loss, int B, int H, int W, int y0, int y1,
                                                          int x0, int x1, const int* __restrict__ y_index, int y_offset,
                                                          long long y_frames) {
  const int hc = y1 - y0, wc = x1 - x0;
  const long long total = static_cast<long long>(B) * H * W;
  const float inv_n = 1.0f / (static_cast<float>(B) * hc * wc);
  float s2 = 0.f, s1 = 0.f, sy = 0.f, syy = 0.f;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(i % W);
    const long long r = i / W;
    const int yy = static_cast<int>(r % H);
    const long long b = r / H;
    float g = 0.f;
    if (yy >= y0 && yy < y1 && x >= x0 && x < x1) {
      // frame bank: the target of sample b is image y_index[b] + y_offset of y (dataset.py:600: y[i + seq_len - 1])
      const long long yb = y_index ? static_cast<long long>(__ldg(y_index + b)) + y_offset : b;
      // an out-of-range window index reads as a zero target instead of faulting (the input side reads zeros through TMA)
      const float t = (y_index && (yb < 0 || yb >= y_frames)) ? 0.f : y[(yb * hc + (yy - y0)) * wc + (x - x0)];
      const float d = pred[i] - t;
      s2 = fmaf(d, d, s2);
      s1 += fabsf(d);
      sy += t;
      syy = fmaf(t, t, syy);
      g = (2.f * d + (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f))) * inv_n;
    }
    if (dpred) dpred[i] = g;
  }
  __shared__ float red[4][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    sy += __shfl_xor_sync(0xffffffffu, sy, o);
    syy += __shfl_xor_sync(0xffffffffu, syy, o);
  }
  if (lane == 0) { red[0][warp] = s2; red[1][warp] = s1; red[2][warp] = sy; red[3][warp] = syy; }
  __syncthreads();
  if (threadIdx.x < 4) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += red[threadIdx.x][w];
    atomicAdd(stats + threadIdx.x, s);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const float done = atomicAdd(stats + 4, 1.0f);
    if (done == static_cast<float>(gridDim.x - 1)) {
      __threadfence();
      const volatile float* vs = stats;
      *loss = (vs[0] + vs[1]) * inv_n;
    }
  }
}
cudaError_t launch_loss_mse_l1(const float* pred, const float* y, float* dpred, float* stats, float* loss, int B, int H,
                               int W, int y0, int y1, int x0, int x1, const int* y_index, int y_offset, long long y_frames,
                               cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(stats, 0, 5 * sizeof(float), s);
  if (e != cudaSuccess) return e;
  loss_mse_l1_kernel<<<148, 256, 0, s>>>(pred, y, dpred, stats, loss, B, H, W, y0, y1, x0, x1, y_index, y_offset, y_frames);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Adam over one flat parameter buffer (train.py:71 torch.optim.Adam(lr, betas): no weight decay, no amsgrad).
// grad_scale folds the 1 / world_size of the data-parallel mean into the update.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, long long n, float lr, float beta1, float beta2,
                                                   float eps, float bc1, float bc2_sqrt, float grad_scale) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float gi = g[i] * grad_scale;
    const float mi = fmaf(beta1, m[i], (1.f - beta1) * gi);
    const float vi = fmaf(beta2, v[i], (1.f - beta2) * gi * gi);
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}
cudaError_t launch_adam(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                        float eps, int step, float grad_scale, cudaStream_t s) {
  const float bc1 = 1.f - powf(beta1, static_cast<float>(step));
  const float bc2_sqrt = sqrtf(1.f - powf(beta2, static_cast<float>(step)));
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  if (grid < 1) grid = 1;
  adam_kernel<<<grid, 256, 0, s>>>(p, g, m, v, n, lr, beta1, beta2, eps, bc1, bc2_sqrt, grad_scale);
  return cudaGetLastError();
}


// The same update with the step count and learning rate read from DEVICE memory, so a captured CUDA graph of the
// training step stays valid as both change: state = {step (as float), lr}.  adam_tick_kernel advances the step and
// derives the bias corrections once; the update kernel reads them.
__global__ void adam_tick_kernel(float* __restrict__ state, float beta1, float beta2) {
  const float step = state[0] + 1.f;
  state[0] = step;
  state[2] = 1.f - powf(beta1, step);            // bc1
  state[3] = sqrtf(1.f - powf(beta2, step));     // sqrt(bc2)
}
__global__ void __launch_bounds__(256) adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                       float* __restrict__ v, long long n, const float* __restrict__ state,
                                                       float beta1, float beta2, float eps, float grad_scale) {
  const float lr = state[1], bc1 = state[2], bc2_sqrt = state[3];
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float gi = g[i] * grad_scale;
    const float mi = fmaf(beta1, m[i], (1.f - beta1) * gi);
    const float vi = fmaf(beta2, v[i], (1.f - beta2) * gi * gi);
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}
cudaError_t launch_adam_dev(float* p, const float* g, float* m, float* v, long long n, float* state, float beta1,
                            float beta2, float eps, float grad_scale, cudaStream_t s) {
  adam_tick_kernel<<<1, 1, 0, s>>>(state, beta1, beta2);
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  if (grid < 1) grid = 1;
  adam_dev_kernel<<<grid, 256, 0, s>>>(p, g, m, v, n, state, beta1, beta2, eps, grad_scale);
  return cudaGetLastError();
}

}  // namespace nint
