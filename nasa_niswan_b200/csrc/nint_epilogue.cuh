// Epilogue of the implicit-GEMM gate convolution: TMEM accumulator -> fused ConvLSTM pointwise math, with
// every global-memory operand of the pointwise math staged through shared memory by TMA.
//
// Why staged: with one thread per pixel (the TMEM lane layout) a warp-wide global access touches 32
// different cache lines; ncu showed the direct version latency-bound on L1 miss tracking at ~35 % of HBM
// bandwidth (profiles/r1b).  Here a loader warp prefetches, per (pixel tile, 16-channel group), the boxes
// the math needs ([16 | 64 channels] x 8 x 16 pixels, swizzled so that the per-pixel 16-byte accesses of
// the epilogue threads are bank-conflict free), the 8 epilogue warps compute in place, and a storer warp
// writes the result boxes back with TMA stores.  TMA's out-of-image handling (zero fill on load, clipping
// on store) replaces every bounds check.
//
//   loader (warps 4/5) --e_full[s]--> math (warps 8-15) --st_ready[s]--> storer (warps 2/3) --e_empty[s]--> loader
#pragma once
#include "nint_common.cuh"
#include "nint_kernels.h"
#include "nint_pair.cuh"

namespace nint {

constexpr int kConvIoWarps = 8;     // warps 0-7: TMA producers / loaders / storers and the MMA issuer (nint_conv_halo.cu)
constexpr int kConvThreads = 512;   // warps 8-15: epilogue math
constexpr int kEpiMaxStages = 4;    // ring depth limit (epilogue stages / forward c slots)
constexpr int kEpiBoxBytes16 = kTilePixels * 16 * 4;   // 16 fp32 channels x 128 pixels = 8 KiB

// host-mapped post-mortem record of a timed-out step hand-off (armed by nint_debug_fail_record; null otherwise)
static __device__ unsigned long long* g_fail_host = nullptr;

// ---- timeline trace (debug_flags & 8): CTA 0 records clock64() stamps per role into a global buffer that
// tools/trace_report.py reads back through nint_debug_read_trace
constexpr int kTraceRoles = 8, kTraceLen = 1024;
__device__ long long g_trace[kTraceRoles * kTraceLen];
struct Tracer {
  long long* dst;
  int n;
  __device__ __forceinline__ Tracer(const ConvGemmParams& p, int role, bool on) {
    dst = (on && (NINT_DBG(p) & 8) && blockIdx.x == 0) ? g_trace + role * kTraceLen : nullptr;
    n = 0;
  }
  __device__ __forceinline__ void stamp() {
    if (dst && n < kTraceLen) dst[n++] = clock64();
  }
};

struct ItemCoord {
  int b, x0, y0;
};
__device__ __forceinline__ ItemCoord decode_tile(const ConvGemmParams& p, int tile) {
  ItemCoord c;
  const int tx = tile % p.tiles_x;
  int r = tile / p.tiles_x;
  const int ty = r % p.tiles_y;
  c.b = p.b0 + r / p.tiles_y;   // padding tiles of the last group: operand loads only (their epilogue I/O is skipped)
  c.x0 = tx * p.tile_w;
  c.y0 = ty * p.tile_h;
  return c;
}

// the tile after c in walk order (x fastest, then y, then the image)
__device__ __forceinline__ void next_tile(const ConvGemmParams& p, ItemCoord& c) {
  c.x0 += p.tile_w;
  if (c.x0 >= p.tiles_x * p.tile_w) {
    c.x0 = 0;
    c.y0 += p.tile_h;
    if (c.y0 >= p.tiles_y * p.tile_h) {
      c.y0 = 0;
      ++c.b;
    }
  }
}

// Work distribution.  The grid is `cpn * n_blocks` clusters (S = 1 or 2 CTAs each).  A cluster owns ONE
// n-block (N slice of the gate columns: its weights can stay resident in shared memory) and walks pixel-tile
// groups; the CTAs of a pair take adjacent groups of G tiles.
struct TileWalk {
  int nb, first_tile, tile_stride, tiles_padded, num_tiles;
  int tiles_step;   // padded tiles of ONE time step; tiles_padded = n_steps * tiles_step (time-fused launch: step-major walk)
};
__device__ __forceinline__ TileWalk make_walk(const ConvGemmParams& p, int S, int crank) {
  TileWalk w;
  const int G = p.group;
  w.num_tiles = p.B * p.tiles_x * p.tiles_y;
  const int groups = (w.num_tiles + S * G - 1) / (S * G);
  const int cpn = static_cast<int>(gridDim.x) / (S * p.n_blocks);
  const int cid = static_cast<int>(blockIdx.x) / S;
  w.nb = cid % p.n_blocks;
  w.first_tile = ((cid / p.n_blocks) * S + crank) * G;
  w.tile_stride = cpn * S * G;
  w.tiles_step = groups * S * G;
  w.tiles_padded = w.tiles_step * p.n_steps;
  return w;
}

// ---- time-fused launch (ConvGemmParams::n_steps > 1): position of a tile group inside the step-major walk, the slot a
// field has in that step, and the per-image hand-off between consecutive steps
struct GroupPos {
  int step, tile0;   // time step of the launch, first tile of the group inside that step
};
// walks the step-major tile sequence without divisions: bases only grow, so the step is advanced by comparison
template <bool FUSED>
struct StepCursor {
  int step, lo;   // current time step, first (padded) tile index of that step
  __device__ __forceinline__ StepCursor() : step(0), lo(0) {}
  __device__ __forceinline__ GroupPos at(const TileWalk& w, int base) {
    GroupPos g;
    if constexpr (FUSED) {
      while (base >= lo + w.tiles_step) {
        ++step;
        lo += w.tiles_step;
      }
      g.step = step;
      g.tile0 = base - lo;
    } else {
      g.step = 0;
      g.tile0 = base;
    }
    return g;
  }
  // (after at(base)) the walk's next group, base + stride, lies in another time step, or there is none
  __device__ __forceinline__ bool last_in_step(const TileWalk& w, int base) const {
    if constexpr (!FUSED) return false;
    const int nb = base + w.tile_stride;
    return nb >= w.tiles_padded || nb >= lo + w.tiles_step;
  }
};
template <bool FUSED>
__device__ __forceinline__ int step_slot(const ConvGemmParams& p, int slot, int d, int ring_bit, int step) {
  if constexpr (!FUSED) return slot;
  if (slot < 0) return slot;
  const int v = slot + d * step;
  return (p.ring_bits >> ring_bit) & 1 ? (v & 1) : v;
}
// whole warp (all lanes poll the same word): block until every tile of image b of the previous step has been stored.
// A wait that lasts ~2 s means a peer CTA is not resident or died: trap instead of hanging the GPU.  With debug flag 2048
// the limit is ~0.1 s and the wait is then abandoned after leaving a record (block, warp, step, image, count) in the
// trace buffer's last row (nint_debug_read_trace), so a dependency bug can be read back instead of killing the context.
__device__ __forceinline__ void wait_prev_step(const ConvGemmParams& p, int step, int b) {
  if (step == 0) return;
  const unsigned* ctr = p.step_done + static_cast<long long>(step - 1) * p.B + (b - p.b0);
  unsigned v;
  long long t0 = 0;
  unsigned spins = 0;
  const bool diag = (NINT_DBG(p) & 2048) != 0;
  for (;;) {
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
    if (v >= p.step_target) break;
    if (spins == 0) t0 = clock64();
    // (diagnostic mode: once one wait has been abandoned every other one gives up at once, so the launch ends quickly)
    if ((++spins & 0x3ff) == 0 &&
        (clock64() - t0 > (diag ? 200000000LL : 4000000000LL) ||
         (diag && *reinterpret_cast<volatile long long*>(g_trace + (kTraceRoles - 1) * kTraceLen) != 0))) {
      if (!diag) {
        // post-mortem in host-mapped memory (a trap destroys the context): plain stores, no function call -- a CALL in
        // a wait that is inlined into every role loop costs the hot loops their uniform registers (measured: forward
        // +22 %, wgrad +17 % when mbar_wait carried one)
        unsigned long long* h = g_fail_host;
        if (h && (threadIdx.x & 31) == 0) {
          h[1] = blockIdx.x;
          h[2] = threadIdx.x;
          h[3] = (static_cast<unsigned long long>(step) << 32) | static_cast<unsigned>(b);
          h[4] = v;
          h[0] = 3;
          __threadfence_system();
        }
        __syncwarp();
        __trap();
      }
      if ((threadIdx.x & 31) != 0) break;
      long long* row = g_trace + (kTraceRoles - 1) * kTraceLen;
      const unsigned long long i = atomicAdd(reinterpret_cast<unsigned long long*>(row), 1ULL);
      if (i < 200) {
        row[1 + 5 * i] = blockIdx.x;
        row[2 + 5 * i] = threadIdx.x >> 5;
        row[3 + 5 * i] = step;
        row[4 + 5 * i] = b;
        row[5 + 5 * i] = v;
      }
      break;
    }
  }
  // No proxy fence: the data was written by TMA stores and is about to be read by TMA loads -- async proxy on both
  // sides, through the L2 -- and only the counter goes through the generic proxy.  (fence.proxy.async compiles to
  // MEMBAR.ALL.GPU + FENCE.VIEW.ASYNC; see TileSignal for what gpu-scope membars did to this kernel.)
}
// whole warp (step and b are warp-uniform; every lane polls the same word: one request, no divergence).
// `seen`: (step, image) this warp checked last -- consecutive tiles of one image cost one look at the counter
template <bool FUSED>
__device__ __forceinline__ void wait_prev_step_warp(const ConvGemmParams& p, int step, int b, int& seen) {
  if constexpr (!FUSED) return;
  if (step == 0) return;
  const int key = step * p.B + (b - p.b0);
  if (key == seen) return;
  seen = key;
  wait_prev_step(p, step, b);
}
// Storer side of the hand-off (one lane): count a tile once this thread's TMA stores of it are complete (not only read).
// The counter update is a RELAXED reduction: the tile's data were written by this thread's own TMA stores, which
// cp.async.bulk.wait_group (without .read) has seen performed at the L2 -- the coherence point the consumers' TMA
// loads read from -- and the reduction is issued after it in program order.  No gpu-scope fence on either side:
// red.release.gpu / fence.acq_rel.gpu (SASS: MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR) made the CTA-pair backward kernel
// fail with "unspecified launch failure" on B200 whenever a cluster processed several tile groups per step, with or
// without the reduction after it, and fence.proxy.async (MEMBAR.ALL.GPU + FENCE.VIEW.ASYNC) still did so once in a few
// hundred training steps.  None of the kernel's bounded waits had fired (nint_debug_fail_record); compute-sanitizer
// and GPU core dumps are closed on this pool, so the cause is unknown.  The fence-free form has run 7 000 training
// steps at the BASELINE geometry without a failure and leaves bit-identical parameters after 400 deterministic
// steps (tools/fused_stress.py --det, NINT_FUSE_STEPS=0 / 2 / 3).
//
// Waiting for a tile's writes right after issuing them would idle the storer for the write latency once per tile, so
// the count of tile k is DEFERRED until tile k+1's stores have been committed (wait_group N: all but the N newest
// groups are complete) -- but only inside a time step: the next step's tiles may depend on this one, so the last tile
// a CTA has in a step is flushed at once.
template <bool FUSED>
struct TileSignal {
  int step, b;   // tile whose stores are committed but not yet counted (b < 0: none)
  __device__ __forceinline__ TileSignal() : step(0), b(-1) {}
  __device__ __forceinline__ void count(const ConvGemmParams& p) {
    unsigned* ctr = p.step_done + static_cast<long long>(step) * p.B + (b - p.b0);
    asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
    b = -1;
  }
  // a tile's stores have just been committed as `newest` bulk groups
  __device__ __forceinline__ void tile_done(const ConvGemmParams& p, int step_, int b_, int newest) {
    if constexpr (!FUSED) return;
    if (b >= 0) {
      if (newest <= 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
      else if (newest == 1) asm volatile("cp.async.bulk.wait_group 1;" ::: "memory");
      else if (newest == 2) asm volatile("cp.async.bulk.wait_group 2;" ::: "memory");
      else if (newest == 3) asm volatile("cp.async.bulk.wait_group 3;" ::: "memory");
      else asm volatile("cp.async.bulk.wait_group 4;" ::: "memory");
      count(p);
    }
    step = step_;
    b = b_;
  }
  __device__ __forceinline__ void flush(const ConvGemmParams& p) {
    if constexpr (!FUSED) return;
    if (b < 0) return;
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    count(p);
  }
};

// shared-memory address of 16-byte chunk `chunk` of pixel row `row` inside a TMA box with ROWB-byte rows
// (ROWB = 32 / 64 / 128 <-> SWIZZLE_32B / 64B / 128B: address bits [4,4+n) ^= bits [7,7+n)); base 1024-aligned
template <int ROWB>
__device__ __forceinline__ uint32_t swz(uint32_t base, int row, int chunk) {
  const uint32_t off = static_cast<uint32_t>(row * ROWB + chunk * 16);
  constexpr uint32_t mask = ROWB / 16 - 1;
  return base + (off ^ (((off >> 7) & mask) << 4));
}
__device__ __forceinline__ void sts128(uint32_t saddr, const float* v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
}
__device__ __forceinline__ void lds128u(uint32_t saddr, uint32_t* v) {
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(saddr));
}
__device__ __forceinline__ void sts128u(uint32_t saddr, const uint32_t* v) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
}
// 8 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// 5-D TMA store shared -> global (bulk async-group completion)
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2,
                                             int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// 8 channels of element type E at a swizzled row <-> 8 fp32 registers.  bf16: one 16-byte chunk of a row with
// ROWB bytes; fp32: two chunks.  `ec` = index of the 8-channel slice inside the row.
template <typename E, int ROWB>
__device__ __forceinline__ void lds8(uint32_t base, int row, int ec, float* v) {
  if constexpr (sizeof(E) == 2) {
    uint32_t u[4];
    lds128u(swz<ROWB>(base, row, ec), u);
#pragma unroll
    for (int j = 0; j < 4; ++j) unpack_bf16x2(u[j], v[2 * j], v[2 * j + 1]);
  } else {
    lds128(swz<ROWB>(base, row, 2 * ec), v);
    lds128(swz<ROWB>(base, row, 2 * ec + 1), v + 4);
  }
}
template <typename E, int ROWB>
__device__ __forceinline__ void sts8(uint32_t base, int row, int ec, const float* v) {
  if constexpr (sizeof(E) == 2) {
    uint32_t u[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) u[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
    sts128u(swz<ROWB>(base, row, ec), u);
  } else {
    sts128(swz<ROWB>(base, row, 2 * ec), v);
    sts128(swz<ROWB>(base, row, 2 * ec + 1), v + 4);
  }
}

// Geometry of one epilogue stage (one 16-channel group of one pixel tile), shared by the three roles.
//   gates : 64 q-columns (4 gates x 16 channels, contiguous in q-order) of E -> 128-byte rows, 1 (bf16) or 2 (fp32) boxes
//   fp32 state boxes (c, dc) : 16 channels -> 64-byte rows;   h : 16 channels of E -> 32- (bf16) or 64-byte rows
template <typename E>
struct EpiGeom {
  static constexpr int kGateBoxes = (64 * sizeof(E)) / 128;           // 1 / 2
  static constexpr int kGateBoxCols = 128 / sizeof(E);                // q columns per gates box: 64 / 32
  static constexpr int kGateBoxBytes = kTilePixels * 128;             // 16 KiB
  static constexpr int kGateBytes = kGateBoxes * kGateBoxBytes;
  static constexpr int kHRowB = 16 * sizeof(E);                       // 32 / 64
  static constexpr int kHBytes = kTilePixels * kHRowB;
};

// gate g (0..3 = i,f,g,o) of the 8-channel half `half` inside the staged gates box(es)
template <typename E>
__device__ __forceinline__ void lds_gate(uint32_t st, int row, int g, int half, float* v) {
  if constexpr (sizeof(E) == 2) lds8<E, 128>(st, row, g * 2 + half, v);
  else lds8<E, 128>(st + (g >> 1) * EpiGeom<E>::kGateBoxBytes, row, (g & 1) * 2 + half, v);
}
template <typename E>
__device__ __forceinline__ void sts_gate(uint32_t st, int row, int g, int half, const float* v) {
  if constexpr (sizeof(E) == 2) sts8<E, 128>(st, row, g * 2 + half, v);
  else sts8<E, 128>(st + (g >> 1) * EpiGeom<E>::kGateBoxBytes, row, (g & 1) * 2 + half, v);
}

// first q-column of the 16-channel group containing hidden channel `ch` (multiple of 16)
__device__ __forceinline__ int group_q0(int ch) { return (ch >> 4) * 64; }

template <int EPI>
__device__ __forceinline__ int epi_groups(const ConvGemmParams& p) {
  return (EPI == EPI_FWD ? p.hcb : p.hc) >> 4;
}

// ====================================================================================================
// Forward epilogue plumbing: TWO rings instead of one stage per channel group.
//   c ring  (p.c_ring slots x 8 KiB): c_{t-1} is prefetched into a slot (deep: hides the HBM latency of the only
//           load the forward epilogue has), updated in place by the math warps and stored back from there;
//   hg ring (p.e_stages x [gates 16 KiB | h 4 KiB]): outputs only.
// With a single ring the 28 KiB stage was held for load latency + math + store (~5000 cycles) and only two fit
// next to the resident weights; split, the c slots turn over in ~4000 cycles / 3 and the hg stages in ~2300 / 2.
//   loader (warp 4) --c_full--> math (warps 8-15) --c_ready--> c storer (warp 3) --c_empty--> loader
//                               math --hg_ready--> hg storer (warp 2) --hg_empty--> math
// ====================================================================================================
struct FwdEpiBars {
  uint64_t *c_full, *c_empty, *c_ready, *hg_ready, *hg_empty;
};
__device__ __forceinline__ uint8_t* fwd_c_slot(const ConvGemmParams& p, uint8_t* sE, int s) { return sE + s * kEpiBoxBytes16; }
__device__ __forceinline__ uint8_t* fwd_hg_stage(const ConvGemmParams& p, uint8_t* sE, int s) {
  return sE + p.c_ring * kEpiBoxBytes16 + s * p.e_stage_bytes;
}

template <typename E, bool FUSED>
__device__ __forceinline__ void fwd_c_loader(const ConvGemmParams& p, uint8_t* sE, const FwdEpiBars& b, const TileWalk& w) {
  const bool leader = elect_one();
  Tracer tr(p, 2, leader);
  const int G = p.group, ngroups = p.hcb >> 4;
  int s = 0, seen = -1;
  uint32_t ph = 0;
  StepCursor<FUSED> cur;
  for (int base = w.first_tile; base < w.tiles_padded; base += w.tile_stride) {
    const GroupPos gp = cur.at(w, base);
    const int slot_c_in = step_slot<FUSED>(p, p.slot_c_in, p.d_c_in, 2, gp.step);
    for (int gi = 0; gi < G; ++gi) {
      const int tile = gp.tile0 + gi;
      if (tile >= w.num_tiles) break;
      const ItemCoord c = decode_tile(p, tile);
      wait_prev_step_warp<FUSED>(p, gp.step, c.b, seen);   // c_{t-1} of this tile comes from the previous step of this launch
      for (int grp = 0; grp < ngroups; ++grp) {
        tr.stamp();
        mbar_wait(&b.c_empty[s], ph ^ 1);
        tr.stamp();
        if (leader) {
          if (p.slot_c_in >= 0) {
            mbar_arrive_expect_tx(&b.c_full[s], kEpiBoxBytes16);
            tma_load_5d(fwd_c_slot(p, sE, s), &p.tm_c, &b.c_full[s], w.nb * p.hcb + grp * 16, c.x0, c.y0, c.b, slot_c_in);
          } else {
            mbar_arrive(&b.c_full[s]);   // zero state: nothing to read, the slot is only an output buffer
          }
        }
        tr.stamp();
        if (++s == p.c_ring) {
          s = 0;
          ph ^= 1;
        }
      }
    }
  }
}

// kind 0: c slots (warp 3), kind 1: h + gates stages (warp 2)
template <typename E, bool FUSED>
__device__ __forceinline__ void fwd_storer(const ConvGemmParams& p, uint8_t* sE, const FwdEpiBars& b, const TileWalk& w, int kind) {
  using GE = EpiGeom<E>;
  const bool leader = elect_one();
  Tracer tr(p, 3, leader && kind == 1);
  const int G = p.group, ngroups = p.hcb >> 4;
  const int ring = kind == 0 ? p.c_ring : p.e_stages;
  uint64_t* ready = kind == 0 ? b.c_ready : b.hg_ready;
  uint64_t* empty = kind == 0 ? b.c_empty : b.hg_empty;
  int s = 0;
  uint32_t ph = 0;
  TileSignal<FUSED> sig;
  StepCursor<FUSED> cur;
  for (int base = w.first_tile; base < w.tiles_padded; base += w.tile_stride) {
    const GroupPos gp = cur.at(w, base);
    const int slot_c_out = step_slot<FUSED>(p, p.slot_c_out, p.d_c_out, 3, gp.step);
    const int slot_h_out = step_slot<FUSED>(p, p.slot_h_out, p.d_h_out, 4, gp.step);
    const int slot_g = step_slot<FUSED>(p, p.slot_g, p.d_g, 31, gp.step);
    for (int gi = 0; gi < G; ++gi) {
      const int tile = gp.tile0 + gi;
      if (tile >= w.num_tiles) break;
      const ItemCoord c = decode_tile(p, tile);
      for (int grp = 0; grp < ngroups; ++grp) {
        tr.stamp();
        mbar_wait(&ready[s], ph);
        tr.stamp();
        if (leader) {
          if (!(NINT_DBG(p) & 1)) {
            const int ch = w.nb * p.hcb + grp * 16;
            if (kind == 0) {
              tma_store_5d(&p.tm_c, fwd_c_slot(p, sE, s), ch, c.x0, c.y0, c.b, slot_c_out);
            } else {
              const uint8_t* st = fwd_hg_stage(p, sE, s);
              tma_store_5d(&p.tm_h, st + p.e_off_h, ch, c.x0, c.y0, c.b, slot_h_out);
              if (p.slot_g >= 0) {
                const int q0 = group_q0(ch);
#pragma unroll
                for (int bx = 0; bx < GE::kGateBoxes; ++bx)
                  tma_store_5d(&p.tm_g, st + bx * GE::kGateBoxBytes, q0 + bx * GE::kGateBoxCols, c.x0, c.y0, c.b, slot_g);
              }
            }
            tma_store_commit();
            tma_store_wait_read();   // the buffer may be overwritten once TMA has read it
          }
          mbar_arrive(&empty[s]);
        }
        tr.stamp();
        if (++s == ring) {
          s = 0;
          ph ^= 1;
        }
      }
      if (leader) sig.tile_done(p, gp.step, c.b, (NINT_DBG(p) & 1) ? 0 : ngroups);
    }
    if (leader && cur.last_in_step(w, base)) sig.flush(p);
  }
  if (leader) tma_store_wait_all();   // global writes complete before the CTA exits
}

template <typename E, bool FUSED>
__device__ __forceinline__ void fwd_math(const ConvGemmParams& p, int warp, int lane, uint32_t tmem_base, uint8_t* sE,
                                         const FwdEpiBars& b, uint64_t* tfull_bar, uint64_t* tempty_bar,
                                         const float* s_bias, const TileWalk& w, uint32_t tempty_remote) {
  using GE = EpiGeom<E>;
  constexpr int DT = ElemTraits<E>::kDtype;
  constexpr bool FAST = (DT == NINT_BF16);
  const int G = p.group, ngroups = p.hcb >> 4;
  const int quad = warp & 3;
  const int half = (warp - kConvIoWarps) >> 2;
  const int row = quad * 32 + lane;
  const bool skip = (NINT_DBG(p) & 1) != 0;
  Tracer tr(p, 4, warp == kConvIoWarps && lane == 0);
  int cs = 0, hs = 0;
  uint32_t cph = 0, hph = 0;
  int abuf = 0;
  uint32_t aphase = 0;
  StepCursor<FUSED> cur;
  for (int base = w.first_tile; base < w.tiles_padded; base += w.tile_stride) {
    bool waited = false;
    const GroupPos gp = cur.at(w, base);
    for (int gi = 0; gi < G; ++gi) {
      const int tile = gp.tile0 + gi;
      if (tile >= w.num_tiles) break;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                             static_cast<uint32_t>(abuf * p.acc_cols + gi * p.n_tile);
      for (int grp = 0; grp < ngroups; ++grp) {
        const uint32_t cslot = smem_u32(fwd_c_slot(p, sE, cs));
        const uint32_t st = smem_u32(fwd_hg_stage(p, sE, hs));
        tr.stamp();
        mbar_wait(&b.c_full[cs], cph);
        mbar_wait(&b.hg_empty[hs], hph ^ 1);
        tr.stamp();
        if (!waited) {
          mbar_wait(&tfull_bar[abuf], aphase);
          tc_fence_after();
          waited = true;
        }
        tr.stamp();
        // model.py:221-229.  accumulator columns of this group: grp*64 + gate*16 + channel
        float a[4][8], cn[8], hn[8];
#pragma unroll
        for (int g = 0; g < 4; ++g) tmem_ld8(taddr + grp * 64 + g * 16 + half * 8, a[g]);
        if (p.slot_c_in >= 0 && !skip) {
          lds8<float, 64>(cslot, row, half, cn);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) cn[j] = 0.f;
        }
        const uint32_t bq = smem_u32(s_bias + w.nb * p.n_tile + grp * 64 + half * 8);
        tmem_ld_wait();
        if (!skip) {
          if (p.bias_q) {   // null: the bias rides in the GEMM (weight row of the input's constant-1 lane, centre tap)
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float bias[8];
              lds128(bq + g * 64, bias);
              lds128(bq + g * 64 + 16, bias + 4);
#pragma unroll
              for (int j = 0; j < 8; ++j) a[g][j] += bias[j];
            }
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            // (the i, f, o pre-activations come out of the GEMM already halved: nint_pointwise.cu pack_w_fwd_kernel)
            const float gi_ = act_sigmoid_halved<FAST>(a[0][j]);
            const float gf = act_sigmoid_halved<FAST>(a[1][j]);
            const float gg = act_tanh<FAST>(a[2][j]);
            const float go = act_sigmoid_halved<FAST>(a[3][j]);
            const float cv = fmaf(cn[j], gf, gi_ * gg);
            cn[j] = cv;
            float hv = go * act_tanh<FAST>(cv);
            if constexpr (DT == NINT_TF32) hv = round_tf32(hv);  // h feeds the next step's tf32 MMA
            hn[j] = hv;
            a[0][j] = gi_; a[1][j] = gf; a[2][j] = gg; a[3][j] = go;
          }
          sts8<float, 64>(cslot, row, half, cn);
          sts8<E, GE::kHRowB>(st + p.e_off_h, row, half, hn);
          if (p.slot_g >= 0) {
#pragma unroll
            for (int g = 0; g < 4; ++g) sts_gate<E>(st, row, g, half, a[g]);
          }
        }
        // results visible to the async proxy (TMA store), then hand both buffers to their storers
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&b.c_ready[cs]);
          mbar_arrive(&b.hg_ready[hs]);
        }
        tr.stamp();
        if (++cs == p.c_ring) {
          cs = 0;
          cph ^= 1;
        }
        if (++hs == p.e_stages) {
          hs = 0;
          hph ^= 1;
        }
      }
    }
    if (!waited) {   // a group made only of padding tiles: still take part in the accumulator handshake
      mbar_wait(&tfull_bar[abuf], aphase);
      tc_fence_after();
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (tempty_remote) mbar_arrive_cluster(tempty_remote + abuf * 8); else mbar_arrive(&tempty_bar[abuf]);
    }
    if (++abuf == p.n_acc) {
      abuf = 0;
      aphase ^= 1;
    }
  }
}

// ------------------------------------------------------------------------------------ loader
// handles the channel groups whose running index n satisfies n % nwhich == which
template <typename E, int EPI, bool FUSED>
__device__ __forceinline__ void epi_loader(const ConvGemmParams& p, uint8_t* sE, uint64_t* e_full, uint64_t* e_empty,
                                           const TileWalk& w, int which, int nwhich) {
  using GE = EpiGeom<E>;
  const bool leader = elect_one();
  Tracer tr(p, 2, leader && which == 0);
  const int G = p.group;
  const int ngroups = epi_groups<EPI>(p);
  int s = 0, n = 0, seen = -1;
  uint32_t ph = 0;
  StepCursor<FUSED> cur;
  for (int base = w.first_tile; base < w.tiles_padded; base += w.tile_stride) {
    const GroupPos gp = cur.at(w, base);
    const int slot_g = step_slot<FUSED>(p, p.slot_g, p.d_g, 31, gp.step);
    const int slot_c_prev = (FUSED && gp.step == p.c_prev_none_step) ? -1 : step_slot<FUSED>(p, p.slot_c_prev, p.d_c_prev, 31, gp.step);
    for (int gi = 0; gi < G; ++gi) {
      const int tile = gp.tile0 + gi;
      if (tile >= w.num_tiles) break;
      const ItemCoord c = decode_tile(p, tile);
      wait_prev_step_warp<FUSED>(p, gp.step, c.b, seen);   // the running dc of this tile comes from the previous step of this launch
      for (int grp = 0; grp < ngroups; ++grp, ++n) {
        const bool mine = (nwhich == 1) || ((n % nwhich) == which);
        if (mine) tr.stamp();
        if (mine) mbar_wait(&e_empty[s], ph ^ 1);
        if (mine) tr.stamp();
        if (mine && leader) {
          uint8_t* st = sE + s * p.e_stage_bytes;
          uint64_t* bar = &e_full[s];
          const uint32_t bytes = GE::kGateBytes + kEpiBoxBytes16 * ((slot_c_prev >= 0) + (p.has_dc_in != 0));
          mbar_arrive_expect_tx(bar, bytes);
          const int q0 = group_q0(grp * 16);
#pragma unroll
          for (int bx = 0; bx < GE::kGateBoxes; ++bx)
            tma_load_5d(st + bx * GE::kGateBoxBytes, &p.tm_g, bar, q0 + bx * GE::kGateBoxCols, c.x0, c.y0, c.b, slot_g);
          // c_t is not read back: it is c_{t-1} f + i g of the values loaded here (model.py:228)
          if (slot_c_prev >= 0)
            tma_load_5d(st + p.e_off_c2, &p.tm_c, bar, grp * 16, c.x0, c.y0, c.b, slot_c_prev);
          if (p.has_dc_in) tma_load_5d(st + p.e_off_dc, &p.tm_dc, bar, grp * 16, c.x0, c.y0, c.b, 0);
        }
        if (mine) tr.stamp();
        if (++s == p.e_stages) {
          s = 0;
          ph ^= 1;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------ storer
// handles the channel groups whose running index n satisfies n % nwhich == which
template <typename E, int EPI, bool FUSED>
__device__ __forceinline__ void epi_storer(const ConvGemmParams& p, uint8_t* sE, uint64_t* st_ready, uint64_t* e_empty,
                                           const TileWalk& w, int which, int nwhich) {
  using GE = EpiGeom<E>;
  const bool leader = elect_one();
  Tracer tr(p, 3, leader && which == 0);
  const int G = p.group;
  const int ngroups = epi_groups<EPI>(p);
  int s = 0, n = 0;
  uint32_t ph = 0;
  TileSignal<FUSED> sig;
  StepCursor<FUSED> cur;
  for (int base = w.first_tile; base < w.tiles_padded; base += w.tile_stride) {
    const GroupPos gp = cur.at(w, base);
    const int slot_g = step_slot<FUSED>(p, p.slot_g, p.d_g, 31, gp.step);
    for (int gi = 0; gi < G; ++gi) {
      const int tile = gp.tile0 + gi;
      if (tile >= w.num_tiles) break;
      const ItemCoord c = decode_tile(p, tile);
      int committed = 0;   // bulk groups this warp commits for this tile
      for (int grp = 0; grp < ngroups; ++grp, ++n) {
        const bool mine = (nwhich == 1) || ((n % nwhich) == which);
        if (mine && !(NINT_DBG(p) & 1)) ++committed;
        if (mine) tr.stamp();
        if (mine) mbar_wait(&st_ready[s], ph);
        if (mine) tr.stamp();
        if (mine && leader) {
          const uint8_t* st = sE + s * p.e_stage_bytes;
          if (!(NINT_DBG(p) & 1)) {
            const int q0 = group_q0(grp * 16);
#pragma unroll
            for (int bx = 0; bx < GE::kGateBoxes; ++bx)
              tma_store_5d(&p.tm_g, st + bx * GE::kGateBoxBytes, q0 + bx * GE::kGateBoxCols, c.x0, c.y0, c.b, slot_g);
            tma_store_5d(&p.tm_dc, st + p.e_off_dc, grp * 16, c.x0, c.y0, c.b, 0);
            tma_store_commit();
            tma_store_wait_read();   // the stage may be overwritten once TMA has read it
          }
          mbar_arrive(&e_empty[s]);
        }
        if (mine) tr.stamp();
        if (++s == p.e_stages) {
          s = 0;
          ph ^= 1;
        }
      }
      if (leader) sig.tile_done(p, gp.step, c.b, committed);
    }
    if (leader && cur.last_in_step(w, base)) sig.flush(p);
  }
  if (leader) tma_store_wait_all();   // global writes complete before the CTA exits
}

// ------------------------------------------------------------------------------------ math (warps 8..15)
// TMEM lane quadrant = warp % 4 (hardware rule); the two warps of a quadrant take the two 8-channel halves
// of the 16-channel group.  `tempty_remote`: CTA-pair mode, shared::cluster address of the leader's tempty_bar[0].
template <typename E, int EPI, bool FUSED>
__device__ __forceinline__ void epi_math(const ConvGemmParams& p, int warp, int lane, uint32_t tmem_base, uint8_t* sE,
                                         uint64_t* e_full, uint64_t* st_ready, uint64_t* tfull_bar, uint64_t* tempty_bar,
                                         const float* s_bias, const float* s_headw, const TileWalk& w,
                                         uint32_t tempty_remote) {
  using GE = EpiGeom<E>;
  constexpr int DT = ElemTraits<E>::kDtype;
  constexpr bool FAST = (DT == NINT_BF16);
  const int G = p.group;
  const int ngroups = epi_groups<EPI>(p);
  const int quad = warp & 3;
  const int half = (warp - kConvIoWarps) >> 2;
  const int row = quad * 32 + lane;
  const bool skip = (NINT_DBG(p) & 1) != 0;
  Tracer tr(p, 4, warp == kConvIoWarps && lane == 0);
  int s = 0;
  uint32_t ph = 0;
  int abuf = 0;
  uint32_t aphase = 0;
  StepCursor<FUSED> cur;
  for (int base = w.first_tile; base < w.tiles_padded; base += w.tile_stride) {
    bool waited = (p.nseg == 0);
    const GroupPos gp = cur.at(w, base);
    const bool have_c_prev = p.slot_c_prev >= 0 && !(FUSED && gp.step == p.c_prev_none_step);
    for (int gi = 0; gi < G; ++gi) {
      const int tile = gp.tile0 + gi;
      if (tile >= w.num_tiles) break;
      const ItemCoord c = decode_tile(p, tile);
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                             static_cast<uint32_t>(abuf * p.acc_cols + gi * p.n_tile);
      float dpred = 0.f;
      if constexpr (EPI == EPI_BWD) {
        if (p.head_dpred) {
          const int y = c.y0 + (row >> 3), x = c.x0 + (row & 7);
          if (y < p.H && x < p.W)
            dpred = p.head_dpred[(FUSED ? gp.step * p.head_dpred_sstride : 0) + c.b * p.head_dpred_bstride + static_cast<long long>(y) * p.W + x];
        }
      }
      for (int grp = 0; grp < ngroups; ++grp) {
        const uint32_t st = smem_u32(sE + s * p.e_stage_bytes);
        tr.stamp();
        mbar_wait(&e_full[s], ph);
        tr.stamp();
        if (!waited) {
          mbar_wait(&tfull_bar[abuf], aphase);
          tc_fence_after();
          waited = true;
        }
        tr.stamp();
        {
        // SURVEY.md section 8 a10: gate backward; accumulator column c = dh_t[c] from the dgrad conv
        float gi_[8], gf[8], gg[8], go[8], cp[8], dc[8], dh[8];
        const int c0 = grp * 16 + half * 8;
        if (p.nseg > 0) {
          tmem_ld8(taddr + c0, dh);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) dh[j] = 0.f;
        }
        if (!skip) {
          lds_gate<E>(st, row, 0, half, gi_);
          lds_gate<E>(st, row, 1, half, gf);
          lds_gate<E>(st, row, 2, half, gg);
          lds_gate<E>(st, row, 3, half, go);
          if (have_c_prev) {
            lds8<float, 64>(st + p.e_off_c2, row, half, cp);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) cp[j] = 0.f;
          }
          if (p.has_dc_in) {
            lds8<float, 64>(st + p.e_off_dc, row, half, dc);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) dc[j] = 0.f;
          }
        }
        float hw[8];
        if (p.head_dpred) {
          lds128(smem_u32(s_headw + c0), hw);
          lds128(smem_u32(s_headw + c0 + 4), hw + 4);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) hw[j] = 0.f;
        }
        if (p.nseg > 0) tmem_ld_wait();
        if (p.dh_ext) {   // explicit upstream dh (cell API): one 32-byte read per thread, not a hot path
          const int y = c.y0 + (row >> 3), x = c.x0 + (row & 7);
          if (y < p.H && x < p.W) {
            float e[8];
            load_elems<float, 8>(p.dh_ext + ((static_cast<long long>(c.b) * p.H + y) * p.W + x) * p.hc + c0, e);
#pragma unroll
            for (int j = 0; j < 8; ++j) dh[j] += e[j];
          }
        }
        if (!skip) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float dhv = fmaf(dpred, hw[j], dh[j]);
            const float tc = act_tanh<FAST>(fmaf(cp[j], gf[j], gi_[j] * gg[j]));   // tanh(c_t), the forward's expression
            const float d_o = dhv * tc;
            const float dcv = fmaf(dhv * go[j], 1.f - tc * tc, dc[j]);
            const float d_i = dcv * gg[j];
            const float d_g = dcv * gi_[j];
            const float d_f = dcv * cp[j];
            dc[j] = dcv * gf[j];
            const float i_ = gi_[j], f_ = gf[j], g_ = gg[j], o_ = go[j];
            gi_[j] = d_i * fmaf(-i_, i_, i_);      // sigma' = s (1 - s) = s - s^2: one FFMA
            gf[j] = d_f * fmaf(-f_, f_, f_);
            gg[j] = d_g * fmaf(-g_, g_, 1.f);      // tanh' = 1 - g^2
            go[j] = d_o * fmaf(-o_, o_, o_);
          }
          if constexpr (DT == NINT_TF32) {
            // dgates are MMA operands of dgrad and wgrad: round to nearest tf32 (the MMA truncates).  The residuals
            // would be lost to the bias gradient (a plain, often nearly cancelling sum of dgates): reduce them over
            // the warp's 32 pixels with a butterfly that halves the values per lane at every step (31 shuffles for
            // 32 columns; lane l ends with column l = gate * 8 + channel) and keep them per channel group.
            float res[32];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float r;
              r = round_tf32(gi_[j]); res[j] = gi_[j] - r; gi_[j] = r;
              r = round_tf32(gf[j]); res[8 + j] = gf[j] - r; gf[j] = r;
              r = round_tf32(gg[j]); res[16 + j] = gg[j] - r; gg[j] = r;
              r = round_tf32(go[j]); res[24 + j] = go[j] - r; go[j] = r;
            }
            if (p.db_resid) {
#pragma unroll
              for (int st_ = 16; st_ >= 1; st_ >>= 1) {
                const bool upper = (lane & st_) != 0;
#pragma unroll
                for (int i = 0; i < st_; ++i) {
                  const float send = upper ? res[i] : res[i + st_];
                  const float keep = upper ? res[i + st_] : res[i];
                  res[i] = keep + __shfl_xor_sync(0xffffffffu, send, st_);
                }
              }
              // lane l owns column (gate = l >> 3, channel = half * 8 + (l & 7)) of this channel group; the slots are
              // private to (CTA, pixel quadrant): the read-modify-write needs no atomics and the sum order is fixed
              float* slot = p.db_resid + (static_cast<long long>(blockIdx.x) * 4 + quad) * (4 * p.hc);
              slot[grp * 64 + (lane >> 3) * 16 + half * 8 + (lane & 7)] += res[0];
            }
          }
          sts8<float, 64>(st + p.e_off_dc, row, half, dc);
          sts_gate<E>(st, row, 0, half, gi_);
          sts_gate<E>(st, row, 1, half, gf);
          sts_gate<E>(st, row, 2, half, gg);
          sts_gate<E>(st, row, 3, half, go);
        }
      
        }
        // results visible to the async proxy (TMA store), then hand the stage to the storer
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&st_ready[s]);
        tr.stamp();
        if (++s == p.e_stages) {
          s = 0;
          ph ^= 1;
        }
      }
    }
    if (p.nseg > 0) {
      if (!waited) {   // a group made only of padding items: still take part in the accumulator handshake
        mbar_wait(&tfull_bar[abuf], aphase);
        tc_fence_after();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        // pair mode: the MMA issuer lives in the leader CTA and waits for the epilogue warps of both CTAs
        if (tempty_remote) mbar_arrive_cluster(tempty_remote + abuf * 8); else mbar_arrive(&tempty_bar[abuf]);
      }
      if (++abuf == p.n_acc) {
        abuf = 0;
        aphase ^= 1;
      }
    }
  }
}

// dump the fp32 accumulators [B,H,W,n_blocks*n_tile] (nint_debug_raw_gates, dgrad, the tangent GEMM); ACC: add them to
// what the dump holds (every element belongs to one thread of the launch: a plain read-add-write)
template <bool ACC>
__device__ __forceinline__ void epi_raw(const ConvGemmParams& p, int warp, int lane, uint32_t tmem_base,
                                        uint64_t* tfull_bar, uint64_t* tempty_bar, const TileWalk& w,
                                        uint32_t tempty_remote) {
  const int G = p.group;
  const int quad = warp & 3;
  const int half = (warp - kConvIoWarps) >> 2;
  const int row = quad * 32 + lane;
  int abuf = 0;
  uint32_t aphase = 0;
  for (int base = w.first_tile; base < w.tiles_padded; base += w.tile_stride) {
    mbar_wait(&tfull_bar[abuf], aphase);
    tc_fence_after();
    for (int gi = 0; gi < G; ++gi) {
      const int tile = base + gi;
      if (tile >= w.num_tiles) break;
      const ItemCoord c = decode_tile(p, tile);
      const int y = c.y0 + (row >> 3), x = c.x0 + (row & 7);
      const bool valid = y < p.H && x < p.W;
      const long long pix = (static_cast<long long>(c.b) * p.H + y) * p.W + x;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                             static_cast<uint32_t>(abuf * p.acc_cols + gi * p.n_tile);
      float* ro = p.raw_out + pix * (p.n_blocks * p.n_tile) + w.nb * p.n_tile;
      for (int c0 = half * 16; c0 < p.n_tile; c0 += 32) {
        float v[16];
        tmem_ld16(taddr + c0, v);
        tmem_ld_wait();
        if constexpr (ACC) {
          if (valid) {
            float o[16];
            load_elems<float, 16>(ro + c0, o);
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] += o[j];
          }
        }
        if (valid) store_elems<float, 16>(ro + c0, v);
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (tempty_remote) mbar_arrive_cluster(tempty_remote + abuf * 8); else mbar_arrive(&tempty_bar[abuf]);
    }
    if (++abuf == p.n_acc) {
      abuf = 0;
      aphase ^= 1;
    }
  }
}

}  // namespace nint
