// Implicit-GEMM gate convolution, "halo" variant (sm_100a): the activation tile is loaded ONCE
// per 64-byte channel chunk, with its k//2 halo, and every tap reads it in place.
//
// The pixel tile is 8 wide x 16 tall.  A halo chunk is (8+2p) x (16+2p) pixels x 64 bytes, written
// by one 5-D TMA box (zero fill outside the image = the conv's zero padding, model.py:204-211).
// For tap (dy, dx) the UMMA A operand is the same buffer seen through a shifted descriptor: start
// address + (dy*(8+2p) + dx) * 64 bytes, 8-row groups (one tile row of 8 pixels) strided by
// SBO = (8+2p) * 64 bytes.  TMA's SWIZZLE_64B and the UMMA SW64 layout both derive the 16-byte
// chunk permutation from shared-memory address bits [7,9) (verified on hardware: the descriptor
// base-offset field must stay 0), so a row-shifted view stays consistent.
//
// CTA pair (cluster of 2, tcgen05 cta_group::2): measured on B200 (tools/micro/mma_rate*.cu) a
// single-CTA M=128 MMA costs 171 / 110 / 88 cycles at N = 256 / 128 / 64 -- a ~60-cycle fixed cost
// per instruction -- while the pair MMA (M=256: 128 pixels from each CTA) runs at the nominal floor
// (128 / 64 / 43 cycles for BOTH SMs).  In pair mode the two CTAs walk different pixel tiles in
// lockstep; each loads its own halo tiles and HALF of every weight stage (rows [r*N/2, (r+1)*N/2)),
// which also halves the weight bytes every SM has to ingest.  The leader CTA (rank 0) issues the MMAs;
// "full" barriers live in the leader (both CTAs' TMA loads complete_tx on them), "empty"/accumulator
// barriers are signalled in both CTAs by multicast tcgen05.commit.
//
// Item groups: G consecutive tiles (G * n_tile <= 256 columns) are accumulated side by side in one
// TMEM buffer and share every weight stage.
//
// Warp roles (16 warps): 0 / 7 activation TMA producers, 6 weight TMA producer, 1 MMA issuer, 2 / 3 epilogue TMA
// stores (2 also allocates TMEM), 4 / 5 epilogue TMA loads, 8-15 epilogue math (nint_epilogue.cuh).
#include "nint_epilogue.cuh"

namespace nint {

constexpr int kHaloCtrlBytes = 1024;
constexpr int kHaloMaxA = 12;
constexpr int kHaloMaxW = 28;
constexpr int kMaxAcc = 4;       // TMEM accumulator buffers (512 columns / acc_cols, at most 4)

__host__ __device__ inline int halo_rows(int ksize) { return (8 + (ksize & ~1)) * (16 + (ksize & ~1)); }
static inline int halo_a_buf_bytes(const ConvGemmParams& p) {
  int m = 0;
  for (int s = 0; s < p.nseg; ++s) {
    const int b = halo_rows(p.seg[s].ksize) * kChunkBytes;
    if (b > m) m = b;
  }
  return (m + 511) & ~511;   // SWIZZLE_64B atoms are 512 bytes: halo buffers only need that alignment
}

static int halo_operand_bytes(int a_buf_bytes, int na, int n_tile, int nw, int ts, int cluster) {
  return (na * a_buf_bytes + nw * ts * (n_tile / cluster) * kChunkBytes + 1023) & ~1023;
}
int conv_halo_smem_bytes(const ConvGemmParams& p) {
  return 1024 + halo_operand_bytes(p.a_buf_bytes, p.na_bufs, p.n_tile, p.num_stages, p.taps_per_stage, p.cluster) +
         p.e_stages * p.e_stage_bytes + p.c_ring * kEpiBoxBytes16 + kHaloCtrlBytes + (4 * p.hc + p.hc) * 4;
}

__device__ __forceinline__ int halo_operand_bytes_dev(int a_buf_bytes, int na, int stage_bytes, int nw) {
  return (na * a_buf_bytes + nw * stage_bytes + 1023) & ~1023;
}

// FUSED: time-fused launch (ConvGemmParams::n_steps > 1).  A template parameter, not a run-time test: the hand-off code
// in every role loop cost the one-launch-per-step forward kernel 19 % when it was merely branched around.
template <typename E, int EPI, bool PAIR, bool FUSED>
__global__ void __launch_bounds__(kConvThreads, 1) conv_halo_kernel(const __grid_constant__ ConvGemmParams p) {
  constexpr int DT = ElemTraits<E>::kDtype;
  constexpr int CE = ElemTraits<E>::kPerChunk;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // broadcast from lane 0: tells the compiler these are warp-uniform, so role loops and descriptor
  // arithmetic live in uniform registers instead of per-thread registers + R2UR moves
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  constexpr int S = PAIR ? 2 : 1;               // 1: single CTA, 2: CTA pair (cta_group::2)
  constexpr bool pair = PAIR;
  const int NA = p.na_bufs, NW = p.num_stages, TS = p.taps_per_stage;
  const int w_rows = p.n_tile / S;              // weight rows (of N) this CTA holds
  const int w_bytes = w_rows * kChunkBytes;     // one tap of one chunk, this CTA's share
  const int stage_bytes = TS * w_bytes;         // a weight stage holds up to TS consecutive taps
  uint8_t* sA = smem;
  uint8_t* sW = sA + NA * p.a_buf_bytes;
  uint8_t* sE = smem + halo_operand_bytes_dev(p.a_buf_bytes, NA, stage_bytes, NW);   // epilogue I/O stages
  uint8_t* ctrl = sE + p.e_stages * p.e_stage_bytes + p.c_ring * kEpiBoxBytes16;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(ctrl);
  uint64_t* a_empty = a_full + kHaloMaxA;
  uint64_t* w_full = a_empty + kHaloMaxA;
  uint64_t* w_empty = w_full + kHaloMaxW;
  uint64_t* tfull_bar = w_empty + kHaloMaxW;
  uint64_t* tempty_bar = tfull_bar + kMaxAcc;
  uint64_t* e_full = tempty_bar + kMaxAcc;
  uint64_t* e_empty = e_full + kEpiMaxStages;
  uint64_t* st_ready = e_empty + kEpiMaxStages;
  uint64_t* hg_ready = st_ready + kEpiMaxStages;   // forward only: h + gates output stages
  uint64_t* hg_empty = hg_ready + kEpiMaxStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ctrl + kHaloCtrlBytes - 16);
  float* s_bias = reinterpret_cast<float*>(ctrl + kHaloCtrlBytes);
  float* s_headw = s_bias + 4 * p.hc;

  uint32_t crank = 0;
  if constexpr (pair) crank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);
  const bool lead_cta = crank == 0;
  // work unit of a CTA iteration = G consecutive tiles ("tile group") accumulated side by side in one
  // TMEM buffer and sharing every weight stage; the two CTAs of a pair take adjacent groups
  const int G = p.group;
  const TileWalk walk = make_walk(p, S, static_cast<int>(crank));
  const bool resident = p.w_resident != 0;   // the whole weight slice of this n-block fits: load it once
  // forward, resident 3x3 weights: TWO warps issue MMAs (alternate chunks).  The issuing thread only runs a few MMAs
  // ahead of the tensor pipe, so one issuer loses its ~500 cycles of per-chunk barrier work as tensor idle time;
  // with two, one warp's waits and commits hide behind the other's MMA stream.
  int chunks_per_tile = 0;
  bool all_k3 = true;
  for (int s = 0; s < p.nseg; ++s) {
    chunks_per_tile += p.seg[s].nchunks;
    all_k3 = all_k3 && p.seg[s].ksize == 3;
  }
  const bool dual = EPI == EPI_FWD && resident && G == 1 && all_k3 && TS == 9 && NA >= 4 && !(NINT_DBG(p) & 32);
  volatile uint32_t* mma_started = reinterpret_cast<volatile uint32_t*>(ctrl + kHaloCtrlBytes - 32);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.nseg; ++s) {
      prefetch_tensormap(&p.seg[s].tmap_act);
      prefetch_tensormap(&p.seg[s].tmap_w);
    }
  }
  if (warp == 3 && lane == 0 && !epi_is_raw(EPI)) {
    prefetch_tensormap(&p.tm_c);
    prefetch_tensormap(&p.tm_g);
    prefetch_tensormap(EPI == EPI_FWD ? &p.tm_h : &p.tm_dc);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NA; ++s) {
      mbar_init(&a_full[s], 1);
      mbar_init(&a_empty[s], 1);
    }
    for (int s = 0; s < NW; ++s) {
      mbar_init(&w_full[s], 1);
      mbar_init(&w_empty[s], 1);
    }
    *mma_started = 0;
    for (int s = 0; s < kMaxAcc; ++s) {
      mbar_init(&tfull_bar[s], (dual && chunks_per_tile >= 2) ? 2 : 1);   // one commit per issuing warp
      mbar_init(&tempty_bar[s], 8 * S);   // the leader waits for the epilogue warps of both CTAs
    }
    for (int s = 0; s < kEpiMaxStages; ++s) {
      mbar_init(&e_full[s], 1);
      mbar_init(&e_empty[s], 1);
      mbar_init(&st_ready[s], 8);         // one arrive per epilogue warp
      mbar_init(&hg_ready[s], 8);
      mbar_init(&hg_empty[s], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (pair) {
      tmem_alloc_pair(tmem_slot, kTmemCols);
    } else {
      tmem_alloc(tmem_slot, kTmemCols);
      tmem_relinquish();
    }
  }
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch) touches no
  // global data, so a CTA of this launch may run it on an SM the previous conv launch of the stream has already left
  // while that launch's last tiles are still in flight elsewhere.  launch_dependents lets the NEXT launch do the same
  // with us; wait blocks until the previous launch has completed and its writes are visible.
  if (p.pdl) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
  }
  if (EPI == EPI_FWD) {
    for (int i = threadIdx.x; i < 4 * p.hc; i += kConvThreads) s_bias[i] = p.bias_q ? p.bias_q[i] : 0.f;
  }
  if (EPI == EPI_BWD) {
    for (int i = threadIdx.x; i < p.hc; i += kConvThreads) s_headw[i] = p.head_w ? p.head_w[i] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (pair) cluster_sync_all();   // the peer's barriers are initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  // ------------------------------------------------------------------ operand TMA producers (both CTAs)
  // Every bulk-async instruction keeps its issuing warp busy for ~440-750 cycles whatever its size, and the
  // cost is per warp, not per SM (tools/micro/tma_rate.cu): the loads are spread over several warps.
  //   a_par / a_npar: this warp issues the activation chunks whose running index c satisfies c % a_npar == a_par,
  //                   or, with by_tile (G == 2), the box of tile a_par of EVERY chunk (halves the time from a free
  //                   halo buffer to its "full" barrier)
  //   do_w: this warp issues the weight stages
  auto produce = [&](bool do_a, int a_par, int a_npar, bool do_w) {
    const bool by_tile = do_a && a_npar == 2 && G == 2;
    const bool leader = elect_one();
    Tracer tr(p, do_w ? 5 : 0, leader && (do_w || a_par == 0));
    int ia = 0, iw = 0, cc = 0, seen = -1;
    uint32_t pa = 0, pw = 0;
    bool first = true;
    StepCursor<FUSED> cur;
    for (int base = walk.first_tile; base < walk.tiles_padded; base += walk.tile_stride) {
      const GroupPos gp = cur.at(walk, base);
      // tiles [g_begin, g_end) of the group are this warp's; the first one is decoded once per group (two divisions),
      // the following ones by stepping the coordinates (next_tile): nothing but adds in front of the TMA issue
      const int g_begin = by_tile ? a_par : 0, g_end = by_tile ? a_par + 1 : G;
      ItemCoord c_first;
      c_first.b = c_first.x0 = c_first.y0 = 0;
      if (do_a) c_first = decode_tile(p, gp.tile0 + g_begin);
      if (FUSED && do_a && gp.step > 0) {
        // time-fused launch: the recurrent operand (h_{t-1} / dgates_{t+1}, with its halo) of these tiles was written by
        // the previous step of THIS launch
        ItemCoord cw = c_first;
        for (int g = g_begin; g < g_end; ++g, next_tile(p, cw))
          if (gp.tile0 + g < walk.num_tiles) wait_prev_step_warp<FUSED>(p, gp.step, cw.b, seen);
      }
      for (int s = 0; s < p.nseg; ++s) {
        const ConvSegment& sg = p.seg[s];
        const int seg_slot = step_slot<FUSED>(p, sg.slot, p.d_seg[s], s, gp.step);
        const int pad = sg.ksize >> 1;
        const int taps = sg.ksize * sg.ksize;
        const uint32_t a_bytes = static_cast<uint32_t>(halo_rows(sg.ksize) * kChunkBytes);
        // weights: 3-D map (element, row of the N tile, chunk-tap index); one box = this CTA's rows of TS taps
        int wtap = (walk.nb * sg.nchunks) * taps;
        for (int ch = 0; ch < sg.nchunks; ++ch, ++cc, wtap += taps) {
          if (do_a && (a_npar == 1 || by_tile || (cc & 1) == a_par)) {   // a_npar is 1 or 2
            tr.stamp();
            mbar_wait(&a_empty[ia], pa ^ 1);
            tr.stamp();
            if (leader) {
              // "full" barriers live in the leader CTA and count the bytes of both CTAs' loads
              if (lead_cta && (!by_tile || a_par == 0)) mbar_arrive_expect_tx(&a_full[ia], a_bytes * G * S);
              uint32_t bar = 0;
              if constexpr (pair) bar = mapa_rank(smem_u32(&a_full[ia]), 0);
              ItemCoord cg = c_first;
              for (int g = g_begin; g < g_end; ++g, next_tile(p, cg)) {
                uint8_t* dst = sA + ia * p.a_buf_bytes + g * p.a_halo_bytes;
                int img = cg.b, slot = seg_slot;
                if (sg.win_start) {   // frame bank: image b of step `slot` is frame win_start[b] + slot (OOB frame = zeros)
                  img = (gp.tile0 + g < walk.num_tiles) ? __ldg(sg.win_start + cg.b) + seg_slot : sg.bank_frames;
                  slot = 0;
                }
                if constexpr (pair)
                  tma_load_5d_pair(dst, &sg.tmap_act, bar, ch * CE, cg.x0 - pad, cg.y0 - pad, img, slot);
                else
                  tma_load_5d(dst, &sg.tmap_act, &a_full[ia], ch * CE, cg.x0 - pad, cg.y0 - pad, img, slot);
              }
            }
            tr.stamp();
          }
          if (++ia == NA) {
            ia = 0;
            pa ^= 1;
          }
          if (!do_w || (resident && !first)) continue;   // resident weights are loaded once
          for (int tap0 = 0; tap0 < taps; tap0 += sg.ts) {   // sg.ts divides taps (conv_halo_plan)
            if (!resident) mbar_wait(&w_empty[iw], pw ^ 1);
            if (leader) {
              if (lead_cta) mbar_arrive_expect_tx(&w_full[iw], static_cast<uint32_t>(sg.ts * w_bytes * S));
              uint8_t* dst = sW + iw * stage_bytes;   // a weight stage is ONE box (all TS taps)
              if constexpr (pair)
                tma_load_3d_pair(dst, &sg.tmap_w, mapa_rank(smem_u32(&w_full[iw]), 0), 0, static_cast<int>(crank) * w_rows, wtap + tap0);
              else
                tma_load_3d(dst, &sg.tmap_w, &w_full[iw], 0, 0, wtap + tap0);
            }
            if (++iw == NW) {
              iw = 0;
              pw ^= 1;
            }
          }
        }
      }
      first = false;
    }
  };
  // ------------------------------------------------------------------ dual MMA issuer (see `dual` above)
  auto issue_dual = [&](int which) {
    const bool leader = elect_one();
    Tracer tr(p, 1, leader && which == 0);
    const bool issue_any = !(NINT_DBG(p) & 2);
    const int n_acc = p.n_acc, acc_cols = p.acc_cols, a_buf_bytes = p.a_buf_bytes;
    const uint32_t idesc = p.idesc;
    const uint32_t w16l = static_cast<uint32_t>(w_bytes >> 4);
    const uint32_t sA_addr = smem_u32(sA), sW_addr = smem_u32(sW);
    const int ntiles = (walk.tiles_padded - walk.first_tile + walk.tile_stride - 1) / walk.tile_stride;
    const int cpt = chunks_per_tile;
    const int total = walk.first_tile < walk.tiles_padded ? ntiles * cpt : 0;
    const uint64_t adesc0 = make_smem_desc_sw64(0, 16, 10 * kChunkBytes);   // 3x3: halo pitch 10 pixels
    const uint64_t bdesc0 = make_smem_desc_sw64(0, 16, 512);
    const uint32_t ahi = static_cast<uint32_t>(adesc0 >> 32), bhi = static_cast<uint32_t>(bdesc0 >> 32);
    // running indices of chunk c (advanced by two chunks per iteration, no divisions in the loop): tile k of this CTA,
    // chunk j inside the tile, halo buffer ia / phase pa, accumulator buffer abuf / phase aphase
    int k = which / cpt, j = which % cpt, ia = which % NA, abuf = k % n_acc;
    uint32_t pa = static_cast<uint32_t>(which / NA) & 1u, aphase = static_cast<uint32_t>(k / n_acc) & 1u;
    for (int c = which; c < total; c += 2) {
      tr.stamp();
      if (j == 0) mbar_wait(&tempty_bar[abuf], aphase ^ 1);
      mbar_wait(&a_full[ia], pa);
      if (k == 0) mbar_wait(&w_full[j], 0);            // resident weights arrive during the first tile
      // chunks enter the tensor pipe strictly in order (deterministic accumulation order, and the tile's first
      // MMA with accumulate = 0 precedes the rest): wait until the other warp has issued all of chunk c-1
      spin_until_at_least(mma_started, static_cast<uint32_t>(c));
      tc_fence_after();
      tr.stamp();
      const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(abuf * acc_cols);
      if (leader && issue_any) {
        const uint32_t alo = static_cast<uint32_t>(adesc0) + ((sA_addr + ia * a_buf_bytes) >> 4);
        const uint32_t blo = static_cast<uint32_t>(bdesc0) + ((sW_addr + j * stage_bytes) >> 4);
#pragma unroll 1
        for (int dy = 0; dy < 3; ++dy) {
          const uint32_t ar = alo + static_cast<uint32_t>(dy * 10 * (kChunkBytes >> 4));
          const uint32_t br = blo + static_cast<uint32_t>(dy * 3) * w16l;
#pragma unroll
          for (int dxc = 0; dxc < 3; ++dxc) {
            const uint32_t acc = (j | dy | dxc) == 0 ? 0u : 1u;
            umma_lohi<DT, pair>(d_tmem, ar + 4 * dxc, ahi, br + dxc * w16l, bhi, idesc, acc);
            umma_lohi<DT, pair>(d_tmem, ar + 4 * dxc + 2, ahi, br + dxc * w16l + 2, bhi, idesc, 1u);
          }
        }
      }
      if (leader) {
        __threadfence_block();
        *mma_started = static_cast<uint32_t>(c + 1);   // chunk c fully issued
      }
      __syncwarp();
      umma_commit_elect<pair>(&a_empty[ia]);
      if (j + 2 >= cpt) umma_commit_elect<pair>(&tfull_bar[abuf]);   // this warp's last chunk of the tile
      tr.stamp();
      j += 2;
      while (j >= cpt) {
        j -= cpt;
        ++k;
        if (++abuf == n_acc) {
          abuf = 0;
          aphase ^= 1;
        }
      }
      ia += 2;
      if (ia >= NA) {
        ia -= NA;
        pa ^= 1;
      }
    }
  };

  // two activation producers when a tile needs many chunk loads (dgrad: K = 4*hc channels, G tiles per chunk)
  const bool a_split = !epi_is_raw(EPI);   // one producer warp cannot issue a box per 1152-cycle chunk (timeline: 670 cycles per box + waits)

  if (warp == 0) {
    if (p.nseg > 0) produce(true, 0, a_split ? 2 : 1, false);
  } else if (warp == 7) {
    if (p.nseg > 0 && a_split) produce(true, 1, 2, false);
  } else if (warp == 6) {
    if (p.nseg > 0) produce(false, 0, 1, true);
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    // The loop body between two tcgen05.mma must stay a handful of uniform-datapath instructions: every kernel
    // parameter it needs is hoisted into a local, descriptors advance by adds (timeline traces showed ~190
    // cycles per MMA of pure issue overhead before, against 64-cycle MMAs).
    if (p.nseg > 0 && lead_cta && dual) {
      issue_dual(0);
    } else if (p.nseg > 0 && lead_cta) {
      const bool leader = elect_one();
      Tracer tr(p, 1, leader);
      const bool issue_any = !(NINT_DBG(p) & 2);
      const int n_acc = p.n_acc, acc_cols = p.acc_cols, nseg = p.nseg, a_buf_bytes = p.a_buf_bytes;
      const uint32_t idesc = p.idesc;
      const uint32_t n_tile = static_cast<uint32_t>(p.n_tile);
      const uint64_t a_halo16 = static_cast<uint64_t>(p.a_halo_bytes >> 4);
      const uint64_t w16 = static_cast<uint64_t>(w_bytes >> 4);
      const uint32_t sA_addr = smem_u32(sA), sW_addr = smem_u32(sW);
      // The K walk of all tiles is one flat sequence of activation chunks.  Barrier round trips cost ~100 cycles
      // each and the tensor pipe's instruction queue is shallow, so the readiness of the NEXT chunk (and of the
      // next tile's accumulator) is awaited before the current chunk's MMAs are issued: between the last MMA of
      // one chunk and the first of the next there is only the tcgen05.commit.
      int cbase = walk.first_tile, cs = 0, cch = 0;
      bool valid = cbase < walk.tiles_padded;
      int ia = 0, iw = 0;
      uint32_t pa = 0, pw = 0;
      int abuf = 0;
      uint32_t aphase = 0;
      bool first = true;
      // with fewer than 3 halo buffers the next chunk cannot be in flight while the current one is consumed:
      // then each chunk is awaited just before its own MMAs
      const bool lookahead = NA >= 3;
      // streaming weights with one stage per chunk: the next chunk's stage is awaited ahead as well
      bool single_stage = true;
      for (int s = 0; s < nseg; ++s) single_stage = single_stage && (p.seg[s].ts == p.seg[s].ksize * p.seg[s].ksize);
      const bool w_ahead = lookahead && !resident && NW >= 3 && single_stage;
      // cur_ready: the current chunk's barriers were already awaited (by the previous iteration's look-ahead)
      bool cur_ready = false;
      int step_hi = walk.tiles_step;
      if (valid && lookahead) {
        mbar_wait(&tempty_bar[abuf], aphase ^ 1);
        mbar_wait(&a_full[ia], pa);
        if (w_ahead) mbar_wait(&w_full[0], 0);
        tc_fence_after();
        cur_ready = true;
      }
      while (valid) {
        // ---- successor of the current chunk
        int nbase = cbase, ns = cs, nch = cch + 1;
        if (nch == p.seg[cs].nchunks) {
          nch = 0;
          if (++ns == nseg) {
            ns = 0;
            nbase += walk.tile_stride;
          }
        }
        const bool nvalid = nbase < walk.tiles_padded;
        const bool last_of_tile = nbase != cbase;
        const int nia = (ia + 1 == NA) ? 0 : ia + 1;
        const uint32_t npa = (ia + 1 == NA) ? pa ^ 1 : pa;
        int nabuf = abuf;
        uint32_t naphase = aphase;
        if (last_of_tile && ++nabuf == n_acc) {
          nabuf = 0;
          naphase ^= 1;
        }
        // 3x3 single-stage chunks take these waits BETWEEN the tap rows of the MMA stream (fast path below): the
        // issuing thread only runs a few MMAs ahead of the tensor pipe, so a 300-cycle block of waits between two
        // chunks idles the pipe, while three ~100-cycle pieces hide behind the rows already issued
        const bool fast = lookahead && issue_any && p.seg[cs].ksize == 3 && p.seg[cs].ts == 9 && G == 2 && (resident || w_ahead);
        // time-fused launch: the first tile group of the NEXT time step is loaded only after other CTAs have finished
        // tiles of this step -- possibly tiles that wait, symmetrically, on this CTA's current one.  Its barriers must
        // not be awaited before the current chunk (the last of this step here) has been issued.
        bool cross = false;
        if constexpr (FUSED) {
          if (last_of_tile) {
            while (cbase >= step_hi) step_hi += walk.tiles_step;   // step_hi: end of the step cbase lies in
            cross = nvalid && (nbase >= step_hi || (NINT_DBG(p) & 4096));
          }
        }
        const bool look = lookahead && !cross;
        tr.stamp();
        if (!cur_ready) {
          if ((cs | cch) == 0) mbar_wait(&tempty_bar[abuf], aphase ^ 1);
          mbar_wait(&a_full[ia], pa);
          if (w_ahead) mbar_wait(&w_full[iw], pw);
          tc_fence_after();
        }
        if (look && !fast && nvalid) {
          if (last_of_tile) mbar_wait(&tempty_bar[nabuf], naphase ^ 1);
          mbar_wait(&a_full[nia], npa);
          if (w_ahead) {
            // the next chunk's single weight stage is the ring slot after the current one
            const int niw = (iw + 1 == NW) ? 0 : iw + 1;
            mbar_wait(&w_full[niw], (iw + 1 == NW) ? pw ^ 1 : pw);
          }
          tc_fence_after();
        }
        cur_ready = look && nvalid;
        tr.stamp();
        // ---- issue the current chunk
        const int ks = p.seg[cs].ksize;
        const int hw = 8 + (ks & ~1);            // halo row pitch in pixels
        const uint32_t sbo = static_cast<uint32_t>(hw * kChunkBytes);
        const int taps = ks * ks;
        const uint64_t row_skip = static_cast<uint64_t>((hw - ks) * (kChunkBytes >> 4));
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(abuf * acc_cols);
        uint32_t accumulate = (cs | cch) != 0 ? 1u : 0u;
        if (resident && (cs | cch) == 0) iw = 0;   // stage index = position inside the tile's K walk
        // tap (dy, dx) = the halo buffer seen through a row-shifted descriptor: start address advances by one
        // pixel (64 B) per tap and skips the rest of the halo row when dx wraps
        uint64_t adesc = make_smem_desc_sw64(sA_addr + ia * a_buf_bytes, 16, sbo);
        int dx = 0;
        if (fast) {
          if (resident && first) {
            mbar_wait(&w_full[iw], pw);
            tc_fence_after();
          }
          const uint64_t bdesc = make_smem_desc_sw64(sW_addr + iw * stage_bytes, 16, 512);
          const uint32_t alo = static_cast<uint32_t>(adesc), blo = static_cast<uint32_t>(bdesc);
          const uint32_t ahi = static_cast<uint32_t>(adesc >> 32), bhi = static_cast<uint32_t>(bdesc >> 32);
          const uint32_t w16l = static_cast<uint32_t>(w16);
          const uint32_t halo16l = static_cast<uint32_t>(a_halo16);
          const uint32_t d1 = d_tmem + n_tile;
          // one tap row: descriptor offsets inside a row are compile-time constants (one pixel = 64 B apart), rows
          // are one halo pitch (10 pixels) apart
          auto issue_row = [&](int dy) {
            if (leader) {
              const uint32_t ar = alo + static_cast<uint32_t>(dy * 10 * (kChunkBytes >> 4));
              const uint32_t br = blo + static_cast<uint32_t>(dy * 3) * w16l;
              if (G == 1) {
#pragma unroll
                for (int dxc = 0; dxc < 3; ++dxc) {
                  const uint32_t acc = (dy | dxc) == 0 ? accumulate : 1u;
                  umma_lohi<DT, pair>(d_tmem, ar + 4 * dxc, ahi, br + dxc * w16l, bhi, idesc, acc);
                  umma_lohi<DT, pair>(d_tmem, ar + 4 * dxc + 2, ahi, br + dxc * w16l + 2, bhi, idesc, 1u);
                }
              } else {
#pragma unroll
                for (int dxc = 0; dxc < 3; ++dxc) {
                  const uint32_t acc = (dy | dxc) == 0 ? accumulate : 1u;
                  umma_lohi<DT, pair>(d_tmem, ar + 4 * dxc, ahi, br + dxc * w16l, bhi, idesc, acc);
                  umma_lohi<DT, pair>(d1, ar + halo16l + 4 * dxc, ahi, br + dxc * w16l, bhi, idesc, acc);
                  umma_lohi<DT, pair>(d_tmem, ar + 4 * dxc + 2, ahi, br + dxc * w16l + 2, bhi, idesc, 1u);
                  umma_lohi<DT, pair>(d1, ar + halo16l + 4 * dxc + 2, ahi, br + dxc * w16l + 2, bhi, idesc, 1u);
                }
              }
            }
            __syncwarp();
          };
          issue_row(0);
          if (look && nvalid && last_of_tile) mbar_wait(&tempty_bar[nabuf], naphase ^ 1);
          issue_row(1);
          if (look && nvalid) {
            mbar_wait(&a_full[nia], npa);
            if (w_ahead) mbar_wait(&w_full[(iw + 1 == NW) ? 0 : iw + 1], (iw + 1 == NW) ? pw ^ 1 : pw);
            tc_fence_after();
          }
          issue_row(2);
          if (!resident) umma_commit_elect<pair>(&w_empty[iw]);
          if (++iw == NW) {
            iw = 0;
            pw ^= 1;
          }
        } else
        for (int tap0 = 0, tsc = p.seg[cs].ts; tap0 < taps; tap0 += tsc) {   // tsc: taps per weight stage of this segment
          if ((!resident || first) && !w_ahead) {
            mbar_wait(&w_full[iw], pw);
            tc_fence_after();
          }
          const uint64_t bdesc = make_smem_desc_sw64(sW_addr + iw * stage_bytes, 16, 512);
          if (leader && issue_any) {
            // single-lane region: the tcgen05.mma stream of one weight stage.  Only the low descriptor words move.
            uint32_t alo = static_cast<uint32_t>(adesc), blo = static_cast<uint32_t>(bdesc);
            const uint32_t ahi = static_cast<uint32_t>(adesc >> 32), bhi = static_cast<uint32_t>(bdesc >> 32);
            const uint32_t w16l = static_cast<uint32_t>(w16), skipl = static_cast<uint32_t>(row_skip);
            int dxl = dx;
            if (G == 1) {
#pragma unroll 3
              for (int j = 0; j < tsc; ++j) {
                umma_lohi<DT, pair>(d_tmem, alo, ahi, blo, bhi, idesc, accumulate);
                umma_lohi<DT, pair>(d_tmem, alo + 2, ahi, blo + 2, bhi, idesc, 1u);
                accumulate = 1;
                blo += w16l;
                alo += kChunkBytes >> 4;
                if (++dxl == ks) {
                  dxl = 0;
                  alo += skipl;
                }
              }
            } else if (G == 2) {
              const uint32_t halo16l = static_cast<uint32_t>(a_halo16);
              const uint32_t d1 = d_tmem + n_tile;
#pragma unroll 3
              for (int j = 0; j < tsc; ++j) {
                umma_lohi<DT, pair>(d_tmem, alo, ahi, blo, bhi, idesc, accumulate);
                umma_lohi<DT, pair>(d1, alo + halo16l, ahi, blo, bhi, idesc, accumulate);
                umma_lohi<DT, pair>(d_tmem, alo + 2, ahi, blo + 2, bhi, idesc, 1u);
                umma_lohi<DT, pair>(d1, alo + halo16l + 2, ahi, blo + 2, bhi, idesc, 1u);
                accumulate = 1;
                blo += w16l;
                alo += kChunkBytes >> 4;
                if (++dxl == ks) {
                  dxl = 0;
                  alo += skipl;
                }
              }
            } else {
              const uint32_t halo16l = static_cast<uint32_t>(a_halo16);
              for (int j = 0; j < tsc; ++j) {
                uint32_t a2 = alo;
                uint32_t d = d_tmem;
                for (int g = 0; g < G; ++g, a2 += halo16l, d += n_tile) {
                  umma_lohi<DT, pair>(d, a2, ahi, blo, bhi, idesc, accumulate);
                  umma_lohi<DT, pair>(d, a2 + 2, ahi, blo + 2, bhi, idesc, 1u);
                }
                accumulate = 1;
                blo += w16l;
                alo += kChunkBytes >> 4;
                if (++dxl == ks) {
                  dxl = 0;
                  alo += skipl;
                }
              }
            }
          }
          __syncwarp();
          accumulate = 1;
          if (!resident) umma_commit_elect<pair>(&w_empty[iw]);
          if (++iw == NW) {
            iw = 0;
            pw ^= 1;
          }
          // advance the warp-uniform descriptor past this stage's TS taps
          const int adv = dx + tsc;
          adesc += static_cast<uint64_t>(tsc * (kChunkBytes >> 4)) + static_cast<uint64_t>(adv / ks) * row_skip;
          dx = adv % ks;
        }
        umma_commit_elect<pair>(&a_empty[ia]);
        if (last_of_tile) {
          umma_commit_elect<pair>(&tfull_bar[abuf]);
          first = false;
        }
        tr.stamp();
        ia = nia; pa = npa; abuf = nabuf; aphase = naphase;
        cbase = nbase; cs = ns; cch = nch;
        valid = nvalid;
      }
    }
  } else if (warp == 2 || warp == 3) {
    // ------------------------------------------------------------------ epilogue TMA stores
    // backward: the two warps alternate channel groups; forward: warp 3 stores c, warp 2 stores h + gates
    if constexpr (EPI == EPI_BWD) epi_storer<E, EPI, FUSED>(p, sE, st_ready, e_empty, walk, warp - 2, 2);
    if constexpr (EPI == EPI_FWD) fwd_storer<E, FUSED>(p, sE, FwdEpiBars{e_full, e_empty, st_ready, hg_ready, hg_empty}, walk, warp == 3 ? 0 : 1);
  } else if (warp == 4 || warp == 5) {
    // ------------------------------------------------------------------ epilogue TMA loads
    // backward: 4 boxes per channel group, two loaders alternate groups; forward: one box per group, warp 4 only
    if constexpr (EPI == EPI_BWD) epi_loader<E, EPI, FUSED>(p, sE, e_full, e_empty, walk, warp - 4, 2);
    if constexpr (EPI == EPI_FWD) {
      if (warp == 4) fwd_c_loader<E, FUSED>(p, sE, FwdEpiBars{e_full, e_empty, st_ready, hg_ready, hg_empty}, walk);
      if (warp == 5 && p.nseg > 0 && lead_cta && dual) issue_dual(1);   // second MMA issuer
    }
  } else if (warp >= kConvIoWarps) {
    // ------------------------------------------------------------------ epilogue math (warps 8-15)
    // the epilogue of either CTA releases the accumulator buffer on the LEADER's "tmem empty" barrier
    uint32_t tempty_remote = 0;
    if constexpr (pair) tempty_remote = mapa_rank(smem_u32(&tempty_bar[0]), 0);
    if constexpr (epi_is_raw(EPI))
      epi_raw<EPI == EPI_RAW_ACC>(p, warp, lane, tmem_base, tfull_bar, tempty_bar, walk, tempty_remote);
    else if constexpr (EPI == EPI_FWD)
      fwd_math<E, FUSED>(p, warp, lane, tmem_base, sE, FwdEpiBars{e_full, e_empty, st_ready, hg_ready, hg_empty}, tfull_bar,
                  tempty_bar, s_bias, walk, tempty_remote);
    else
      epi_math<E, EPI, FUSED>(p, warp, lane, tmem_base, sE, e_full, st_ready, tfull_bar, tempty_bar, s_bias, s_headw, walk,
                       tempty_remote);
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (pair) cluster_sync_all();   // no CTA may exit (or free TMEM) while its peer still uses the pair's resources
  if (warp == 2) {
    tc_fence_after();
    if constexpr (pair) tmem_dealloc_pair(tmem_base, kTmemCols); else tmem_dealloc(tmem_base, kTmemCols);
  }
}

// shared-memory plan: epilogue I/O stages, tiles per group, taps per weight stage, stage / halo-buffer counts
int conv_halo_plan(int epi, int dtype, ConvGemmParams& p) {
  const int esize = dtype == NINT_BF16 ? 2 : 4;
  // ---- epilogue stage layout (nint_epilogue.cuh): backward [gates][c_{t-1}][dc], forward [gates][h] + c ring
  const int gate_bytes = kTilePixels * 64 * esize;
  p.c_ring = 0;
  if (epi == EPI_FWD) {
    // forward: output stages [gates][h] plus a separate ring of c slots (nint_epilogue.cuh)
    const int g = p.slot_g >= 0 ? gate_bytes : 0;
    p.e_off_h = g;
    p.e_off_c = p.e_off_c2 = p.e_off_dc = 0;
    p.e_stage_bytes = (g + kTilePixels * 16 * esize + 1023) & ~1023;
    p.c_ring = 3;
  } else if (epi == EPI_BWD) {
    p.e_off_c = p.e_off_c2 = gate_bytes;
    p.e_off_dc = p.e_off_c2 + kEpiBoxBytes16;
    p.e_off_h = 0;
    p.e_stage_bytes = p.e_off_dc + kEpiBoxBytes16;
  } else {
    p.e_off_c = p.e_off_c2 = p.e_off_dc = p.e_off_h = 0;
    p.e_stage_bytes = 0;
  }
  p.a_halo_bytes = halo_a_buf_bytes(p);
  if (p.a_halo_bytes == 0) p.a_halo_bytes = 1024;
  const int total = 227 * 1024 - 1024 - kHaloCtrlBytes - (4 * p.hc + p.hc) * 4 - 1024 - p.c_ring * kEpiBoxBytes16;
  const int w_bytes = (p.n_tile / p.cluster) * kChunkBytes;
  const int ns_max = epi_is_raw(epi) ? 0 : (epi == EPI_FWD ? 2 : 3), ns_min = epi_is_raw(epi) ? 0 : 2;
  int max_k = 1;
  for (int s = 0; s < p.nseg; ++s) if (p.seg[s].ksize > max_k) max_k = p.seg[s].ksize;
  // ---- plan A: weights resident.  One stage per (segment, chunk) holding all taps; needs >= 3 halo buffers.
  if (p.nseg > 0) {
    int n_st = 0, ts = p.seg[0].ksize * p.seg[0].ksize;
    bool same_k = true;
    for (int s = 0; s < p.nseg; ++s) {
      n_st += p.seg[s].nchunks;
      same_k = same_k && (p.seg[s].ksize * p.seg[s].ksize == ts);
    }
    const long long res_bytes = static_cast<long long>(n_st) * ts * w_bytes;
    if (same_k && n_st <= kHaloMaxW) {
      for (int ns = ns_max; ns >= ns_min; --ns) {
        const long long rem = static_cast<long long>(total) - ns * p.e_stage_bytes - res_bytes;
        if (rem < 3LL * p.a_halo_bytes) continue;
        p.w_resident = 1;
        p.e_stages = ns;
        p.group = 1;
        p.a_buf_bytes = p.a_halo_bytes;
        p.na_bufs = static_cast<int>(rem / p.a_halo_bytes) > 6 ? 6 : static_cast<int>(rem / p.a_halo_bytes);
        p.taps_per_stage = ts;
        for (int s = 0; s < p.nseg; ++s) p.seg[s].ts = ts;
        p.num_stages = n_st;
        p.acc_cols = p.n_tile;
        p.n_acc = 512 / p.acc_cols > kMaxAcc ? kMaxAcc : 512 / p.acc_cols;
        return 0;
      }
    }
  }
  // ---- plan B: weights stream through a ring of stages.
  p.w_resident = 0;
  // tiles per group: fill one 256-column accumulator buffer, at most 4 (2 for the memory-bound backward
  // epilogue, whose stages need the shared memory more than the weight stages need the reuse)
  int gmax = 256 / p.n_tile;
  if (gmax > (epi == EPI_BWD ? 2 : 4)) gmax = (epi == EPI_BWD ? 2 : 4);
  if (gmax < 1 || p.nseg == 0) gmax = 1;
  // taps per weight stage: every barrier round trip of the MMA-issuing thread costs ~100 cycles and every TMA box
  // ~450-750 cycles of its producer warp, so a stage should carry all taps of a chunk when it fits
  int want = (1536 + p.n_tile - 1) / p.n_tile;
  if (want > max_k * max_k) want = max_k * max_k;
  // per segment: the largest divisor of its tap count that is <= cand (segments of one launch can have different
  // kernel sizes -- the dgrad of a layer reads its own dgates through k_l and the layer above's through k_{l+1});
  // a stage is sized for the largest of them
  auto seg_ts = [&](int s, int cand) {
    const int taps = p.seg[s].ksize * p.seg[s].ksize;
    int t = cand < taps ? cand : taps;
    while (taps % t) --t;
    return t;
  };
  auto stage_ts = [&](int cand) {
    int m = 1;
    for (int s = 0; s < p.nseg; ++s) if (seg_ts(s, cand) > m) m = seg_ts(s, cand);
    return m;
  };
  // preference order: >= 3 halo buffers (the MMA issuer waits one chunk ahead) with 3 weight stages of `want` taps,
  // first with three epilogue stages then two; after that relax the tap count, then the group size, then the buffers
  int NS = -1, G = 1, ts = 1, min_na = 3;
  if (p.plan_g > 0 && p.plan_g < gmax) gmax = p.plan_g;               // experiment knobs (NINT_PLAN_G / NINT_PLAN_NS)
  const int ns_hi = (p.plan_ns >= ns_min && p.plan_ns <= ns_max) ? p.plan_ns : ns_max;
  for (int pass = 0; pass < 2 && NS < 0; ++pass, min_na = 2)
    for (int cand = want; cand >= 1 && NS < 0; --cand) {
      if (cand < want && stage_ts(cand) == stage_ts(cand + 1)) continue;   // same plan as the previous candidate
      for (int g = gmax; g >= 1 && NS < 0; --g)
        for (int ns = ns_hi; ns >= ns_min; --ns)
          if (total - ns * p.e_stage_bytes >= min_na * g * p.a_halo_bytes + 3 * stage_ts(cand) * w_bytes) {
            NS = ns;
            G = g;
            ts = stage_ts(cand);
            for (int s = 0; s < p.nseg; ++s) p.seg[s].ts = seg_ts(s, cand);
            break;
          }
    }
  if (NS < 0) return 1;
  p.e_stages = NS;
  p.group = G;
  p.a_buf_bytes = G * p.a_halo_bytes;
  p.acc_cols = G * p.n_tile;
  p.n_acc = 512 / p.acc_cols > kMaxAcc ? kMaxAcc : 512 / p.acc_cols;
  const int budget = total - NS * p.e_stage_bytes;
  int nw = 3;
  int na = (budget - nw * ts * w_bytes) / p.a_buf_bytes;
  if (na > 6) na = 6;
  if (na < 1) na = 1;
  nw = (budget - na * p.a_buf_bytes) / (ts * w_bytes);
  if (nw > kHaloMaxW) nw = kHaloMaxW;
  if (nw < 1) return 1;
  p.na_bufs = na;
  p.taps_per_stage = ts;
  p.num_stages = nw;
  return 0;
}

template <typename E, int EPI, bool PAIR, bool FUSED>
static cudaError_t launch_h(const ConvGemmParams& p, int num_sms, cudaStream_t stream) {
  const int smem = conv_halo_smem_bytes(p);
  if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(conv_halo_kernel<E, EPI, PAIR, FUSED>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  constexpr int S = PAIR ? 2 : 1;
  const int tiles = p.B * p.tiles_x * p.tiles_y;
  const int groups = (tiles + S * p.group - 1) / (S * p.group) * (p.n_steps > 1 ? p.n_steps : 1);
  int cpn = num_sms / (S * p.n_blocks);   // clusters per n-block
  if (cpn > groups) cpn = groups;
  if (cpn <= 0) return cudaErrorInvalidConfiguration;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cpn * p.n_blocks * S);
  cfg.blockDim = dim3(kConvThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (PAIR) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = S;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (FUSED) {
    // CTAs of a time-fused launch wait for each other's tiles: every one of them must be resident at once
    static int max_units = -1;   // co-resident CTAs (single) / clusters (pair) of this instantiation at this smem size
    static int max_units_smem = -1, max_units_dev = -1;   // ... on this device
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return cudaErrorInvalidDevice;
    if (max_units < 0 || max_units_smem != smem || max_units_dev != dev) {
      int n = 0;
      cudaError_t e;
      if (PAIR) {
        cfg.attrs = attr;
        cfg.numAttrs = na;
        e = cudaOccupancyMaxActiveClusters(&n, conv_halo_kernel<E, EPI, PAIR, FUSED>, &cfg);
      } else {
        int per_sm = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, conv_halo_kernel<E, EPI, PAIR, FUSED>, kConvThreads, smem);
        n = per_sm * num_sms;
      }
      if (e != cudaSuccess) return e;
      max_units = n;
      max_units_smem = smem;
      max_units_dev = dev;
    }
    if (cpn * p.n_blocks > max_units) cpn = max_units / p.n_blocks;
    if (cpn <= 0) return cudaErrorInvalidConfiguration;
    cfg.gridDim = dim3(cpn * p.n_blocks * S);
  }
  if (p.pdl) {   // may start while the previous kernel of the stream drains (the kernel calls griddepcontrol.wait)
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, conv_halo_kernel<E, EPI, PAIR, FUSED>, p);
}

template <typename E, bool PAIR>
static cudaError_t launch_e(int epi, const ConvGemmParams& p, int num_sms, cudaStream_t stream) {
  const bool fused = p.n_steps > 1;
  if (epi == EPI_FWD) return fused ? launch_h<E, EPI_FWD, PAIR, true>(p, num_sms, stream) : launch_h<E, EPI_FWD, PAIR, false>(p, num_sms, stream);
  if (epi == EPI_BWD) return fused ? launch_h<E, EPI_BWD, PAIR, true>(p, num_sms, stream) : launch_h<E, EPI_BWD, PAIR, false>(p, num_sms, stream);
  if (fused) return cudaErrorInvalidValue;
  if (epi == EPI_RAW_ACC) return launch_h<E, EPI_RAW_ACC, PAIR, false>(p, num_sms, stream);
  return launch_h<E, EPI_RAW, PAIR, false>(p, num_sms, stream);
}

cudaError_t launch_conv_halo(int epi, int dtype, const ConvGemmParams& p, int num_sms, cudaStream_t stream) {
  if (p.tile_w != 8 || p.tile_h != 16) return cudaErrorInvalidValue;
  if (p.cluster != 1 && p.cluster != 2) return cudaErrorInvalidValue;
  if (p.cluster == 2 && (p.n_tile % 32)) return cudaErrorInvalidValue;
  if (p.n_acc < 1 || p.n_acc > kMaxAcc || p.n_acc * p.acc_cols > kTmemCols) return cudaErrorInvalidValue;
  if (!epi_is_raw(epi) && (p.e_stages < 2 || p.e_stages > kEpiMaxStages)) return cudaErrorInvalidValue;
  if (dtype == NINT_BF16)
    return p.cluster == 2 ? launch_e<__nv_bfloat16, true>(epi, p, num_sms, stream)
                          : launch_e<__nv_bfloat16, false>(epi, p, num_sms, stream);
  return p.cluster == 2 ? launch_e<float, true>(epi, p, num_sms, stream) : launch_e<float, false>(epi, p, num_sms, stream);
}

// debug: arm (first call) and read the host-mapped post-mortem record of the time-fused step hand-off (wait_prev_step);
// readable after a trap has destroyed the context
cudaError_t fail_record(unsigned long long* out5) {
  static unsigned long long* host = nullptr;
  if (!host) {
    cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&host), 64, cudaHostAllocMapped);
    if (e != cudaSuccess) return e;
    for (int i = 0; i < 8; ++i) host[i] = 0;
    unsigned long long* dev = nullptr;
    e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&dev), host, 0);
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(g_fail_host, &dev, sizeof(dev));
    if (e != cudaSuccess) return e;
  }
  for (int i = 0; i < 5; ++i) out5[i] = reinterpret_cast<volatile unsigned long long*>(host)[i];
  return cudaSuccess;
}

// debug: copy the timeline trace of CTA 0 (see Tracer) to the host
cudaError_t read_trace(long long* host, int n) {
  if (n > kTraceRoles * kTraceLen) n = kTraceRoles * kTraceLen;
  return cudaMemcpyFromSymbol(host, g_trace, static_cast<size_t>(n) * sizeof(long long));
}
cudaError_t clear_trace() {
  static long long zeros[kTraceRoles * kTraceLen] = {0};
  return cudaMemcpyToSymbol(g_trace, zeros, sizeof(zeros));
}

}  // namespace nint
