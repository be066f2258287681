"""Integer-lattice cases for exact (bit-for-bit) checks of the CUDA kernels.  TEST INFRASTRUCTURE ONLY.

Inputs, weights and upstream gradients are small integers, and the recurrent state sits at points where every
activation and every activation derivative is a power of two (sigmoid(0) = 1/2, tanh(0) = 0, tanh(>= 24) = 1).  Then
every product of the gate convolution, its dgrad and its wgrad is a multiple of a known power-of-two grid, every
partial sum is exactly representable in fp32, and the correct result is unique whatever the accumulation order, the
split-K factor, the tile walk or the atomics.  The kernels must then equal the fp64 reference here with no tolerance:
a dropped, duplicated or misplaced term changes the result.

The one rounding the kernels do on the way is emulated: the gate gradients (dgates) are stored in the operand format
(bf16 round-to-nearest-even, tf32 round-to-nearest ties-away) before dgrad and wgrad read them.  In tf32 mode the
bias gradient also receives the rounding residuals (nint_api.cu resid_on: B*T*H*W <= 2^20), so it is the sum of the
unrounded dgates.

Three constructions (``case_a``, ``case_b``, ``case_c``):

* A -- the forward implicit GEMM alone (``Plan.debug_raw_gates``): dense small integers, the gate pre-activations
  equal an fp64 ``conv2d``.
* B -- one cell step forward and backward (``Plan.cell_forward`` / ``cell_backward``).  Channels interleave *live*
  (nonzero values, zero weight columns: the pre-activations stay exactly the bias) and *silent* (zero values, lattice
  weight columns: dgrad is nonzero).  Each hidden channel is in one of three modes that make different gate rows of
  dgates nonzero: 1) b_g = 0, c0 small -> f, g rows; 2) b_g = 40 (g = 1) -> i, f rows; 3) c0 = +-48 (tanh(c') = +-1),
  dh_out small -> o, f, g rows.  h' is exact only in mode 3 (``h_mask``).
* C -- whole ConvLSTM BPTT in the zero state: all biases 0 and layer 0's weights zero on the live x channels, so h
  and c are exactly 0 at every step and layer and pred equals the head bias.  The backward still runs every kernel:
  dgates are nonzero in the g rows, dh flows through time and down the layers, wgrad is nonzero in layer 0's live x
  columns and in every bias, and x.grad is nonzero on the silent channels.

``reference(case, dtype, order, defect)`` evaluates a case; ``headroom`` proves exactness (every sum of absolute
terms stays within 2^20 grid steps: 4 bits below fp32's 24 because tensor-core accumulation is not documented to be
IEEE-exact); ``coverage`` reports which tiles, taps, channel chunks, gate rows and images receive nonzero terms;
``DEFECTS`` are planted bugs applied to the reference to show that an exact comparison detects them.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F

TILE_W, TILE_H = 8, 16           # pixel tile of every conv kernel (nint_api.cu pick_tile): 8 wide, 16 high
CHUNK = 16                       # channel granularity checked: the tf32 K chunk (the bf16 one is 32 = two of these)
HEADROOM_BITS = 20
RESID_MAX_PIXEL_STEPS = 1 << 20  # nint_api.cu kResidMaxPixelSteps
DEFECTS = ("drop_ragged_tile", "drop_splitk_share", "shift_top_halo", "swap_gate_quarters", "drop_tf32_residual",
           "double_step")
SPLITK_SHARES = 4


# ------------------------------------------------------------------------------------------------ lattice values
class _Rng:
    def __init__(self, seed):
        self.g = torch.Generator().manual_seed(seed)

    def ints(self, shape, lo, hi, density=1.0, nonzero=False):
        """integers in [lo, hi] (fp64); with ``nonzero`` zero draws are pushed to +-1; ``density`` < 1 keeps that share"""
        v = torch.randint(lo, hi + 1, shape, generator=self.g).double()
        if nonzero:
            v = torch.where(v == 0, torch.where(torch.rand(shape, generator=self.g) < 0.5, -1.0, 1.0).double(), v)
        if density < 1:
            v = v * (torch.rand(shape, generator=self.g) < density).double()
        return v

    def signs(self, shape):
        return torch.where(torch.rand(shape, generator=self.g) < 0.5, -1.0, 1.0).double()


def live_channels(n: int) -> torch.Tensor:
    """live/silent pattern of one channel segment: even channels live, so every chunk of >= 2 channels has both"""
    return torch.arange(n) % 2 == 0


def _edge_pixels(H, W):
    """the four image corners, a pixel of the last (possibly ragged) tile row and one of the last tile column"""
    ty, tx = TILE_H * ((H - 1) // TILE_H), TILE_W * ((W - 1) // TILE_W)
    return [(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1), (ty + (H - 1 - ty) // 2, W // 2),
            (H // 2, tx + (W - 1 - tx) // 2)]


def case_a(B, C, hc, k, H, W, precision, seed=0):
    """forward implicit GEMM: dense x, h0 in [-2, 2] and weights in [-1, 1]"""
    r = _Rng(seed)
    return dict(kind="A", precision=precision, B=B, T=1, C=C, H=H, W=W, hidden=[hc], ks=[k],
                x=r.ints((B, 1, C, H, W), -2, 2), h0=r.ints((B, hc, H, W), -2, 2),
                w=r.ints((4 * hc, C + hc, k, k), -1, 1))


def case_b(B, C, hc, k, H, W, precision, seed=0, wdensity=0.25):
    """one cell step (T = 1, L = 1) with the three gate modes interleaved over the hidden channels; the upstream
    gradients thin out on large grids so that the bias gradient's sum stays within the exactness headroom"""
    r = _Rng(seed)
    dd = min(0.7, 2000.0 / (B * H * W))
    lx, lh = live_channels(C), live_channels(hc)
    x = r.ints((B, C, H, W), -2, 2, 0.6) * lx.view(1, C, 1, 1)
    h0 = r.ints((B, hc, H, W), -2, 2, 0.6) * lh.view(1, hc, 1, 1)
    w = r.ints((4 * hc, C + hc, k, k), -1, 1, wdensity)
    w[:, torch.cat([lx, lh])] = 0
    mode = torch.arange(hc) % 3 + 1
    bias = torch.zeros(4 * hc, dtype=torch.float64)
    bias[2 * hc:3 * hc][mode == 2] = 40.0
    m = lambda i: (mode == i).view(1, hc, 1, 1).double()
    c0 = r.ints((B, hc, H, W), -3, 3) * (m(1) + m(2)) + 48.0 * r.signs((B, hc, H, W)) * m(3)
    dc_out = r.ints((B, hc, H, W), -2, 2, dd)
    dh_out = r.ints((B, hc, H, W), -2, 2, dd) * m(3)
    for y, xx in _edge_pixels(H, W):   # every edge pixel carries an upstream gradient in every image
        dc_out[:, :, y, xx] = r.ints((B, hc), -2, 2, nonzero=True)
    return dict(kind="B", precision=precision, B=B, T=1, C=C, H=H, W=W, hidden=[hc], ks=[k],
                x=x.unsqueeze(1), w=w, bias=bias, h0=h0, c0=c0, dh_out=dh_out, dc_out=dc_out,
                h_mask=(mode == 3))


def case_c(B, T, C, H, W, hidden, ks, precision, seed=0, wdensity=0.06, ddensity=0.15, xdensity=0.5,
           return_sequence=False, wide_step=None, shared_frames=False):
    """whole-model BPTT in the zero state; upstream gradients: a sparse integer dpred (and dseq).  shared_frames:
    sample b is the window frames[b : b+T] of one record (``frames``, ``starts``), so consecutive samples share T-1
    frames, as the sliding windows of a frame bank do"""
    r = _Rng(seed)
    lx = live_channels(C)
    frames = starts = None
    if shared_frames:
        frames = r.ints((B + T - 1, C, H, W), -2, 2, xdensity) * lx.view(1, C, 1, 1)
        starts = torch.arange(B)
        x = torch.stack([frames[s:s + T] for s in starts.tolist()])
    else:
        x = r.ints((B, T, C, H, W), -2, 2, xdensity) * lx.view(1, 1, C, 1, 1)
    ws, cin = [], C
    for l, (hc, k) in enumerate(zip(hidden, ks)):
        w = r.ints((4 * hc, cin + hc, k, k), -1, 1, wdensity)
        if l == 0:
            w[:, :C][:, lx] = 0
        ws.append(w)
        cin = hc
    hw = r.ints((1, hidden[-1], 1, 1), -2, 2)
    hw.view(-1)[0] = 1.0
    hb = torch.tensor([0.75], dtype=torch.float64)
    dpred = r.ints((B, 1, H, W), -1, 1, ddensity)
    for y, xx in _edge_pixels(H, W):
        dpred[:, 0, y, xx] = r.ints((B,), -1, 1, nonzero=True)
    dseq = r.ints((B, T, H, W), -1, 1, ddensity / 2) if return_sequence else None
    if wide_step is not None:
        # one 12-bit head gradient: its dgates need rounding in both operand formats, and in tf32 the rounding residual
        # reaches the bias gradient.  Put early in the backward walk (late t) it would be carried down to the finest
        # grid of the later steps and cost the exactness headroom, so it sits at step 0 (dseq) or in a T = 1 case.
        assert wide_step == 0 and (return_sequence or T == 1)
        (dseq[:, 0] if return_sequence else dpred[:, 0])[0, H // 2, W // 2] = 2049.0
    return dict(kind="C", precision=precision, B=B, T=T, C=C, H=H, W=W, hidden=list(hidden), ks=list(ks), x=x,
                ws=ws, bs=[torch.zeros(4 * hc, dtype=torch.float64) for hc in hidden], hw=hw, hb=hb, dpred=dpred,
                dseq=dseq, return_sequence=return_sequence, wide=wide_step is not None, frames=frames, starts=starts)


def resid_on(case) -> bool:
    """tf32 training plans add the dgates rounding residuals to the bias gradient (nint_api.cu resid_on, 148 SMs)"""
    return case["precision"] == "tf32" and case["B"] * case["T"] * case["H"] * case["W"] <= RESID_MAX_PIXEL_STEPS


# ------------------------------------------------------------------------------------------------ arithmetic helpers
def round_tf32(t: torch.Tensor) -> torch.Tensor:
    """cvt.rna.tf32.f32 on fp32: round to nearest, ties away from zero, on the 13 dropped mantissa bits"""
    bits = t.contiguous().view(torch.int32)
    return ((bits + 0x1000) & ~0x1FFF).view(torch.float32)


def to_operand(t: torch.Tensor, precision: str) -> torch.Tensor:
    """the kernels' rounding of fp32 dgates into the MMA operand format, evaluated at t's dtype"""
    f = t.float()
    if t.dtype == torch.float64 and not torch.equal(f.double(), t):
        raise ArithmeticError("a dgate is not an fp32 value: the case is not exact")
    r = f.to(torch.bfloat16).float() if precision == "bf16" else round_tf32(f)
    return r.to(t.dtype)


def grid(t: torch.Tensor) -> float:
    """the coarsest power of two that divides every element of t (inf for an all-zero tensor)"""
    a = t[t != 0].abs().double()
    if a.numel() == 0:
        return math.inf
    m, e = torch.frexp(a)
    mi = (m * 2.0 ** 53).long()
    tz = torch.log2((mi & -mi).double()).round().long()
    return 2.0 ** float((e.long() - 53 + tz).min())


def _conv(inp, w, pad, defect=None):
    """conv2d with zero padding, skipping channels that are zero in the input or in the weights (exact: they add 0)"""
    keep = (inp != 0).flatten(2).any(2).any(0) & (w != 0).flatten(2).any(2).any(0)
    if not bool(keep.any()):
        return inp.new_zeros(inp.shape[0], w.shape[0], *inp.shape[2:])
    out = F.conv2d(inp[:, keep], w[:, keep], padding=pad)
    if defect == "shift_top_halo":      # the first tile row reads its window one row too low
        out[:, :, :TILE_H] = F.conv2d(F.pad(inp[:, keep], (0, 0, 1, 0))[:, :, :-1], w[:, keep], padding=pad)[:, :, :TILE_H]
    return out


def _dgrad(dg, w, pad, defect=None):
    """dcomb = dg (*) flip(W): the transposed gate convolution, skipping all-zero dgate rows"""
    rows = (dg != 0).flatten(2).any(2).any(0)
    if not bool(rows.any()):
        return dg.new_zeros(dg.shape[0], w.shape[1], *dg.shape[2:])
    out = F.conv_transpose2d(dg[:, rows], w[rows], padding=pad)
    if defect == "shift_top_halo":
        sh = F.pad(dg[:, rows], (0, 0, 1, 0))[:, :, :-1]
        out[:, :, :TILE_H] = F.conv_transpose2d(sh, w[rows], padding=pad)[:, :, :TILE_H]
    return out


def _wgrad(dg, comb, k, perm=None):
    """dW[n, c, dy, dx] = sum_{b,y,x} dg[b,n,y,x] comb[b,c,y+dy-p,x+dx-p], as one pixel-major GEMM per tap;
    ``perm`` reorders the pixels (the K dimension) of every GEMM"""
    B, N, H, W = dg.shape
    gw = dg.new_zeros(N, comb.shape[1], k, k)
    rows = (dg != 0).flatten(2).any(2).any(0)
    cols = (comb != 0).flatten(2).any(2).any(0)
    if not bool(rows.any()) or not bool(cols.any()):
        return gw
    p = k // 2
    a = dg[:, rows].permute(0, 2, 3, 1).reshape(-1, int(rows.sum()))
    cp = F.pad(comb[:, cols], (p, p, p, p))
    if perm is not None:
        a = a[perm]
    sub = dg.new_zeros(int(rows.sum()), int(cols.sum()), k, k)
    for dy in range(k):
        for dx in range(k):
            win = cp[:, :, dy:dy + H, dx:dx + W].permute(0, 2, 3, 1).reshape(-1, sub.shape[1])
            if perm is not None:
                win = win[perm]
            sub[:, :, dy, dx] = a.t() @ win
    gw[rows.nonzero()[:, 0].unsqueeze(1), cols.nonzero()[:, 0].unsqueeze(0)] = sub
    return gw


def _pixsum(t, perm=None):
    """sum over (b, y, x) per channel, pixels optionally reordered"""
    a = t.permute(0, 2, 3, 1).reshape(-1, t.shape[1])
    return (a[perm] if perm is not None else a).sum(0)


def _tile_mask(B, H, W, defect):
    """1 on the pixels a wgrad defect keeps, 0 on those it drops (None: keeps all)"""
    if defect == "drop_ragged_tile":      # the bottom-right tile of the last image
        m = torch.ones(B, 1, H, W, dtype=torch.float64)
        m[-1, :, TILE_H * ((H - 1) // TILE_H):, TILE_W * ((W - 1) // TILE_W):] = 0
        return m
    if defect == "drop_splitk_share":     # one of SPLITK_SHARES contiguous shares of the (image, tile) walk
        ty, tx = (H + TILE_H - 1) // TILE_H, (W + TILE_W - 1) // TILE_W
        n = B * ty * tx
        lo, hi = n * 1 // SPLITK_SHARES, n * 2 // SPLITK_SHARES
        if hi == lo:
            hi = lo + 1
        m = torch.ones(B, 1, H, W, dtype=torch.float64)
        for i in range(lo, hi):
            b, rest = divmod(i, ty * tx)
            y, xx = divmod(rest, tx)
            m[b, :, y * TILE_H:(y + 1) * TILE_H, xx * TILE_W:(xx + 1) * TILE_W] = 0
        return m
    return None


def _swap_go(t, hc):
    """planted q-order bug: the g and o quarters of a gate tensor trade places"""
    return torch.cat([t[:, :2 * hc], t[:, 3 * hc:], t[:, 2 * hc:3 * hc]], 1)


# ------------------------------------------------------------------------------------------------ reference
def reference(case, dtype=torch.float64, order: Optional[int] = None, defect: Optional[str] = None,
              stats: Optional[dict] = None) -> Dict[str, torch.Tensor]:
    """The case evaluated at ``dtype``.  ``order``: a seed that permutes the pixel order of every wgrad / bias sum and
    the time order in which the per-step gradient contributions are added.  ``defect``: one of DEFECTS, planted.
    ``stats``: filled with per-sum headroom (``stats['headroom']``) and coverage maps."""
    if case["kind"] == "A":
        return _reference_a(case, dtype, defect, stats)
    return _reference_bptt(case, dtype, order, defect, stats)


def _note(stats, name, abs_sum, gamma):
    if stats is None or not math.isfinite(gamma):
        return
    v = float(abs_sum.max()) / gamma
    hr = stats.setdefault("headroom", {})
    hr[name] = max(hr.get(name, 0.0), v)


def _reference_a(case, dtype, defect, stats):
    x, h0, w = case["x"][:, 0].to(dtype), case["h0"].to(dtype), case["w"].to(dtype)
    hc, k = case["hidden"][0], case["ks"][0]
    inp = torch.cat([x, h0], 1)
    if defect == "drop_splitk_share":        # one K chunk of the h segment never reaches the accumulator
        inp = inp.clone()
        inp[:, case["C"]:case["C"] + CHUNK] = 0
    out = _conv(inp, w, k // 2, defect)
    if defect == "swap_gate_quarters":
        out = _swap_go(out, hc)
    if defect == "drop_ragged_tile":
        out = out * _tile_mask(case["B"], case["H"], case["W"], defect).to(dtype)
    if stats is not None:
        m = F.conv2d(inp.abs().double(), w.abs().double(), padding=k // 2)
        _note(stats, "gates", m, grid(inp) * grid(w))
        cov = _new_cov(stats, case)
        cov["pix"] |= (m != 0).any(1)
        cov["quarters"] |= torch.stack([(m[:, q * hc:(q + 1) * hc] != 0).any() for q in range(4)])
        cov["qchunks"][0] |= _qchunks(m.ne(0).any(3).any(2).any(0), hc)
        cov["cin"][0] |= ((inp != 0).flatten(2).any(2).any(0) & (w != 0).flatten(2).any(2).any(0))
        cov["taps"][0] |= _tap_hits(inp, w, k, forward=True)
    return {"gates": out}


def _reference_bptt(case, dtype, order, defect, stats):
    kind, prec = case["kind"], case["precision"]
    B, T, C, H, W = case["B"], case["T"], case["C"], case["H"], case["W"]
    hidden, ks = case["hidden"], case["ks"]
    L = len(hidden)
    x = case["x"].to(dtype)
    if kind == "B":
        Ws, bs = [case["w"].to(dtype)], [case["bias"].to(dtype)]
        h_init, c_init = [case["h0"].to(dtype)], [case["c0"].to(dtype)]
    else:
        Ws, bs = [w.to(dtype) for w in case["ws"]], [b.to(dtype) for b in case["bs"]]
        h_init = [torch.zeros(B, hc, H, W, dtype=dtype) for hc in hidden]
        c_init = [torch.zeros(B, hc, H, W, dtype=dtype) for hc in hidden]
    resid = resid_on(case)
    perm = tperm = None
    if order is not None:
        g = torch.Generator().manual_seed(order)
        perm = torch.randperm(B * H * W, generator=g)
        tperm = torch.randperm(T, generator=g).tolist()
    cov = _new_cov(stats, case) if stats is not None else None

    # ---- forward, saving what backward needs
    hs = [[h_init[l]] for l in range(L)]
    cs = [[c_init[l]] for l in range(L)]
    gates = [[None] * T for _ in range(L)]
    for t in range(T):
        inp = x[:, t]
        for l in range(L):
            k, hc = ks[l], hidden[l]
            comb = torch.cat([inp, hs[l][t]], 1)
            pre = _conv(comb, Ws[l], k // 2) + bs[l].view(1, -1, 1, 1)
            if stats is not None:
                _note(stats, f"gates{l}", F.conv2d(comb.abs().double(), Ws[l].abs().double(), padding=k // 2),
                      grid(comb) * grid(Ws[l]))
            i, f, gg, o = torch.split(pre, hc, 1)
            i, f, gg, o = torch.sigmoid(i), torch.sigmoid(f), torch.tanh(gg), torch.sigmoid(o)
            c = cs[l][t] * f + i * gg
            h = o * torch.tanh(c)
            gates[l][t] = (i, f, gg, o)
            hs[l].append(h)
            cs[l].append(c)
            inp = h
    out: Dict[str, torch.Tensor] = {}
    if kind == "B":
        out["c"], out["h"] = cs[0][1], hs[0][1]
    else:
        hw, hb = case["hw"].to(dtype), case["hb"].to(dtype)
        out["pred"] = F.conv2d(hs[L - 1][T], hw, hb)
        if case["return_sequence"]:
            out["seq"] = torch.cat([F.conv2d(hs[L - 1][t + 1], hw, hb) for t in range(T)], 1)

    # ---- backward
    dtop = torch.zeros(B, T, H, W, dtype=dtype)      # head gradient per step (the kernels' dpred operand)
    if kind == "C":
        if case["dseq"] is not None:
            dtop += case["dseq"].to(dtype)
        dtop[:, T - 1] += case["dpred"][:, 0].to(dtype)
    gw = [torch.zeros_like(w) for w in Ws]
    gb = [torch.zeros_like(b) for b in bs]
    contrib = [[None] * T for _ in range(L)]     # (wgrad, bias) of every (layer, step), summed at the end
    dh_next = [torch.zeros(B, hc, H, W, dtype=dtype) for hc in hidden]
    dc_next = [torch.zeros(B, hc, H, W, dtype=dtype) for hc in hidden]
    habs = [None] * L                            # |terms| of dh_next (headroom of the dgrad accumulator)
    hgam = [math.inf] * L
    if kind == "B":
        dh_next[0] = case["dh_out"].to(dtype)
        dc_next[0] = case["dc_out"].to(dtype)
    dx = torch.zeros(B, T, C, H, W, dtype=dtype)
    # |terms| and grid of each wgrad GEMM, accumulated over all steps: the kernels reduce the T*B*tiles pixels of a
    # layer in one tensor-core accumulation, and the bias gradient is a column of it (the ones lane / ones panel)
    wabs = [torch.zeros(w.shape, dtype=torch.float64) for w in Ws] if stats is not None else None
    babs = [torch.zeros(b.shape, dtype=torch.float64) for b in bs] if stats is not None else None
    rabs = [torch.zeros(b.shape, dtype=torch.float64) for b in bs] if stats is not None else None
    wgam, bgam, rgam = [math.inf] * L, [math.inf] * L, [math.inf] * L
    mask = _tile_mask(B, H, W, defect)
    for t in reversed(range(T)):
        dx_from_above = None
        above_abs, above_gam = None, math.inf
        for l in reversed(range(L)):
            hc, k = hidden[l], ks[l]
            p = k // 2
            dh = dh_next[l]
            if dx_from_above is not None:
                dh = dh + dx_from_above
            i, f, gg, o = gates[l][t]
            head = None
            if kind == "C" and l == L - 1:
                head = dtop[:, t:t + 1] * hw.view(1, -1, 1, 1)
                dh = dh + head
            if stats is not None:
                terms = [a for a in (habs[l], above_abs) if a is not None]
                gam = min(hgam[l], above_gam)
                if head is not None:
                    terms.append(head.abs().double())
                    gam = min(gam, grid(head))
                if terms:
                    _note(stats, f"dh{l}", sum(terms), gam)
            tc = torch.tanh(cs[l][t + 1])
            do = dh * tc
            dcv = dc_next[l] + dh * o * (1 - tc * tc)
            if stats is not None:
                a1, a2 = (dh * o * (1 - tc * tc)), dc_next[l]
                _note(stats, f"dc{l}", a1.abs().double() + a2.abs().double(), min(grid(a1), grid(a2)))
            di, dgv, df = dcv * gg, dcv * i, dcv * cs[l][t]
            dc_next[l] = dcv * f
            dpre = torch.cat([di * i * (1 - i), df * f * (1 - f), dgv * (1 - gg * gg), do * o * (1 - o)], 1)
            dg = to_operand(dpre, prec)
            if defect == "swap_gate_quarters":
                dg = _swap_go(dg, hc)
            inp = x[:, t] if l == 0 else hs[l - 1][t + 1]
            comb = torch.cat([inp, hs[l][t]], 1)
            wdg = dg if mask is None else dg * mask.to(dtype)
            bsrc = dpre if (resid and defect != "drop_tf32_residual") else dg
            if mask is not None:
                bsrc = bsrc * mask.to(dtype)
            contrib[l][t] = (_wgrad(wdg, comb, k, perm), _pixsum(bsrc, perm))
            dcomb = _dgrad(dg, Ws[l], p, defect)
            cin = inp.shape[1]
            if stats is not None:
                adg = dg.abs().double()
                ad = _dgrad(adg, Ws[l].abs().double(), p)
                gd = grid(dg) * grid(Ws[l])
                habs[l], hgam[l] = ad[:, cin:], gd
                above_abs, above_gam = ad[:, :cin], gd
                if l == 0:
                    _note(stats, "dx", ad[:, :cin], gd)
                wabs[l] += _wgrad(adg, comb.abs().double(), k)
                wgam[l] = min(wgam[l], grid(dg) * grid(comb))
                babs[l] += adg.sum((0, 2, 3))
                bgam[l] = min(bgam[l], grid(dg))
                if resid:                  # the rounding residuals the tf32 epilogue adds to the same bias element
                    rabs[l] += (dpre - dg).abs().double().sum((0, 2, 3))
                    rgam[l] = min(rgam[l], grid(dpre))
                _cover(cov, l, dg, comb, Ws[l], k, hc, cin)
            dx_from_above = dcomb[:, :cin] if l > 0 else None
            if l == 0:
                dx[:, t] = dcomb[:, :cin]
            dh_next[l] = dcomb[:, cin:]
    steps = tperm if tperm is not None else list(reversed(range(T)))
    for l in range(L):
        for t in steps:
            gw[l] += contrib[l][t][0]
            gb[l] += contrib[l][t][1]
        if defect == "double_step":
            gw[l] += contrib[l][0][0]
            gb[l] += contrib[l][0][1]
        if stats is not None:
            _note(stats, f"dw{l}", wabs[l], wgam[l])
            _note(stats, f"db{l}", babs[l], bgam[l])
            if resid:
                _note(stats, f"db{l}+resid", babs[l] + rabs[l], min(bgam[l], rgam[l]))
    if stats is not None and kind == "B":      # dh of the cell: the h columns of the last dgrad (asserted output)
        _note(stats, "dh_in", habs[0], hgam[0])
    if kind == "B":
        out.update(dx=dx[:, 0], dh=dh_next[0], dc=dc_next[0], gw=gw[0], gb=gb[0])
    else:
        for l in range(L):
            out[f"gw{l}"], out[f"gb{l}"] = gw[l], gb[l]
        out["ghw"] = sum((dtop[:, t:t + 1] * hs[L - 1][t + 1]).sum((0, 2, 3)) for t in range(T)).view(1, -1, 1, 1)
        out["ghb"] = dtop.sum().view(1)
        out["dx"] = dx
    return out


# ------------------------------------------------------------------------------------------------ coverage
def _new_cov(stats, case):
    if "cov" not in stats:
        B, H, W = case["B"], case["H"], case["W"]
        cins = [case["C"]] + case["hidden"][:-1]
        stats["cov"] = dict(
            pix=torch.zeros(B, H, W, dtype=torch.bool),
            quarters=torch.zeros(4, dtype=torch.bool),
            qchunks=[torch.zeros(4, (hc + CHUNK - 1) // CHUNK, dtype=torch.bool) for hc in case["hidden"]],
            cin=[torch.zeros(ci + hc, dtype=torch.bool) for ci, hc in zip(cins, case["hidden"])],
            cins=cins,
            taps=[torch.zeros(k, k, dtype=torch.bool) for k in case["ks"]])
    return stats["cov"]


def _qchunks(rows_nz, hc):
    """[4hc] nonzero flags -> [4, chunks]: which 16-channel chunk of which gate quarter is nonzero"""
    n = (hc + CHUNK - 1) // CHUNK
    r = F.pad(rows_nz.view(4, hc).float(), (0, n * CHUNK - hc))
    return r.view(4, n, CHUNK).any(2)


def _tap_hits(act, w, k, forward):
    """[k, k]: does tap (dy, dx) multiply a nonzero weight with a nonzero value that lies inside the image?
    forward: act = conv input [B, Cin, H, W]; otherwise act = dgates [B, N, H, W] (dgrad)"""
    p = k // 2
    H, W = act.shape[2:]
    hit = torch.zeros(k, k, dtype=torch.bool)
    for dy in range(k):
        for dx in range(k):
            wt = w[:, :, dy, dx] != 0
            sel = wt.any(0) if forward else wt.any(1)     # channels (forward) / dgate rows (dgrad) the tap reads
            if not bool(sel.any()):
                continue
            a = (act[:, sel] != 0).any(1)
            # forward: out[y] reads act[y + dy - p]; dgrad: dcomb[y] reads dg[y + p - dy]
            sy, sx = (dy - p, dx - p) if forward else (p - dy, p - dx)
            ys = slice(max(0, sy), min(H, H + sy))
            xs = slice(max(0, sx), min(W, W + sx))
            hit[dy, dx] = bool(a[:, ys, xs].any())
    return hit


def _cover(cov, l, dg, comb, w, k, hc, cin):
    nz = dg != 0
    cov["pix"] |= nz.any(1)
    rows = nz.flatten(2).any(2).any(0)
    cov["quarters"] |= rows.view(4, hc).any(1)
    cov["qchunks"][l] |= _qchunks(rows, hc)
    # a channel of the conv input is covered when a nonzero term reaches its wgrad column or its dgrad output
    wg_cols = (comb != 0).flatten(2).any(2).any(0) & bool(rows.any())
    dg_cols = (w[rows] != 0).flatten(2).any(2).any(0) if bool(rows.any()) else torch.zeros(w.shape[1], dtype=torch.bool)
    cov["cin"][l] |= wg_cols | dg_cols
    cov["taps"][l] |= _tap_hits(dg, w, k, forward=False)


def headroom(case) -> float:
    """worst sum of |terms| over an output's grid step, over every sum the kernels accumulate in fp32"""
    stats: dict = {}
    reference(case, stats=stats)
    return max(stats["headroom"].values())


def coverage(case) -> Dict[str, bool]:
    """which places receive nonzero terms of the sums the kernels accumulate (dgates for the backward cases)"""
    stats: dict = {}
    reference(case, stats=stats)
    return summarize_coverage(case, stats["cov"])


def summarize_coverage(case, cov) -> Dict[str, bool]:
    B, H, W = case["B"], case["H"], case["W"]
    pix = cov["pix"]
    ty, tx = TILE_H * ((H - 1) // TILE_H), TILE_W * ((W - 1) // TILE_W)
    res = {
        "corners": all(bool(pix[:, y, xx].any()) for y, xx in ((0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1))),
        "last_tile_row": bool(pix[:, ty:].any()),
        "last_tile_col": bool(pix[:, :, tx:].any()),
        "every_image": bool(pix.flatten(1).any(1).all()),
        "every_tap": all(bool(t.all()) for t in cov["taps"]),
    }
    ok = True
    for ci, c in zip(cov["cins"], cov["cin"]):   # x segment and h segment are chunked separately
        for lo, hi in ((0, ci), (ci, c.numel())):
            for s in range(lo, hi, CHUNK):
                ok &= bool(c[s:min(s + CHUNK, hi)].any())
    res["every_channel_chunk"] = ok
    q = cov["quarters"]
    if case["kind"] == "C":
        # zero state: only the g rows of dgates are nonzero (di = dc*g = 0, df = dc*c_prev = 0, do = dh*tanh(c) = 0)
        res["g_rows"] = bool(q[2])
        res["every_gate_chunk"] = all(bool(qc[2].all()) for qc in cov["qchunks"])
    else:
        res["every_gate_row"] = bool(q.all())
        res["every_gate_chunk"] = all(bool(qc.all()) for qc in cov["qchunks"])
    return res


def defects_for(case) -> List[str]:
    """the planted defects that apply to a case's construction"""
    if case["kind"] == "A":
        return ["drop_ragged_tile", "drop_splitk_share", "shift_top_halo", "swap_gate_quarters"]
    d = ["drop_ragged_tile", "drop_splitk_share", "shift_top_halo", "swap_gate_quarters"]
    if case["kind"] == "C":
        d.append("double_step")
        if resid_on(case) and case["wide"]:
            d.append("drop_tf32_residual")
    return d


# ------------------------------------------------------------------------------------------------ the suite's cases
# (B, C, hidden, k, H, W): one exact tile; ragged in x and y with cin = 33; 5x5 taps; two n-blocks; the widest hidden
# size; 7x7 taps on a grid barely larger than the kernel; 1x1 (no halo); BASELINE cfg 2's grid
A_SHAPES = [(1, 32, 64, 3, 8, 16), (2, 33, 64, 3, 9, 17), (3, 8, 16, 5, 11, 13), (2, 21, 128, 3, 20, 24),
            (1, 3, 256, 3, 12, 20), (2, 16, 16, 7, 10, 12), (5, 21, 64, 1, 8, 16), (2, 21, 64, 3, 90, 144)]
# input channel counts around the K chunk of each operand format (16 tf32 / 32 bf16 channels = 64 bytes)
CHUNK_EDGES = {"tf32": (15, 16, 17), "bf16": (31, 32, 33)}
# hidden sizes that run padded to the kernels' granularity
B_PADDED = [(2, 21, 10, 3, 9, 17), (1, 21, 70, 3, 12, 20), (1, 3, 192, 3, 12, 20)]
_SPARSE = dict(xdensity=0.04, ddensity=0.008, wdensity=0.03)
C_CASES = {
    "h32_h16_k3_k5_17x13": dict(B=2, T=3, C=9, H=17, W=13, hidden=[32, 16], ks=[3, 5]),
    "h64_k3_33x9_T4": dict(B=2, T=4, C=21, H=33, W=9, hidden=[64], ks=[3], shared_frames=True),
    "h64_k5_16x40": dict(B=2, T=3, C=21, H=16, W=40, hidden=[64], ks=[5]),
    "h128_h64_k3_12x20": dict(B=2, T=3, C=9, H=12, W=20, hidden=[128, 64], ks=[3, 3]),
    "h256_k3_T1_wide": dict(B=1, T=1, C=3, H=12, W=20, hidden=[256], ks=[3], wide_step=0),
    # 40 images of 5 x 3 tiles: several tile groups per cluster and step in the time-fused launch
    "b40_40x36_T4": dict(B=40, T=4, C=21, H=40, W=36, hidden=[64], ks=[3], **_SPARSE),
    "seq_h32_h16_wide": dict(B=2, T=3, C=9, H=17, W=13, hidden=[32, 16], ks=[3, 5], return_sequence=True, wide_step=0),
    # BASELINE cfg 2 at its batch size (bf16 only: the configuration the benchmark trains)
    "cfg2_b32": dict(B=32, T=3, C=21, H=90, W=144, hidden=[64], ks=[3], xdensity=0.03, ddensity=0.01, wdensity=0.04),
}
C_BF16_ONLY = ("cfg2_b32",)


def suite_cases():
    """(id, case) of every lattice case the GPU tests run"""
    out = []
    for prec in ("tf32", "bf16"):
        shapes = A_SHAPES + [s for s in ((2, c, 64, 3, 9, 17) for c in CHUNK_EDGES[prec]) if s not in A_SHAPES]
        out += [(f"A-{prec}-" + "_".join(map(str, s)), case_a(*s, prec)) for s in shapes]
        out += [(f"B-{prec}-" + "_".join(map(str, s)), case_b(*s, prec)) for s in A_SHAPES + B_PADDED]
        out += [(f"C-{prec}-{n}", c_case(n, prec)) for n in C_CASES if prec == "bf16" or n not in C_BF16_ONLY]
    return out


def c_case(name, precision):
    kw = dict(C_CASES[name])
    return case_c(kw.pop("B"), kw.pop("T"), kw.pop("C"), kw.pop("H"), kw.pop("W"), kw.pop("hidden"), kw.pop("ks"),
                  precision, **kw)
