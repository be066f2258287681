"""CPU reference for input gradients through the frame bank and the preprocessing.  TEST INFRASTRUCTURE ONLY.

``fuse_inputs_torch`` restates ``convlstm_oracle.fuse_inputs`` (stack, z-score, static attributes, geophysical halo) in
differentiable torch, equal to the numpy oracle bit for bit, so autograd gives the reference gradient w.r.t. the raw
fields.  ``fuse_adjoint_reference`` is the adjoint in the order ``nint_fuse_inputs_adjoint`` promises: every source
element sums its halo preimages in fp32 in increasing padded row, then padded column (statics: frames first), and the
z-scored channels then divide by std.  ``scatter_windows`` adds per-window input gradients into the frames they were
cut from, in (t, b) order, as ``nint_backward_input_bank`` does.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

import torch

Tensor = torch.Tensor


def _halo_rows(H: int, Hp: int):
    top = (Hp - H) // 2
    return top, Hp - H - top


def fuse_inputs_torch(levels3d: Tensor, emis2d: Tensor, mean: Tensor, std: Tensor,
                      target_hw: Optional[Tuple[int, int]] = None, mode: str = "reflect",
                      statics: Optional[Tensor] = None) -> Tensor:
    """``convlstm_oracle.fuse_inputs`` in torch: levels3d [N,L,H,W], emis2d [N,H,W] fp32 -> [N,L+1+S,Hp,Wp]"""
    X = torch.cat([levels3d, emis2d[:, None]], dim=1)
    X = (X - mean.reshape(1, -1, 1, 1)) / std.reshape(1, -1, 1, 1)
    if statics is not None:
        X = torch.cat([X, statics[None].expand(X.shape[0], -1, -1, -1)], dim=1)
    if target_hw is None:
        return X
    H, W = X.shape[-2:]
    left = (target_hw[1] - W) // 2
    right = target_hw[1] - W - left
    if left > W or right > W:
        raise AttributeError("The requested padding size is larger than width size of the input image.")
    X = torch.cat([X[..., W - left:], X, X[..., :right]], dim=-1)
    top, bot = _halo_rows(H, target_hw[0])
    if top + 1 > H or bot + 1 > H:
        raise AttributeError("The requested padding size is larger than height size of the input image.")
    upper, lower = X[..., 1:top + 1, :], X[..., H - bot - 1:H - 1, :]
    if mode == "reflect":
        upper, lower = upper.flip(-2), lower.flip(-2)
    elif mode == "reference_rnn":      # np.fliplr on a (T, C, rows, W) slab reverses the channels
        upper, lower = upper.flip(1), lower.flip(1)
    else:
        raise ValueError(mode)
    return torch.cat([upper, X, lower], dim=-2)


def _preimages(H: int, W: int, Hp: int, Wp: int, mode: str):
    """per source pixel, the three row slots (upper halo, interior, lower halo) and three column slots (left copy,
    interior, right copy) in increasing padded order: (valid mask [H,W], padded row, padded col, channel-flipped)"""
    top, bot = _halo_rows(H, Hp)
    left = (Wp - W) // 2
    ys = torch.arange(H).view(H, 1).expand(H, W)
    xs = torch.arange(W).view(1, W).expand(H, W)
    flip = mode == "reference_rnn"
    j = (H - 2 - ys) if mode == "reflect" else ys - (H - bot - 1)
    rows = [((ys >= 1) & (ys <= top), (top - ys) if mode == "reflect" else ys - 1, flip),
            (torch.ones_like(ys, dtype=torch.bool), top + ys, False),
            ((j >= 0) & (j < bot), top + H + j, flip)]
    cols = [(xs + left - W >= 0, xs + left - W), (torch.ones_like(xs, dtype=torch.bool), xs + left),
            (xs + left + W < Wp, xs + left + W)]
    out = []
    for rok, yp, fl in rows:
        for cok, xp in cols:
            ok = rok & cok
            out.append((ok, yp.clamp(0, Hp - 1), xp.clamp(0, Wp - 1), fl))
    return out


def fuse_adjoint_reference(dframes: Tensor, std: Tensor, levels: int, n_static: int, height: int, width: int,
                           mode: str = "reflect") -> Dict[str, Optional[Tensor]]:
    """dframes [N,C,Hp,Wp] fp32 -> {"levels3d" [N,L,H,W], "emis2d" [N,H,W], "statics" [S,H,W] or None}, summed in
    the kernel's order (fp32, padded row then column; statics: frame, row, column) and divided by std (IEEE)"""
    N, C, Hp, Wp = dframes.shape
    assert C == levels + 1 + n_static and dframes.dtype == torch.float32
    taps = _preimages(height, width, Hp, Wp, mode)
    rev = dframes.flip(1)                      # channel C-1-c of the halo rows in mode reference_rnn
    gathered = [torch.where(ok, (rev if fl else dframes)[:, :, yp, xp], torch.zeros(())) for ok, yp, xp, fl in taps]
    acc = torch.zeros(N, levels + 1, height, width)
    for g in gathered:
        acc = acc + g[:, :levels + 1]
    z = acc / std.reshape(1, -1, 1, 1).float()
    stat = None
    if n_static:
        stat = torch.zeros(n_static, height, width)
        for n in range(N):
            for g in gathered:
                stat = stat + g[n, levels + 1:]
    return {"levels3d": z[:, :levels], "emis2d": z[:, levels], "statics": stat}


def scatter_windows(dx: Tensor, starts: Sequence[int], n_frames: int) -> Tensor:
    """dx [B,T,C,H,W] of windows cut from frames starts[b] .. starts[b]+T-1 -> [n_frames,C,H,W], frame f summing its
    terms in (t, b) order; frames outside [0, n_frames) are dropped"""
    B, T = dx.shape[:2]
    out = torch.zeros((n_frames,) + tuple(dx.shape[2:]), dtype=dx.dtype)
    for t in range(T):
        for b in range(B):
            f = int(starts[b]) + t
            if 0 <= f < n_frames:
                out[f] += dx[b, t]
    return out
