"""Preprocessing fusion on the GPU (north-star item 4): what the reference's RNN dataset does on the host per
sample (dataset.py:520-537 stack + z-score, dataset.py:67-98 cyclic-longitude / reflect-latitude halo), as one
memory-bound kernel (`nint_fuse_inputs`).  The README's 20-level module has no shipped code: for more than one
level this follows the single-level code path and its parity is unpinned upstream (SURVEY.md section 0)."""
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from . import _lib

MODES = {"reflect": 0, "reference_rnn": 1}
_DTYPES = {"bf16": (_lib.DTYPE_BF16, torch.bfloat16), "tf32": (_lib.DTYPE_TF32, torch.float32),
           "fp32": (_lib.DTYPE_TF32, torch.float32)}


def input_layout(channels: int) -> Tuple[int, int]:
    """(c_pad, ones_lane) of the model's channels-last input layout for `channels` input channels: channels padded to
    a multiple of 32 with zero lanes, the first padding lane holding 1.0 (the bias gradient rides on it; -1 when the
    channel count is already a multiple of 32).  Same rule as nint_plan_input_layout."""
    c_pad = (channels + 31) // 32 * 32
    return c_pad, (channels if c_pad > channels else -1)


class FrameBank:
    """The record resident in HBM in the model's own operand layout (the B200 form of dataset.py:551-637, where
    E33OMA90D_CRNN keeps the whole file in RAM and cuts windows with sliding_window_view): `frames` [N, Hp, Wp, c_pad]
    of bf16 (bf16 models) or tf32-rounded fp32, and optionally `targets` [N, Hy, Wy] fp32.  A training batch is then B
    window-start indices: sample b = frames[i_b : i_b + T], target = targets[i_b + T - 1] (dataset.py:600-601); the
    kernels read both through those indices, so a step uploads 4 B bytes instead of B windows.

    Input gradients: after `requires_grad_()`, every `ConvLSTM.forward_windows` over the bank under grad mode adds, on
    backward, dL/dx of its windows into `grad` [N, C, Hp, Wp] fp32 (frame win_start[b] + t gets sample b's step t), like
    `.grad` of a leaf.  `field_grads()` takes that back through the preprocessing of `from_fields` to the raw fields.

    Tangents (forward mode): `tangent(dframes)` and `tangent_from_fields(...)` give a perturbation direction of every
    frame in the bank's layout, which `ConvLSTM.jvp_windows` reads through the same window starts."""

    def __init__(self, frames: torch.Tensor, channels: int, precision: str = "bf16", targets: Optional[torch.Tensor] = None):
        if precision not in _DTYPES:
            raise ValueError(f"precision must be one of {sorted(_DTYPES)}")
        c_pad, ones = input_layout(channels)
        if frames.dim() != 4 or frames.shape[-1] != c_pad or frames.dtype != _DTYPES[precision][1] or not frames.is_cuda:
            raise ValueError(f"frames must be a CUDA tensor [N, H, W, {c_pad}] of {_DTYPES[precision][1]}")
        self.frames, self.channels, self.c_pad, self.ones_lane, self.precision = frames.contiguous(), channels, c_pad, ones, precision
        if targets is not None:
            if targets.dim() != 3 or targets.shape[0] != frames.shape[0] or targets.dtype != torch.float32 or \
                    targets.device != frames.device:
                raise ValueError("targets must be [N, Hy, Wy] fp32 on the frames' device")
            targets = targets.contiguous()
        self.targets = targets
        self.grad: Optional[Tensor] = None
        self._anchor: Optional[Tensor] = None   # zero-size leaf that requires grad: it puts the forward into the graph
        self._fields: Optional[dict] = None      # from_fields: what the preprocessing adjoint needs (field_grads)

    def requires_grad_(self, flag: bool = True) -> "FrameBank":
        """Collect dL/d(frames) in `grad`, fp32 [N, C, Hp, Wp] zeros (flag=False drops it).  That is 4*C*Hp*Wp bytes per
        frame: 497 MB for 384 frames of 21 x 100 x 154, 22.7 GB for a year of half-hourly frames.  The bank's own
        rounding to bf16 / tf32 counts as identity (straight through), as it does for x.grad of explicit windows."""
        if flag and self.grad is None:
            N, Hp, Wp, _ = self.frames.shape
            self.grad = torch.zeros((N, self.channels, Hp, Wp), dtype=torch.float32, device=self.frames.device)
            self._anchor = torch.zeros(0, dtype=torch.float32, device=self.frames.device, requires_grad=True)
        elif not flag:
            self.grad = self._anchor = None
        return self

    @property
    def requires_grad(self) -> bool:
        return self.grad is not None

    def zero_grad(self):
        if self.grad is not None:
            self.grad.zero_()

    def field_grads(self) -> Dict[str, Optional[Tensor]]:
        """`grad` taken back through the preprocessing of `from_fields` (nint_fuse_inputs_adjoint): {"levels3d"
        [N, L, H, W], "emis2d" [N, H, W], "statics" [S, H, W] summed over the frames, or None without statics}."""
        if self._fields is None:
            raise RuntimeError("field_grads needs a bank built by FrameBank.from_fields; for frames given directly, "
                               "bank.grad is dL/dx of those frames")
        if self.grad is None:
            raise RuntimeError("field_grads: the bank collects no gradient; call requires_grad_() before the forward")
        return fuse_inputs_adjoint(self.grad, **self._fields)

    def tangent(self, dframes: torch.Tensor) -> torch.Tensor:
        """A tangent (perturbation direction) of every frame, dframes [N, C, Hp, Wp] fp32 or bf16, packed into this bank's
        layout with the constant-1 lane 0 -> [N, Hp, Wp, c_pad] for ConvLSTM.jvp_windows."""
        N, Hp, Wp, _ = self.frames.shape
        if not dframes.is_cuda or dframes.device != self.frames.device or dframes.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("dframes must be a float32 or bfloat16 tensor on the bank's device")
        if tuple(dframes.shape) != (N, self.channels, Hp, Wp):
            raise ValueError(f"dframes has shape {tuple(dframes.shape)}, expected {(N, self.channels, Hp, Wp)}")
        if dframes.dtype == torch.bfloat16 and self.precision != "bf16":
            raise TypeError("bf16 tangents need a bf16 bank")
        out = torch.empty_like(self.frames)
        with _lib.on_device(dframes.device):
            _lib.check(_lib.load().nint_pack_frames(_DTYPES[self.precision][0], _lib.ptr(dframes.contiguous()),
                                                    _lib.X_BF16 if dframes.dtype == torch.bfloat16 else _lib.X_FP32, N,
                                                    self.channels, Hp, Wp, self.c_pad, -1, _lib.ptr(out),
                                                    _lib.stream_ptr(dframes.device)), "nint_pack_frames")
        return out

    def tangent_from_fields(self, d_levels3d: Optional[Tensor] = None, d_emis2d: Optional[Tensor] = None,
                            d_statics: Optional[Tensor] = None) -> torch.Tensor:
        """The tangent of the frames of a bank built by `from_fields` for perturbations of its raw fields (d_levels3d
        [N, L, H, W], d_emis2d [N, H, W], d_statics [S, H, W] fp32; None = zero): the linear part of the fusion -- the
        z-score without its mean, the same static channels, halo and mode -- written by the same kernel into the bank
        layout with the constant-1 lane 0, rounded as the bank is.  -> [N, Hp, Wp, c_pad] for ConvLSTM.jvp_windows."""
        if self._fields is None:
            raise RuntimeError("tangent_from_fields needs a bank built by FrameBank.from_fields; pack frame tangents with "
                               "FrameBank.tangent")
        f = self._fields
        N, Hp, Wp, _ = self.frames.shape
        L, S, H, W, dev = f["levels"], f["n_static"], f["height"], f["width"], self.frames.device
        zeros = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=dev)
        lev = zeros(N, L, H, W) if d_levels3d is None else d_levels3d
        emis = zeros(N, H, W) if d_emis2d is None else d_emis2d
        stat = (zeros(S, H, W) if d_statics is None else d_statics) if S else None
        if d_statics is not None and not S:
            raise ValueError("this bank has no static fields")
        mean0 = zeros(L + 1)
        _, _, _, _, _, _, _, stat = _check_fuse_args(lev, emis, mean0, f["std"], (Hp, Wp), f["mode"], stat)
        if tuple(lev.shape) != (N, L, H, W):
            raise ValueError(f"d_levels3d has shape {tuple(lev.shape)}, expected {(N, L, H, W)}")
        out = torch.empty_like(self.frames)
        vp = _lib.ptr
        with _lib.on_device(dev):
            _lib.check(_lib.load().nint_fuse_inputs_bank(vp(lev.contiguous()), vp(emis.contiguous()), vp(mean0),
                                                         vp(f["std"]), vp(stat) if S else None, S, N, L, H, W, Hp, Wp,
                                                         MODES[f["mode"]], _DTYPES[self.precision][0], self.c_pad, -1,
                                                         vp(out), _lib.stream_ptr(dev)), "nint_fuse_inputs_bank")
        return out

    def __len__(self):
        return self.frames.shape[0]

    def num_windows(self, seq_len: int) -> int:
        return len(self) - seq_len + 1

    def check_windows(self, win_start: torch.Tensor, seq_len: int):
        """Host-side bounds check when the indices are on the host (device indices are trusted: an out-of-range frame
        reads as zeros through TMA, it cannot fault)."""
        if not win_start.is_cuda and win_start.numel():
            lo, hi = int(win_start.min()), int(win_start.max())
            if lo < 0 or hi + seq_len > len(self):
                raise IndexError(f"window starts [{lo}, {hi}] with {seq_len} steps leave the bank of {len(self)} frames")

    def check_plan(self, plan):
        c_pad, ones, dt = plan.input_layout()
        if (c_pad, ones, dt) != (self.c_pad, self.ones_lane, self.frames.dtype) or plan.C != self.channels:
            raise ValueError("this frame bank was built for a different model (channels / precision)")

    @classmethod
    def from_frames(cls, x: torch.Tensor, precision: str = "bf16", targets: Optional[torch.Tensor] = None) -> "FrameBank":
        """x [N, C, H, W] fp32 or bf16 on the GPU (already normalised / padded, e.g. a dataset's X before windowing)."""
        if not x.is_cuda or x.dim() != 4 or x.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("x must be a CUDA tensor [N, C, H, W] of float32 or bfloat16")
        if x.dtype == torch.bfloat16 and precision != "bf16":
            raise TypeError("bf16 frames need precision='bf16'")
        N, C, H, W = x.shape
        c_pad, ones = input_layout(C)
        code, dt = _DTYPES[precision]
        frames = torch.empty((N, H, W, c_pad), dtype=dt, device=x.device)
        with _lib.on_device(x.device):
            _lib.check(_lib.load().nint_pack_frames(code, _lib.ptr(x.contiguous()),
                                                    _lib.X_BF16 if x.dtype == torch.bfloat16 else _lib.X_FP32, N, C, H, W,
                                                    c_pad, ones, _lib.ptr(frames), _lib.stream_ptr(x.device)),
                       "nint_pack_frames")
        return cls(frames, C, precision, targets)

    @classmethod
    def from_fields(cls, levels3d: torch.Tensor, emis2d: torch.Tensor, mean: torch.Tensor, std: torch.Tensor,
                    target_hw: Optional[Tuple[int, int]] = None, mode: str = "reflect",
                    statics: Optional[torch.Tensor] = None, precision: str = "bf16",
                    targets: Optional[torch.Tensor] = None) -> "FrameBank":
        """The preprocessing fusion (stack levels + emission, z-score, static attributes, geophysical halo) written
        straight into the bank by ONE kernel: levels3d [N, L, H, W], emis2d [N, H, W] raw fields -> frames
        [N, Hp, Wp, c_pad].  Same arithmetic as `fuse_inputs` followed by the model's input packing."""
        lead, L, H, W, S, Hp, Wp, statics = _check_fuse_args(levels3d, emis2d, mean, std, target_hw, mode, statics)
        if len(lead) != 1:
            raise ValueError("from_fields takes one leading frame dimension: levels3d [N, L, H, W]")
        C = L + 1 + S
        c_pad, ones = input_layout(C)
        if c_pad > 64:
            raise ValueError(f"{C} input channels: the fused bank kernel handles up to 64; use fuse_inputs + from_frames")
        code, dt = _DTYPES[precision]
        frames = torch.empty((lead[0], Hp, Wp, c_pad), dtype=dt, device=levels3d.device)
        with _lib.on_device(levels3d.device):
            _lib.check(_lib.load().nint_fuse_inputs_bank(_lib.ptr(levels3d.contiguous()), _lib.ptr(emis2d.contiguous()),
                                                         _lib.ptr(mean.contiguous()), _lib.ptr(std.contiguous()),
                                                         _lib.ptr(statics) if S else None, S, lead[0], L, H, W, Hp, Wp,
                                                         MODES[mode], code, c_pad, ones, _lib.ptr(frames),
                                                         _lib.stream_ptr(levels3d.device)), "nint_fuse_inputs_bank")
        bank = cls(frames, C, precision, targets)
        bank._fields = _adjoint_record(std, L, S, H, W, mode)
        return bank


def _check_fuse_args(levels3d, emis2d, mean, std, target_hw, mode, statics):
    if mode not in MODES:
        raise ValueError(f"mode must be one of {sorted(MODES)}")
    checked = [("levels3d", levels3d), ("emis2d", emis2d), ("mean", mean), ("std", std)]
    if statics is not None:
        checked.append(("statics", statics))
    for name, t in checked:
        if not t.is_cuda:
            raise RuntimeError(f"{name} must be a CUDA tensor: the preprocessing kernel has no CPU fallback")
        if t.dtype != torch.float32:
            raise TypeError(f"{name} must be float32 (got {t.dtype})")
        if t.device != levels3d.device:
            raise RuntimeError(f"{name} is on {t.device}, levels3d on {levels3d.device}")
    lead = tuple(levels3d.shape[:-3])
    L, H, W = levels3d.shape[-3:]
    if tuple(emis2d.shape) != lead + (H, W):
        raise ValueError(f"emis2d has shape {tuple(emis2d.shape)}, expected {lead + (H, W)}")
    if mean.numel() != L + 1 or std.numel() != L + 1:
        raise ValueError(f"mean/std need {L + 1} entries")
    S = 0
    if statics is not None:
        if statics.dim() != 3 or tuple(statics.shape[1:]) != (H, W):
            raise ValueError(f"statics has shape {tuple(statics.shape)}, expected (S, {H}, {W})")
        S = statics.shape[0]
        statics = statics.contiguous()
    Hp, Wp = (H, W) if target_hw is None else (int(target_hw[0]), int(target_hw[1]))
    return lead, L, H, W, S, Hp, Wp, statics


def normalise_static_attributes(fields: torch.Tensor) -> torch.Tensor:
    """dataset.py:100-122: every static field [S, H, W] z-scored with its own spatial mean / (population) std.  Done
    once per dataset, not per sample."""
    f = fields.to(torch.float32)
    return (f - f.mean(dim=(1, 2), keepdim=True)) / f.std(dim=(1, 2), keepdim=True, unbiased=False)


def fuse_inputs(levels3d: torch.Tensor, emis2d: torch.Tensor, mean: torch.Tensor, std: torch.Tensor,
                target_hw: Optional[Tuple[int, int]] = None, mode: str = "reflect",
                statics: Optional[torch.Tensor] = None) -> torch.Tensor:
    """levels3d [..., L, H, W], emis2d [..., H, W] (same leading dims, e.g. [T] or [B, T]), mean/std [L+1],
    statics [S, H, W] (already z-scored, `normalise_static_attributes`; appended to every frame as channels L+1..,
    dataset.py:532-533) -> [..., L+1+S, Hp, Wp] fp32 on the same CUDA device.  `target_hw=None` keeps the grid size
    (no halo).  Differentiable w.r.t. levels3d, emis2d and statics (not mean / std) when one of them requires grad:
    the backward is nint_fuse_inputs_adjoint."""
    lead, L, H, W, S, Hp, Wp, statics = _check_fuse_args(levels3d, emis2d, mean, std, target_hw, mode, statics)
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (levels3d, emis2d, statics)):
        return torch.ops.nint.fuse_inputs(levels3d, emis2d, mean, std, statics, Hp, Wp, MODES[mode])
    return _fuse_planar(levels3d, emis2d, mean, std, statics, Hp, Wp, MODES[mode])


def _fuse_planar(levels3d, emis2d, mean, std, statics, Hp, Wp, mode):
    lead = tuple(levels3d.shape[:-3])
    L, H, W = levels3d.shape[-3:]
    S = 0 if statics is None else statics.shape[0]
    frames = 1
    for d in lead:
        frames *= d
    out = torch.empty(lead + (L + 1 + S, Hp, Wp), dtype=torch.float32, device=levels3d.device)
    vp = _lib.ptr
    with _lib.on_device(levels3d.device):
        _lib.check(_lib.load().nint_fuse_inputs(vp(levels3d.contiguous()), vp(emis2d.contiguous()), vp(mean.contiguous()),
                                                vp(std.contiguous()), vp(statics) if S else None, S, frames, L, H, W, Hp, Wp,
                                                mode, vp(out), _lib.stream_ptr(levels3d.device)),
                   "nint_fuse_inputs")
    return out


@torch.library.custom_op("nint::fuse_inputs", mutates_args=(), device_types="cuda")
def _fuse_inputs_op(levels3d: Tensor, emis2d: Tensor, mean: Tensor, std: Tensor, statics: Optional[Tensor],
                    padded_height: int, padded_width: int, mode: int) -> Tensor:
    """fuse_inputs as a differentiable op (nint_fuse_inputs; backward nint_fuse_inputs_adjoint)"""
    return _fuse_planar(levels3d.detach(), emis2d.detach(), mean.detach(), std.detach(),
                        None if statics is None else statics.detach(), padded_height, padded_width, mode)


@_fuse_inputs_op.register_fake
def _(levels3d, emis2d, mean, std, statics, padded_height, padded_width, mode):
    C = levels3d.shape[-3] + 1 + (0 if statics is None else statics.shape[0])
    return levels3d.new_empty(tuple(levels3d.shape[:-3]) + (C, padded_height, padded_width))


def _fuse_setup_context(ctx, inputs, output):
    levels3d, _, _, std, statics, _, _, mode = inputs
    ctx.std, ctx.mode, ctx.lead = std, mode, tuple(levels3d.shape[:-3])
    ctx.shape = (levels3d.shape[-3], 0 if statics is None else statics.shape[0]) + tuple(levels3d.shape[-2:])


def _fuse_backward(ctx, dout):
    L, S, H, W = ctx.shape
    need = ctx.needs_input_grad
    mode = next(k for k, v in MODES.items() if v == ctx.mode)
    g = fuse_inputs_adjoint(dout.reshape((-1,) + tuple(dout.shape[-3:])), ctx.std, L, S, H, W, mode,
                            want=(need[0], need[1], need[4]))
    dl = None if g["levels3d"] is None else g["levels3d"].reshape(ctx.lead + (L, H, W))
    de = None if g["emis2d"] is None else g["emis2d"].reshape(ctx.lead + (H, W))
    return dl, de, None, None, g["statics"], None, None, None


torch.library.register_autograd("nint::fuse_inputs", _fuse_backward, setup_context=_fuse_setup_context)


def _adjoint_record(std, levels, n_static, height, width, mode):
    """what fuse_inputs_adjoint needs besides the gradient: kept by banks built from raw fields"""
    return dict(std=std.detach().contiguous().clone(), levels=int(levels), n_static=int(n_static), height=int(height),
                width=int(width), mode=mode)


def fuse_inputs_adjoint(dframes: Tensor, std: Tensor, levels: int, n_static: int, height: int, width: int,
                        mode: str = "reflect", want=(True, True, True)) -> Dict[str, Optional[Tensor]]:
    """Adjoint of `fuse_inputs` (nint_fuse_inputs_adjoint): dframes [N, levels+1+n_static, Hp, Wp] fp32 ->
    {"levels3d" [N, levels, H, W], "emis2d" [N, H, W], "statics" [n_static, H, W] summed over the N frames} (None
    where `want` says no, and for statics when there are none).  Every source element sums its halo copies in fp32 in
    padded row-major order, then the z-scored channels divide by std."""
    if mode not in MODES:
        raise ValueError(f"mode must be one of {sorted(MODES)}")
    C = levels + 1 + n_static
    if not dframes.is_cuda or dframes.dtype != torch.float32 or dframes.dim() != 4 or dframes.shape[1] != C:
        raise ValueError(f"dframes must be a CUDA fp32 tensor [N, {C}, Hp, Wp]")
    if not std.is_cuda or std.device != dframes.device or std.dtype != torch.float32 or std.numel() != levels + 1:
        raise ValueError(f"std must be {levels + 1} fp32 values on the gradient's device")
    N, _, Hp, Wp = dframes.shape
    new = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dframes.device)
    out = {"levels3d": new(N, levels, height, width) if want[0] else None,
           "emis2d": new(N, height, width) if want[1] else None,
           "statics": new(n_static, height, width) if want[2] and n_static > 0 else None}
    vp = _lib.ptr
    with _lib.on_device(dframes.device):
        _lib.check(_lib.load().nint_fuse_inputs_adjoint(vp(dframes.detach().contiguous()), vp(std.contiguous()), N, levels,
                                                        n_static, height, width, Hp, Wp, MODES[mode], vp(out["levels3d"]),
                                                        vp(out["emis2d"]), vp(out["statics"]),
                                                        _lib.stream_ptr(dframes.device)), "nint_fuse_inputs_adjoint")
    return out
