"""torch.library registration of the ConvLSTM hot path (SURVEY.md section 8b: "a thin C-ABI torch custom-op layer").

`torch.ops.nint.convlstm_forward` / `convlstm_forward_bank` / `convlstm_backward` / `cell_forward` / `cell_backward`
(and the stateful, frame-bank input-gradient and preprocessing variants below) are ordinary dispatcher ops with CUDA-only implementations that call libnint.so through `engine.Plan`; autograd,
fake-tensor tracing and CUDA-graph capture see them as opaque ops.  A plan (geometry, TMA descriptors, workspace with
the BPTT state) is host-side state the ops cannot carry in their arguments, so it travels as an integer handle into a
registry of live plans.  There is no CPU implementation on purpose: calling the ops with CPU tensors raises from the
dispatcher."""
import itertools
import weakref
from typing import List, Optional, Tuple

import torch
from torch import Tensor

_PLANS = weakref.WeakValueDictionary()
_ids = itertools.count(1)


def register_plan(plan) -> int:
    """Handle under which the ops find `plan`; the registry does not keep the plan alive."""
    op_id = getattr(plan, "op_id", None)
    if op_id is None:
        op_id = next(_ids)
        plan.op_id = op_id
        _PLANS[op_id] = plan
    return op_id


def _plan(plan_id: int):
    plan = _PLANS.get(plan_id)
    if plan is None:
        raise RuntimeError(f"ConvLSTM plan {plan_id} no longer exists (its module released the workspace)")
    return plan


def _set_params(plan, params):
    if len(params) != 2 * plan.L + 2:
        raise ValueError(f"expected {2 * plan.L + 2} parameter tensors, got {len(params)}")
    for l in range(plan.L):
        plan.set_weights(l, params[2 * l], params[2 * l + 1])
    plan.set_head(params[-2], params[-1])


@torch.library.custom_op("nint::convlstm_forward", mutates_args=(), device_types="cuda")
def convlstm_forward(x: Tensor, params: List[Tensor], plan_id: int) -> Tuple[Tensor, Tensor]:
    """model.py:253-274.  params = [layers.0.conv.weight, layers.0.conv.bias, ..., conv.weight, conv.bias];
    returns (pred [B,1,H,W], hs [B,T,H,W] or an empty tensor when the plan has no per-step head)."""
    plan = _plan(plan_id)
    _set_params(plan, params)
    pred, seq = plan.forward(x)
    return pred, (seq if seq is not None else pred.new_empty(0))


@convlstm_forward.register_fake
def _(x, params, plan_id):
    plan = _plan(plan_id)
    B, T, _, H, W = x.shape
    return (x.new_empty((B, 1, H, W), dtype=torch.float32),
            x.new_empty((B, T, H, W) if plan.return_sequence else (0,), dtype=torch.float32))


@torch.library.custom_op("nint::convlstm_forward_bank", mutates_args=(), device_types="cuda")
def convlstm_forward_bank(frames: Tensor, win_start: Tensor, params: List[Tensor], plan_id: int) -> Tuple[Tensor, Tensor]:
    """The same forward with the input read from an HBM-resident frame bank [N,H,W,c_pad] (dataset.py:551-637):
    sample b = frames win_start[b] .. win_start[b] + T - 1."""
    plan = _plan(plan_id)
    _set_params(plan, params)
    pred, seq = plan.forward_bank(frames, win_start)
    return pred, (seq if seq is not None else pred.new_empty(0))


@convlstm_forward_bank.register_fake
def _(frames, win_start, params, plan_id):
    plan = _plan(plan_id)
    B, H, W = win_start.shape[0], frames.shape[1], frames.shape[2]
    return (frames.new_empty((B, 1, H, W), dtype=torch.float32),
            frames.new_empty((B, plan.T, H, W) if plan.return_sequence else (0,), dtype=torch.float32))


@torch.library.custom_op("nint::convlstm_backward", mutates_args=(), device_types="cuda")
def convlstm_backward(dpred: Tensor, dseq: Optional[Tensor], plan_id: int, generation: int, need_dx: bool) -> List[Tensor]:
    """BPTT of the plan's last forward (train.py:109): gradients in the order of `params`, then dx when asked for."""
    plan = _plan(plan_id)
    if plan.generation != generation:
        raise RuntimeError("the activations this backward needs are gone: either a later forward() with the same shape "
                           "overwrote the ConvLSTM workspace, or this forward was already back-propagated once (BPTT "
                           "turns the saved gates into their gradients in place); run the forward again")
    gw, gb, ghw, ghb = plan.backward(dpred, dseq)
    grads = []
    for l in range(plan.L):
        grads += [gw[l], gb[l]]
    grads += [ghw, ghb]
    if need_dx:
        grads.append(plan.backward_input())
    return grads


@convlstm_backward.register_fake
def _(dpred, dseq, plan_id, generation, need_dx):
    plan = _plan(plan_id)
    out, cin = [], plan.C
    for hc, k in zip(plan.hidden, plan.ksize):
        out += [dpred.new_empty((4 * hc, cin + hc, k, k)), dpred.new_empty((4 * hc,))]
        cin = hc
    out += [dpred.new_empty((1, plan.hidden[-1], 1, 1)), dpred.new_empty((1,))]
    if need_dx:
        out.append(dpred.new_empty((plan.B, plan.T, plan.C, plan.H, plan.W)))
    return out


def _setup_context(ctx, inputs, output):
    ctx.plan_id = inputs[-1]
    ctx.generation = _plan(ctx.plan_id).generation


def _backward(ctx, dpred, dseq):
    plan = _plan(ctx.plan_id)
    need_dx = bool(ctx.needs_input_grad[0])
    if need_dx and not plan.input_grad:
        raise RuntimeError("gradient w.r.t. the input needs a plan made with input_grad=True (ConvLSTM.forward makes one "
                           "when x.requires_grad)")
    grads = convlstm_backward(dpred, dseq if plan.return_sequence else None, ctx.plan_id, ctx.generation, need_dx)
    dx = grads.pop() if need_dx else None
    return dx, grads, None


def _backward_bank(ctx, dpred, dseq):
    plan = _plan(ctx.plan_id)
    grads = convlstm_backward(dpred, dseq if plan.return_sequence else None, ctx.plan_id, ctx.generation, False)
    return None, None, grads, None


torch.library.register_autograd("nint::convlstm_forward", _backward, setup_context=_setup_context)
torch.library.register_autograd("nint::convlstm_forward_bank", _backward_bank, setup_context=_setup_context)


# ---- the same forwards from an explicit initial state, returning the final state (nn.LSTM's (h0, c0) -> (h_n, c_n)).
# h0 / c0 hold one tensor per layer [B,Hc_l,H,W]; an empty tensor stands for the zero state of that layer.
def _given(ts):
    return [None if t.numel() == 0 else t for t in ts]


def _state_outputs(plan, pred, seq):
    hT, cT = zip(*plan.final_state())
    return pred, (seq if seq is not None else pred.new_empty(0)), list(hT), list(cT)


def _state_fakes(ref, plan, B, H, W, T):
    states = [ref.new_empty((B, hc, H, W), dtype=torch.float32) for hc in plan.hidden]
    return (ref.new_empty((B, 1, H, W), dtype=torch.float32),
            ref.new_empty((B, T, H, W) if plan.return_sequence else (0,), dtype=torch.float32),
            states, [torch.empty_like(s) for s in states])


@torch.library.custom_op("nint::convlstm_forward_state", mutates_args=(), device_types="cuda")
def convlstm_forward_state(x: Tensor, params: List[Tensor], h0: List[Tensor], c0: List[Tensor],
                           plan_id: int) -> Tuple[Tensor, Tensor, List[Tensor], List[Tensor]]:
    """convlstm_forward started from (h0[l], c0[l]); returns (pred, seq, [h_T per layer], [c_T per layer])."""
    plan = _plan(plan_id)
    _set_params(plan, params)
    pred, seq = plan.forward(x, list(zip(_given(h0), _given(c0))))
    return _state_outputs(plan, pred, seq)


@convlstm_forward_state.register_fake
def _(x, params, h0, c0, plan_id):
    B, T, _, H, W = x.shape
    return _state_fakes(x, _plan(plan_id), B, H, W, T)


@torch.library.custom_op("nint::convlstm_forward_bank_state", mutates_args=(), device_types="cuda")
def convlstm_forward_bank_state(frames: Tensor, win_start: Tensor, params: List[Tensor], h0: List[Tensor],
                                c0: List[Tensor], plan_id: int) -> Tuple[Tensor, Tensor, List[Tensor], List[Tensor]]:
    """convlstm_forward_bank started from (h0[l], c0[l]); returns (pred, seq, [h_T per layer], [c_T per layer])."""
    plan = _plan(plan_id)
    _set_params(plan, params)
    pred, seq = plan.forward_bank(frames, win_start, list(zip(_given(h0), _given(c0))))
    return _state_outputs(plan, pred, seq)


@convlstm_forward_bank_state.register_fake
def _(frames, win_start, params, h0, c0, plan_id):
    plan = _plan(plan_id)
    return _state_fakes(frames, plan, win_start.shape[0], frames.shape[1], frames.shape[2], plan.T)


@torch.library.custom_op("nint::convlstm_backward_state", mutates_args=(), device_types="cuda")
def convlstm_backward_state(dpred: Optional[Tensor], dseq: Optional[Tensor], dh_T: List[Tensor], dc_T: List[Tensor],
                            plan_id: int, generation: int, need_dx: bool, need_state: bool) -> List[Tensor]:
    """convlstm_backward with upstream gradients of the final state (an empty tensor: none): the gradients in the order
    of `params`, then dx when asked for, then [dh0 per layer] + [dc0 per layer] when asked for."""
    plan = _plan(plan_id)
    if plan.generation != generation:
        raise RuntimeError("the activations this backward needs are gone: either a later forward() with the same shape "
                           "overwrote the ConvLSTM workspace, or this forward was already back-propagated once (BPTT "
                           "turns the saved gates into their gradients in place); run the forward again")
    gw, gb, ghw, ghb = plan.backward(dpred, dseq, dh_T=_given(dh_T), dc_T=_given(dc_T))
    grads = []
    for l in range(plan.L):
        grads += [gw[l], gb[l]]
    grads += [ghw, ghb]
    if need_dx:
        grads.append(plan.backward_input())
    if need_state:
        dh0, dc0 = plan.backward_initial_state()
        grads += dh0 + dc0
    return grads


@convlstm_backward_state.register_fake
def _(dpred, dseq, dh_T, dc_T, plan_id, generation, need_dx, need_state):
    plan = _plan(plan_id)
    ref = dh_T[0]
    out, cin = [], plan.C
    for hc, k in zip(plan.hidden, plan.ksize):
        out += [ref.new_empty((4 * hc, cin + hc, k, k)), ref.new_empty((4 * hc,))]
        cin = hc
    out += [ref.new_empty((1, plan.hidden[-1], 1, 1)), ref.new_empty((1,))]
    if need_dx:
        out.append(ref.new_empty((plan.B, plan.T, plan.C, plan.H, plan.W)))
    if need_state:
        out += [ref.new_empty((plan.B, hc, plan.H, plan.W)) for hc in plan.hidden] * 2
    return out


def _setup_context_state(ctx, inputs, output):
    _setup_context(ctx, inputs, output)
    ctx.set_materialize_grads(False)     # an unused output (pred, or a layer's h_T / c_T) contributes no launch


def _backward_state_common(ctx, dpred, dseq, dh_T, dc_T, need_dx, needs_h0, needs_c0):
    plan = _plan(ctx.plan_id)
    need_state = any(needs_h0) or any(needs_c0)
    if need_state and not plan.state_grad:
        raise RuntimeError("gradient w.r.t. the initial state needs a plan made with state_grad=True (ConvLSTM.forward "
                           "makes one when the state requires grad)")
    empty = lambda: torch.empty(0, dtype=torch.float32, device=plan.device)
    grads = convlstm_backward_state(dpred, dseq if plan.return_sequence else None,
                                    [empty() if g is None else g for g in dh_T], [empty() if g is None else g for g in dc_T],
                                    ctx.plan_id, ctx.generation, need_dx, need_state)
    dh0 = dc0 = [None] * plan.L
    if need_state:
        dh0 = [g if n else None for g, n in zip(grads[-2 * plan.L:-plan.L], needs_h0)]
        dc0 = [g if n else None for g, n in zip(grads[-plan.L:], needs_c0)]
        del grads[-2 * plan.L:]
    dx = grads.pop() if need_dx else None
    return dx, grads, dh0, dc0


def _backward_state(ctx, dpred, dseq, dh_T, dc_T):
    plan = _plan(ctx.plan_id)
    need_dx = bool(ctx.needs_input_grad[0])
    if need_dx and not plan.input_grad:
        raise RuntimeError("gradient w.r.t. the input needs a plan made with input_grad=True (ConvLSTM.forward makes one "
                           "when x.requires_grad)")
    dx, grads, dh0, dc0 = _backward_state_common(ctx, dpred, dseq, dh_T, dc_T, need_dx, ctx.needs_input_grad[2],
                                                 ctx.needs_input_grad[3])
    return dx, grads, dh0, dc0, None


def _backward_bank_state(ctx, dpred, dseq, dh_T, dc_T):
    _, grads, dh0, dc0 = _backward_state_common(ctx, dpred, dseq, dh_T, dc_T, False, ctx.needs_input_grad[3],
                                                ctx.needs_input_grad[4])
    return None, None, grads, dh0, dc0, None


torch.library.register_autograd("nint::convlstm_forward_state", _backward_state, setup_context=_setup_context_state)
torch.library.register_autograd("nint::convlstm_forward_bank_state", _backward_bank_state,
                                setup_context=_setup_context_state)


# ---- a frame-bank forward whose input gradient is wanted: its backward adds dL/dx of every window into the gradient
# of the bank's frames (FrameBank.grad).  `anchor` is a zero-size leaf of the bank that requires grad, so autograd
# records the node even when no parameter or state does (sensitivity maps of a frozen model); `dframes` is the bank's
# gradient [N,C,Hp,Wp] fp32, which the forward only hands to the backward.
@torch.library.custom_op("nint::convlstm_forward_bank_dx", mutates_args=(), device_types="cuda")
def convlstm_forward_bank_dx(frames: Tensor, win_start: Tensor, params: List[Tensor], h0: List[Tensor],
                             c0: List[Tensor], anchor: Tensor, dframes: Tensor,
                             plan_id: int) -> Tuple[Tensor, Tensor, List[Tensor], List[Tensor]]:
    """convlstm_forward_bank_state on a plan made with input_grad=True; returns (pred, seq, [h_T], [c_T])."""
    plan = _plan(plan_id)
    _set_params(plan, params)
    pred, seq = plan.forward_bank(frames, win_start, list(zip(_given(h0), _given(c0))))
    return _state_outputs(plan, pred, seq)


@convlstm_forward_bank_dx.register_fake
def _(frames, win_start, params, h0, c0, anchor, dframes, plan_id):
    plan = _plan(plan_id)
    return _state_fakes(frames, plan, win_start.shape[0], frames.shape[1], frames.shape[2], plan.T)


@torch.library.custom_op("nint::bank_input_grad_", mutates_args=("dframes",), device_types="cuda")
def bank_input_grad_(dframes: Tensor, plan_id: int, generation: int) -> None:
    """dframes[win_start[b] + t] += dL/dx[b, t] of the plan's last backward, which must be the one that took the plan to
    `generation` (nint_backward_input_bank)."""
    plan = _plan(plan_id)
    if plan.generation != generation:
        raise RuntimeError("the frame-bank input gradient must follow the backward of its forward at once")
    plan.backward_input_bank(dframes)


@bank_input_grad_.register_fake
def _(dframes, plan_id, generation):
    return None


def _setup_context_bank_dx(ctx, inputs, output):
    _setup_context_state(ctx, inputs, output)
    ctx.dframes = inputs[6]      # not saved for backward: later backwards mutate it, and this one adds to it


def _backward_bank_dx(ctx, dpred, dseq, dh_T, dc_T):
    _, grads, dh0, dc0 = _backward_state_common(ctx, dpred, dseq, dh_T, dc_T, False, ctx.needs_input_grad[3],
                                                ctx.needs_input_grad[4])
    bank_input_grad_(ctx.dframes, ctx.plan_id, ctx.generation + 1)     # the backward above bumped the generation once
    return None, None, grads, dh0, dc0, None, None, None


torch.library.register_autograd("nint::convlstm_forward_bank_dx", _backward_bank_dx, setup_context=_setup_context_bank_dx)


# ---- ConvLSTMCell (model.py:216-231): one fused step from an explicit state, differentiable w.r.t. x, h, c and the
# parameters like the reference's autograd module
@torch.library.custom_op("nint::cell_forward", mutates_args=(), device_types="cuda")
def cell_forward(x: Tensor, h: Tensor, c: Tensor, weight: Tensor, bias: Optional[Tensor],
                 plan_id: int) -> Tuple[Tensor, Tensor]:
    plan = _plan(plan_id)
    plan.set_weights(0, weight, bias)
    return plan.cell_forward(x, h, c)


@cell_forward.register_fake
def _(x, h, c, weight, bias, plan_id):
    return torch.empty_like(h), torch.empty_like(c)


@torch.library.custom_op("nint::cell_backward", mutates_args=(), device_types="cuda")
def cell_backward(dh: Optional[Tensor], dc: Optional[Tensor], plan_id: int, generation: int) -> List[Tensor]:
    """[dx, dh_in, dc_in, grad_weight, grad_bias] of the plan's last cell_forward."""
    plan = _plan(plan_id)
    if plan.generation != generation:
        raise RuntimeError("the activations of this ConvLSTMCell step are gone (already back-propagated once)")
    return list(plan.cell_backward(dh, dc))


@cell_backward.register_fake
def _(dh, dc, plan_id, generation):
    plan = _plan(plan_id)
    ref = dh if dh is not None else dc
    hc, k = plan.hidden[0], plan.ksize[0]
    shape = (plan.B, hc, plan.H, plan.W)
    return [ref.new_empty((plan.B, plan.C, plan.H, plan.W)), ref.new_empty(shape), ref.new_empty(shape),
            ref.new_empty((4 * hc, plan.C + hc, k, k)), ref.new_empty((4 * hc,))]


class _CellToken:
    """Dies with the autograd node of one cell step: returns the step's plan to the cell's pool."""


def _cell_setup_context(ctx, inputs, output):
    ctx.plan_id = inputs[-1]
    plan = _plan(ctx.plan_id)
    ctx.generation = plan.generation
    ctx.has_bias = inputs[4] is not None
    release = getattr(plan, "release", None)
    if release is not None:        # training plans come from ConvLSTMCell's pool (one plan per step awaiting backward)
        ctx.token = _CellToken()
        weakref.finalize(ctx.token, release)


def _cell_backward(ctx, dh, dc):
    plan = _plan(ctx.plan_id)
    if not plan.training:
        raise RuntimeError("this ConvLSTMCell step ran without autograd state (torch.no_grad or no tensor required grad)")
    if dh is None and dc is None:
        return None, None, None, None, None, None
    dx, dhi, dci, gw, gb = cell_backward(dh, dc, ctx.plan_id, ctx.generation)
    return dx, dhi, dci, gw, (gb if ctx.has_bias else None), None


torch.library.register_autograd("nint::cell_forward", _cell_backward, setup_context=_cell_setup_context)
