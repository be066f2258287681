"""Drop-in replacements for the reference's `model.py` ConvLSTM classes (model.py:196-274).

Same constructor signatures, parameter names/shapes (`layers.{l}.conv.weight|bias`,
`conv.weight|bias`; checkpoint contract utils.py:27,39), default initialisation and forward
contracts, so `train.py`, `utils.py` and the notebooks can `from model import ConvLSTM`
unchanged.  The arithmetic runs in libnint.so (hand-written sm_100a kernels behind the C ABI of
include/nint.h); there is no CPU or eager-PyTorch fallback.
"""
import weakref
from collections import OrderedDict
from typing import Sequence

import torch
import torch.nn as nn

from . import ops
from .engine import Plan

_MAX_CACHED_PLANS = 4
_MAX_CELL_PLANS = 256


def _deterministic_default() -> bool:
    """The reference pins run-to-run reproducibility with `seed()` (utils.py:77-88: cudnn.deterministic = True); the
    same switch (or torch.use_deterministic_algorithms) selects the fixed-order gradient reductions here."""
    return bool(torch.backends.cudnn.deterministic or torch.are_deterministic_algorithms_enabled())


class _PlanCache:
    """LRU of plans (each owns a device workspace and a ctypes handle).  Plans are derived state: copying or pickling
    the owning module (copy.deepcopy, torch.save(model), swa_utils.AveragedModel) yields an EMPTY cache."""

    def __init__(self):
        self._plans = OrderedDict()

    def get(self, key, factory):
        p = self._plans.get(key)
        if p is None:
            p = factory()
            self._plans[key] = p
            while len(self._plans) > _MAX_CACHED_PLANS:
                self._plans.popitem(last=False)
        else:
            self._plans.move_to_end(key)
        return p

    def clear(self):
        self._plans.clear()

    def __deepcopy__(self, memo):
        return type(self)()

    def __getstate__(self):
        return {}

    def __setstate__(self, state):
        self.__init__()


class _CellPlanPool(_PlanCache):
    """Training plans of a standalone cell: every step that awaits its backward owns one (its saved gates live in the
    plan's workspace), so a user loop `for t: h, c = cell(x[t], (h, c))` followed by one `backward()` works like the
    reference's autograd module.  A plan returns to the pool when its autograd node dies."""

    def __init__(self):
        super().__init__()
        self._free = {}
        self._all = []      # strong references: the op registry and the autograd nodes only hold plan ids

    def acquire(self, key, factory):
        free = self._free.setdefault(key, [])
        if free:
            return free.pop()
        if len(self._all) >= _MAX_CELL_PLANS:
            raise RuntimeError(f"more than {_MAX_CELL_PLANS} ConvLSTMCell steps are awaiting backward()")
        plan = factory()
        self._all.append(plan)
        ref = weakref.ref(plan)
        plan.release = lambda f=free, r=ref: f.append(r()) if r() is not None else None
        return plan

    def clear(self):
        super().clear()
        self._free.clear()
        self._all.clear()


class ConvLSTMCell(nn.Module):
    """model.py:196-231.  `forward(x, (h, c)) -> (h, c)`: one fused step on the GPU, differentiable w.r.t. x, h, c and
    the parameters (the step's backward is one fused gate-backward launch, two dgrad launches and one wgrad launch)."""

    def __init__(self, input_channels, hidden_channels, kernel_size, bias=True, precision="bf16"):
        super().__init__()
        self.input_channels = input_channels
        self.hidden_channels = hidden_channels
        self.kernel_size = kernel_size
        self.padding = kernel_size // 2
        self.bias = bias
        self.precision = precision
        # parameter container only (never called): same names, shapes and default init as the reference
        self.conv = nn.Conv2d(in_channels=self.input_channels + self.hidden_channels,
                              out_channels=4 * self.hidden_channels, kernel_size=self.kernel_size,
                              padding=self.padding, bias=self.bias)
        self._plans = _CellPlanPool()

    def forward(self, x, hidden_state):
        h, c = hidden_state
        if not x.is_cuda:
            raise RuntimeError("ConvLSTMCell runs on CUDA (B200) only: there is no CPU fallback")
        training = torch.is_grad_enabled() and (x.requires_grad or h.requires_grad or c.requires_grad or
                                                any(p.requires_grad for p in self.parameters()))
        B, _, H, W = x.shape
        key = (B, H, W, self.precision, x.device, training, _deterministic_default())
        if training:
            plan = self._plans.acquire(key, lambda: self._make_plan(B, H, W, x.device, True))
        else:
            plan = self._plans.get(key, lambda: self._make_plan(B, H, W, x.device, False))
        return torch.ops.nint.cell_forward(x, h, c, self.conv.weight, self.conv.bias, ops.register_plan(plan))

    def _make_plan(self, B, H, W, device, training):
        plan = Plan(B, 1, H, W, self.input_channels, [self.hidden_channels], [self.kernel_size],
                    precision=self.precision, training=training, device=device, input_grad=training,
                    deterministic=training and _deterministic_default())
        hw = torch.zeros(1, self.hidden_channels, 1, 1, device=device)
        plan.set_head(hw, torch.zeros(1, device=device))
        return plan


class ConvLSTM(nn.Module):
    """model.py:234-274.  `forward(x[B,T,C,H,W]) -> [B,1,H,W]` (head on the last layer's h at the
    last step).  `return_sequence=True` restates the commented-out variant (model.py:264,272,274)
    that test.ipynb:273 was run against: returns `(pred, hs[B,T,H,W])`.
    `precision`: "bf16" (bf16 operands, fp32 accumulate/state) or "tf32".
    x may be fp32 or (bf16 precision) bf16; `forward_windows(bank, starts)` reads the windows from an HBM-resident
    `preprocess.FrameBank` instead (dataset.py:551-637).

    Both take `hidden_state`, the initial state as a list of L pairs (h_l, c_l) [B, Hc_l, H, W] fp32 (None: zeros, for
    all layers or, as a pair of Nones, for one), and `return_state`: then the result is (out, [(h_T, c_T) per layer])
    with `out` what the call returns without it.  Gradients flow to the initial state when it requires grad and from
    any use of the final state, so windows of one long record can be chained (truncated BPTT: pass the detached final
    state of window k as the initial state of window k+1).  Precision: h0 enters the gate convolution rounded to the
    operand format like every h_t (bf16 on bf16 plans, tf32 on tf32 plans); c0 stays fp32.  Two forwards of one shape
    share a workspace, so a window must be back-propagated before the next forward of the same shape."""

    def __init__(self, input_channels, hidden_channels: Sequence[int], kernel_size: Sequence[int], num_layers,
                 precision: str = "bf16", return_sequence: bool = False):
        super().__init__()
        assert len(hidden_channels) == num_layers, "The length of hidden_channels should be equal to num_layers"
        assert len(kernel_size) == num_layers, "The length of kernel_size should be equal to num_layers"
        self.num_layers = num_layers
        self.input_channels = input_channels
        self.precision = precision
        self.return_sequence = return_sequence
        layers = []
        for i in range(self.num_layers):
            in_ch = input_channels if i == 0 else hidden_channels[i - 1]
            layers.append(ConvLSTMCell(in_ch, hidden_channels[i], kernel_size[i], precision=precision))
        self.layers = nn.ModuleList(layers)
        self.conv = nn.Conv2d(hidden_channels[-1], 1, 1)
        self._plans = _PlanCache()

    def _params(self):
        ps = []
        for cell in self.layers:
            ps += [cell.conv.weight, cell.conv.bias]
        return ps + [self.conv.weight, self.conv.bias]

    def plan_for_shape(self, B, T, H, W, device, training, set_params=True, input_grad=False, state_grad=False,
                       tangent=False, second_order=False, param_tangent=False):
        device = torch.device(device)
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        det = bool(training) and _deterministic_default()
        key = (B, T, H, W, bool(training), self.return_sequence, self.precision, device, bool(input_grad),
               bool(state_grad), det, bool(tangent), bool(second_order), bool(param_tangent))
        hidden = [c.hidden_channels for c in self.layers]
        ks = [c.kernel_size for c in self.layers]
        plan = self._plans.get(key, lambda: Plan(B, T, H, W, self.input_channels, hidden, ks, precision=self.precision,
                                                 training=training, return_sequence=self.return_sequence,
                                                 device=device, deterministic=det, input_grad=input_grad,
                                                 state_grad=state_grad, tangent=tangent, second_order=second_order,
                                                 param_tangent=param_tangent))
        if set_params:
            for l, cell in enumerate(self.layers):
                plan.set_weights(l, cell.conv.weight, cell.conv.bias)
            plan.set_head(self.conv.weight, self.conv.bias)
        return plan

    def plan_for(self, x, training, set_params=True, input_grad=False, state_grad=False, tangent=False,
                 second_order=False, param_tangent=False):
        B, T, C, H, W = x.size()
        if C != self.input_channels:
            raise ValueError(f"expected {self.input_channels} input channels, got {C}")
        return self.plan_for_shape(B, T, H, W, x.device, training, set_params, input_grad, state_grad, tangent,
                                   second_order, param_tangent)

    def _wants_grad(self, params):
        return torch.is_grad_enabled() and any(p.requires_grad for p in params)

    def _state_requires_grad(self, hidden_state):
        return (hidden_state is not None and torch.is_grad_enabled() and
                any(t is not None and t.requires_grad for pair in hidden_state for t in pair))

    def _stateful(self, op, inputs, plan, hidden_state, return_state, extra=()):
        """the *_state op from `hidden_state` (`extra`: arguments between c0 and plan_id); the result as forward
        returns it"""
        plan.check_state(hidden_state)
        pairs = hidden_state if hidden_state is not None else [(None, None)] * self.num_layers
        empty = torch.empty(0, dtype=torch.float32, device=plan.device)     # the ops' stand-in for a zero state
        h0 = [empty if h is None else h for h, _ in pairs]
        c0 = [empty if c is None else c for _, c in pairs]
        pred, seq, hT, cT = op(*inputs, self._params(), h0, c0, *extra, ops.register_plan(plan))
        out = (pred, seq) if self.return_sequence else pred
        return (out, list(zip(hT, cT))) if return_state else out

    def forward(self, x, hidden_state=None, return_state=False):
        if not x.is_cuda:
            raise RuntimeError("ConvLSTM runs on CUDA (B200) only: there is no CPU fallback; move the module and "
                               "its input to the GPU")
        params = self._params()
        need_dx = torch.is_grad_enabled() and x.requires_grad
        state_req = self._state_requires_grad(hidden_state)
        training = need_dx or state_req or self._wants_grad(params)
        # the final state is in the graph when returned from a recorded call: it may be used by the loss
        state_grad = training and (state_req or return_state)
        plan = self.plan_for(x, training, set_params=False, input_grad=need_dx,     # the op repacks the weights it is
                             state_grad=state_grad)                                  # handed
        if hidden_state is not None or return_state:
            return self._stateful(torch.ops.nint.convlstm_forward_state, (x,), plan, hidden_state, return_state)
        # torch.library op (ops.py): forward = nint_forward (T x L fused cell steps + head), autograd = nint_backward
        pred, seq = torch.ops.nint.convlstm_forward(x, params, ops.register_plan(plan))
        return (pred, seq) if self.return_sequence else pred

    def forward_windows(self, bank, win_start, seq_len, hidden_state=None, return_state=False):
        """bank: preprocess.FrameBank (frames resident in HBM in the operand layout); win_start: int tensor [B] of
        window start frames -> the same outputs as forward(x) with x[b] = frames[win_start[b] : win_start[b]+T].
        hidden_state / return_state: as in forward.
        A bank that collects gradients (bank.requires_grad_()) gets dL/dx of these windows added into bank.grad by the
        backward, under grad mode, also when no parameter requires grad."""
        params = self._params()
        starts = win_start.to(device=bank.frames.device, dtype=torch.int32).contiguous()
        bank.check_windows(win_start, seq_len)
        N, H, W, _ = bank.frames.shape
        need_dx = torch.is_grad_enabled() and bank.requires_grad
        state_req = self._state_requires_grad(hidden_state)
        training = need_dx or state_req or self._wants_grad(params)
        plan = self.plan_for_shape(starts.shape[0], int(seq_len), H, W, bank.frames.device, training,
                                   set_params=False, input_grad=need_dx,
                                   state_grad=training and (state_req or return_state))
        bank.check_plan(plan)
        if need_dx:
            return self._stateful(torch.ops.nint.convlstm_forward_bank_dx, (bank.frames, starts), plan, hidden_state,
                                  return_state, extra=(bank._anchor, bank.grad))
        if hidden_state is not None or return_state:
            return self._stateful(torch.ops.nint.convlstm_forward_bank_state, (bank.frames, starts), plan, hidden_state,
                                  return_state)
        pred, seq = torch.ops.nint.convlstm_forward_bank(bank.frames, starts, params, ops.register_plan(plan))
        return (pred, seq) if self.return_sequence else pred

    def _jvp_result(self, pred, seq, final, dpred, dseq, dfinal, return_state):
        out = (pred, seq) if self.return_sequence else pred
        dout = (dpred, dseq) if self.return_sequence else dpred
        return ((out, final), (dout, dfinal)) if return_state else (out, dout)

    @staticmethod
    def _tangent_state(plan, state_tangent):
        if not plan.check_state(state_tangent):
            return None, None
        return [h for h, _ in state_tangent], [c for _, c in state_tangent]

    def param_direction(self, direction):
        """A parameter direction as a dict keyed by named_parameters() names (`layers.{l}.conv.weight|bias`,
        `conv.weight|bias`; the format of torch.func.functional_call) -> (layers, head) for Plan.set_param_tangent.
        Missing keys are zero; unknown keys and shapes other than the parameter's raise."""
        params = dict(self.named_parameters())
        unknown = sorted(set(direction) - set(params))
        if unknown:
            raise KeyError(f"parameter direction has unknown keys {unknown}; expected names from named_parameters()")
        for name, t in direction.items():
            if tuple(t.shape) != tuple(params[name].shape):
                raise ValueError(f"direction[{name!r}] has shape {tuple(t.shape)}, expected {tuple(params[name].shape)}")

        def pair(w_name, b_name):
            dw, db = direction.get(w_name), direction.get(b_name)
            if dw is None and db is None:
                return None
            return (torch.zeros_like(params[w_name]) if dw is None else dw, db)

        layers = [pair(f"layers.{l}.conv.weight", f"layers.{l}.conv.bias") for l in range(self.num_layers)]
        return (None if all(e is None for e in layers) else layers), pair("conv.weight", "conv.bias")

    def _tangent_plan(self, plan, param_tangent):
        if param_tangent is not None:
            plan.set_param_tangent(*self.param_direction(param_tangent))

    def jvp(self, x, dx, hidden_state=None, state_tangent=None, return_state=False, param_tangent=None):
        """Forward-mode derivative at fixed parameters, the tangent-linear model of `forward`: returns (out, dout) with
        `out` what forward(x, hidden_state) returns and `dout` its derivative in the direction (dx, state_tangent), like
        torch.func.jvp's (primals_out, tangents_out).  dx [B,T,C,H,W] (None: zero); state_tangent: per layer (dh0, dc0)
        [B,Hc_l,H,W] fp32 (None: zero, for all layers or one tensor).  return_state: ((out, [(h_T, c_T)]),
        (dout, [(dh_T, dc_T)])).  A tangent pass costs about two to three forwards (DESIGN.md section 10, f7).  A
        direction is exact up to the rounding of the tangent operands (bf16 / tf32 like h), not a difference of two
        nonlinear runs.  The outputs carry no autograd graph.
        param_tangent: a direction in parameter space as well, a dict keyed by named_parameters() names (missing keys:
        zero; see param_direction), so dout = J_x dx + J_state dstate + J_theta dtheta and the result compares directly
        with torch.func.jvp(lambda p: functional_call(model, p, x), (params,), (param_tangent,)).  It costs one more
        gate GEMM per step and layer that has a direction.  For many directions on one forward (a Laplace or Lanczos
        loop) use the plan: Plan.set_param_tangent.  A call with param_tangent uses its own cached plan (the flag's
        buffers); alternating calls with and without it at one shape keep both plans' workspaces."""
        if not x.is_cuda:
            raise RuntimeError("ConvLSTM runs on CUDA (B200) only: there is no CPU fallback")
        if param_tangent is None:
            plan = self.plan_for(x, True, tangent=True)
        else:
            plan = self.plan_for(x, True, param_tangent=True)
        dh0, dc0 = self._tangent_state(plan, state_tangent)
        with torch.no_grad():
            pred, seq = plan.forward(x, hidden_state)
            final = plan.final_state() if return_state else None
            self._tangent_plan(plan, param_tangent)
            dpred, dseq, dfinal = plan.forward_tangent(dx, dh0, dc0)
        return self._jvp_result(pred, seq, final, dpred, dseq, dfinal, return_state)

    def jvp_windows(self, bank, win_start, seq_len, dbank, hidden_state=None, state_tangent=None, return_state=False,
                    param_tangent=None):
        """`jvp` over frame-bank windows (forward_windows): dbank [N,Hp,Wp,c_pad] holds the tangent of every frame of
        `bank` in its layout (FrameBank.tangent / FrameBank.tangent_from_fields), cut at the same window starts.
        param_tangent: as in `jvp`."""
        starts = win_start.to(device=bank.frames.device, dtype=torch.int32).contiguous()
        bank.check_windows(win_start, seq_len)
        N, H, W, _ = bank.frames.shape
        if param_tangent is None:
            plan = self.plan_for_shape(starts.shape[0], int(seq_len), H, W, bank.frames.device, True, tangent=True)
        else:
            plan = self.plan_for_shape(starts.shape[0], int(seq_len), H, W, bank.frames.device, True, param_tangent=True)
        bank.check_plan(plan)
        dh0, dc0 = self._tangent_state(plan, state_tangent)
        with torch.no_grad():
            pred, seq = plan.forward_bank(bank.frames, starts, hidden_state)
            final = plan.final_state() if return_state else None
            self._tangent_plan(plan, param_tangent)
            dpred, dseq, dfinal = plan.forward_tangent_bank(dbank, dh0, dc0)
        return self._jvp_result(pred, seq, final, dpred, dseq, dfinal, return_state)

    def _loss_seeds(self, loss_fn, pred, seq, dpred, dseq):
        """(loss, u, du): loss_fn at what forward returns, u = its gradient and du = its tangent in the direction the
        tangent pass gave, by torch.func on the (small) output tensors"""
        out = (pred, seq) if self.return_sequence else pred
        dout = (dpred, dseq) if self.return_sequence else dpred
        (u, loss), (du, _) = torch.func.jvp(torch.func.grad_and_value(loss_fn), (out,), (dout,))
        return loss.detach(), u, du

    def _param_results(self, plan, param_direction, wrt_params):
        """({name: grad}, {name: hvp}) of the last second-order pass when wrt_params"""
        if not wrt_params:
            return None
        g, h = plan.backward_second_order_params()
        names = [n for n, _ in self.named_parameters()]
        return dict(zip(names, g)), dict(zip(names, h))

    def hvp(self, x, dx, loss_fn, hidden_state=None, state_tangent=None, param_direction=None, wrt_params=False):
        """Second-order adjoint at fixed parameters: returns (loss, grad, hvp) with loss = loss_fn(forward(x,
        hidden_state)), grad its gradient and hvp = H v its Hessian-vector product w.r.t. (x, initial state) in the
        direction v = (dx, state_tangent), the exact Hessian including the curvature of the recurrence (not the
        Gauss-Newton part of jvp + backward).  grad and hvp are (d/dx [B,T,C,H,W], [(d/dh0, d/dc0)] per layer when
        hidden_state is given, else None).  loss_fn maps what forward returns to a scalar and must be differentiable
        twice by torch.func (MSE + L1 is: L1 has zero curvature almost everywhere).  dx / state_tangent as in `jvp`.
        Cost: a forward, a tangent pass and a second-order pass (DESIGN.md section 10, f8).  For many directions on one
        forward (Newton-CG, Lanczos) use the plan directly: plan = model.plan_for(x, True, second_order=True),
        plan.forward(x), then per direction plan.forward_tangent(...) and plan.backward_second_order(u, du), with u, du
        from the outputs as here; the forward's activations stay intact for one ordinary backward at the end.
        param_direction: a direction in parameter space as well (a dict keyed by named_parameters() names, missing keys
        zero; see param_direction), so v = (dx, state_tangent, param_direction) is a joint direction and every mixed
        block of the Hessian enters.  wrt_params=True: grad and hvp are (x part, state part, {name: tensor}) with the
        parameter block as the third entry -- the exact H_theta.v of Lanczos, sharpness, Newton-CG and influence
        functions (Plan.backward_second_order_params for many directions on one forward).  Both use a plan with
        param_tangent=True, which keeps the tangent dh and the pass's dgates of every step (DESIGN.md section 10, f9)."""
        if not x.is_cuda:
            raise RuntimeError("ConvLSTM runs on CUDA (B200) only: there is no CPU fallback")
        with_params = param_direction is not None or wrt_params
        plan = self.plan_for(x, True, second_order=True, param_tangent=with_params)
        dh0, dc0 = self._tangent_state(plan, state_tangent)
        with torch.no_grad():
            pred, seq = plan.forward(x, hidden_state)
            if with_params:
                plan.set_param_tangent(*self.param_direction(param_direction or {}))
            dpred, dseq, _ = plan.forward_tangent(dx, dh0, dc0)
        loss, u, du = self._loss_seeds(loss_fn, pred, seq, dpred, dseq)
        state = plan.check_state(hidden_state)
        gx, hx, gs, hs = plan.backward_second_order(u, du, state=state)
        pr = self._param_results(plan, param_direction, wrt_params)
        if pr is not None:
            return loss, (gx, gs, pr[0]), (hx, hs, pr[1])
        return loss, (gx, gs), (hx, hs)

    def hvp_windows(self, bank, win_start, seq_len, dbank, loss_fn, hidden_state=None, state_tangent=None,
                    param_direction=None, wrt_params=False):
        """`hvp` over frame-bank windows (forward_windows / jvp_windows): the direction of the frames is dbank
        [N,Hp,Wp,c_pad] (FrameBank.tangent / tangent_from_fields).  grad and hvp are (d/dframes [N,C,Hp,Wp] fp32, state
        pairs or None): every window's contribution is summed into the frames it read.  bank.grad is not touched.
        param_direction / wrt_params: as in `hvp`."""
        starts = win_start.to(device=bank.frames.device, dtype=torch.int32).contiguous()
        bank.check_windows(win_start, seq_len)
        N, H, W, _ = bank.frames.shape
        with_params = param_direction is not None or wrt_params
        plan = self.plan_for_shape(starts.shape[0], int(seq_len), H, W, bank.frames.device, True, second_order=True,
                                   param_tangent=with_params)
        bank.check_plan(plan)
        dh0, dc0 = self._tangent_state(plan, state_tangent)
        with torch.no_grad():
            pred, seq = plan.forward_bank(bank.frames, starts, hidden_state)
            if with_params:
                plan.set_param_tangent(*self.param_direction(param_direction or {}))
            dpred, dseq, _ = plan.forward_tangent_bank(dbank, dh0, dc0)
        loss, u, du = self._loss_seeds(loss_fn, pred, seq, dpred, dseq)
        new = lambda: torch.zeros((N, bank.channels, H, W), dtype=torch.float32, device=bank.frames.device)
        gf, hf = new(), new()
        gs, hs = plan.backward_second_order_bank(u, du, gf, hf, state=plan.check_state(hidden_state))
        pr = self._param_results(plan, param_direction, wrt_params)
        if pr is not None:
            return loss, (gf, gs, pr[0]), (hf, hs, pr[1])
        return loss, (gf, gs), (hf, hs)

    def release_workspaces(self):
        self._plans.clear()
        for cell in self.layers:
            cell._plans.clear()
