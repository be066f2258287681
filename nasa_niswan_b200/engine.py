"""Host-side plan object: one `nint_plan` (include/nint.h) plus the torch-allocated workspace it
is bound to.  PyTorch is plumbing here (device memory, streams); every byte of compute happens
in libnint.so."""
import ctypes
from typing import List, Optional, Sequence

import torch

from . import _lib

PRECISIONS = {"bf16": _lib.DTYPE_BF16, "tf32": _lib.DTYPE_TF32, "fp32": _lib.DTYPE_TF32}

_ptr = _lib.ptr


class Plan:
    """Geometry + workspace for `ConvLSTM(in_channels, hidden, ksize, L)` on inputs [B,T,C,H,W].

    Every libnint call runs under `torch.cuda.device(self.device)` on torch's current stream of THAT device, and every
    tensor handed in must live on it: the library launches on the CUDA runtime's current device."""

    def __init__(self, batch: int, seq_len: int, height: int, width: int, in_channels: int,
                 hidden: Sequence[int], ksize: Sequence[int], precision: str = "bf16", training: bool = False,
                 return_sequence: bool = False, device=None, deterministic: bool = False, input_grad: bool = False,
                 state_grad: bool = False, tangent: bool = False, second_order: bool = False,
                 param_tangent: bool = False):
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(PRECISIONS)}")
        if len(hidden) != len(ksize):
            raise ValueError("hidden and ksize must have the same length")
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: the ConvLSTM hot path has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.B, self.T, self.H, self.W, self.C = batch, seq_len, height, width, in_channels
        self.hidden, self.ksize, self.L = list(hidden), list(ksize), len(hidden)
        self.training, self.return_sequence, self.precision = bool(training), bool(return_sequence), precision
        self.deterministic, self.input_grad, self.state_grad = bool(deterministic), bool(input_grad), bool(state_grad)
        self.second_order, self.param_tangent = bool(second_order), bool(param_tangent)
        # the second-order pass reads the tangent pass's history; a parameter direction rides in the tangent pass
        self.tangent = bool(tangent) or self.second_order or self.param_tangent
        cfg = _lib.NintConfig()
        cfg.batch, cfg.seq_len, cfg.height, cfg.width = batch, seq_len, height, width
        cfg.in_channels, cfg.num_layers = in_channels, self.L
        for i, (h, k) in enumerate(zip(hidden, ksize)):
            cfg.hidden[i], cfg.ksize[i] = h, k
        cfg.dtype, cfg.training, cfg.return_sequence = PRECISIONS[precision], int(training), int(return_sequence)
        cfg.flags = ((_lib.FLAG_DETERMINISTIC if deterministic else 0) | (_lib.FLAG_INPUT_GRAD if input_grad else 0) |
                     (_lib.FLAG_STATE_GRAD if state_grad else 0) | (_lib.FLAG_TANGENT if tangent else 0) |
                     (_lib.FLAG_SECOND_ORDER if second_order else 0) | (_lib.FLAG_PARAM_TANGENT if param_tangent else 0))
        self._h = ctypes.c_void_p()
        _lib.check(self.lib.nint_plan_create(ctypes.byref(cfg), ctypes.byref(self._h)), "nint_plan_create")
        self.workspace_bytes = self.lib.nint_plan_workspace_bytes(self._h)
        with _lib.on_device(self.device):
            self.workspace = torch.empty(self.workspace_bytes, dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.nint_plan_bind(self._h, _ptr(self.workspace), self.workspace_bytes, self._stream()),
                       "nint_plan_bind")
        self.generation = 0          # bumped by every forward and every backward: BPTT consumes the saved activations
        self._weight_keys = [None] * (self.L + 1)
        self._keep = None            # tensors the queued kernels still read (frame bank, window indices)
        self._tkeep = None           # the tangent frames of the last forward_tangent_bank (the params call reads them)
        self._stateful = False       # the last forward was given an initial state (it stays in the workspace)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self.lib.nint_plan_destroy(h)

    def _stream(self):
        return _lib.stream_ptr(self.device)

    def _check_dev(self, t: torch.Tensor, name: str, shape=None, dtypes=(torch.float32,)):
        if not t.is_cuda:
            raise RuntimeError(f"{name} must be a CUDA tensor: the ConvLSTM hot path has no CPU fallback")
        if t.device != self.device:
            raise RuntimeError(f"{name} is on {t.device} but this plan (workspace, parameters) lives on {self.device}")
        if t.dtype not in dtypes:
            raise TypeError(f"{name} must be {' or '.join(str(d) for d in dtypes)} (got {t.dtype})")
        if shape is not None and tuple(t.shape) != tuple(shape):
            raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {tuple(shape)}")

    def input_layout(self):
        """(c_pad, ones_lane, torch dtype) of the channels-last operand layout a frame bank for this plan must have."""
        c_pad, ones, eb = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        _lib.check(self.lib.nint_plan_input_layout(self._h, ctypes.byref(c_pad), ctypes.byref(ones), ctypes.byref(eb)),
                   "nint_plan_input_layout")
        return c_pad.value, ones.value, (torch.bfloat16 if eb.value == 2 else torch.float32)

    # ---- parameters
    def set_weights(self, layer: int, weight: torch.Tensor, bias: Optional[torch.Tensor], force=True):
        """Repacks the fp32 OIHW masters into operand panels (two small kernels).  Done on EVERY call by default:
        tensor version counters are not a safe cache key -- torch's fused optimizers update parameters in place
        without bumping them, and a stale panel cache silently trains / evaluates with old weights."""
        key = (weight.data_ptr(), weight._version, None if bias is None else (bias.data_ptr(), bias._version))
        if not force and self._weight_keys[layer] == key:
            return
        hc = self.hidden[layer]
        cin = self.C if layer == 0 else self.hidden[layer - 1]
        self._check_dev(weight, "weight", (4 * hc, cin + hc, self.ksize[layer], self.ksize[layer]))
        if bias is not None:
            self._check_dev(bias, "bias", (4 * hc,))
        w = weight.detach().contiguous()
        b = None if bias is None else bias.detach().contiguous()
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_plan_set_weights(self._h, layer, _ptr(w), _ptr(b), self._stream()),
                       "nint_plan_set_weights")
        self._weight_keys[layer] = key

    def set_head(self, weight: torch.Tensor, bias: torch.Tensor, force=True):
        key = (weight.data_ptr(), weight._version, bias.data_ptr(), bias._version)
        if not force and self._weight_keys[self.L] == key:
            return
        self._check_dev(weight, "head weight", (1, self.hidden[-1], 1, 1))
        self._check_dev(bias, "head bias", (1,))
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_plan_set_head(self._h, _ptr(weight.detach().contiguous()),
                                                   _ptr(bias.detach().contiguous()), self._stream()), "nint_plan_set_head")
        self._weight_keys[self.L] = key

    # ---- state
    def reset_state(self):
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_plan_reset_state(self._h, self._stream()), "nint_plan_reset_state")
        self._stateful = False

    def _state_shape(self, layer: int):
        return (self.B, self.hidden[layer], self.H, self.W)

    def check_state(self, state) -> bool:
        """Validates an initial state (see _initial_state); True when it holds at least one tensor."""
        if state is None:
            return False
        state = list(state)
        if len(state) != self.L or not all(isinstance(pair, (tuple, list)) and len(pair) == 2 for pair in state):
            raise ValueError(f"the initial state must be a list of {self.L} (h, c) pairs, one per layer")
        for l, (h, c) in enumerate(state):
            for t, name in ((h, f"h0[{l}]"), (c, f"c0[{l}]")):
                if t is not None:
                    self._check_dev(t, name, self._state_shape(l))
        return any(t is not None for pair in state for t in pair)

    def _initial_state(self, state):
        """Makes `state` the initial state of the next forward: None, or per layer (h, c) [B,Hc_l,H,W] fp32 where a
        missing tensor (None) means zeros.  A plan keeps a state it was given, and plans are cached and shared, so a
        forward without a state resets the one an earlier forward was given; otherwise it issues no call."""
        given = self.check_state(state)
        if self._stateful:
            self.reset_state()
        if not given:
            return
        for l, (h, c) in enumerate(state):
            if h is None and c is None:
                continue
            shape = self._state_shape(l)
            zero = lambda: torch.zeros(shape, dtype=torch.float32, device=self.device)
            self.set_state(l, zero() if h is None else h, zero() if c is None else c)
        self._stateful = True

    def set_state(self, layer: int, h: torch.Tensor, c: torch.Tensor):
        shape = (self.B, self.hidden[layer], self.H, self.W)
        self._check_dev(h, "h", shape)
        self._check_dev(c, "c", shape)
        h, c = h.detach().contiguous(), c.detach().contiguous()
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_plan_set_state(self._h, layer, _ptr(h), _ptr(c), self._stream()), "nint_plan_set_state")

    def get_state(self, layer: int):
        shape = (self.B, self.hidden[layer], self.H, self.W)
        h = torch.empty(shape, dtype=torch.float32, device=self.device)
        c = torch.empty(shape, dtype=torch.float32, device=self.device)
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_plan_get_state(self._h, layer, _ptr(h), _ptr(c), self._stream()), "nint_plan_get_state")
        return h, c

    def final_state(self):
        """[(h_T, c_T) per layer] of the last forward, fp32 [B,Hc_l,H,W]"""
        return [self.get_state(l) for l in range(self.L)]

    # ---- compute
    def _outputs(self):
        pred = torch.empty((self.B, 1, self.H, self.W), dtype=torch.float32, device=self.device)
        seq = (torch.empty((self.B, self.T, self.H, self.W), dtype=torch.float32, device=self.device)
               if self.return_sequence else None)
        return pred, seq

    def forward(self, x: torch.Tensor, state=None):
        """x [B,T,C,H,W] fp32, or bf16 on a bf16 plan (host-staged windows: half the PCIe bytes, identical results).
        state: optional initial [(h, c) per layer] (see _initial_state); None starts from zeros."""
        self._check_dev(x, "x", (self.B, self.T, self.C, self.H, self.W), dtypes=(torch.float32, torch.bfloat16))
        if x.dtype == torch.bfloat16 and self.precision != "bf16":
            raise TypeError("bf16 inputs need precision='bf16' (a tf32 plan would lose input precision)")
        x = x.detach().contiguous()
        self._initial_state(state)
        self._keep = self._tkeep = None     # no frame bank behind this forward
        pred, seq = self._outputs()
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_forward_ex(self._h, _ptr(x), _lib.X_BF16 if x.dtype == torch.bfloat16 else _lib.X_FP32,
                                                _ptr(pred), _ptr(seq), self._stream()), "nint_forward")
        self.generation += 1
        return pred, seq

    def forward_bank(self, frames: torch.Tensor, win_start: torch.Tensor, state=None):
        """frames: frame bank [N,H,W,c_pad] in this plan's operand layout (preprocess.FrameBank); win_start: int32 [B]
        on the device -- sample b reads frames win_start[b] .. win_start[b]+T-1 through the TMA descriptors.
        state: as in forward."""
        c_pad, _, dt = self.input_layout()
        if frames.dim() != 4 or tuple(frames.shape[1:]) != (self.H, self.W, c_pad):
            raise ValueError(f"frame bank has shape {tuple(frames.shape)}, expected (N, {self.H}, {self.W}, {c_pad})")
        self._check_dev(frames, "frame bank", dtypes=(dt,))
        self._check_dev(win_start, "win_start", (self.B,), dtypes=(torch.int32,))
        if not frames.is_contiguous() or not win_start.is_contiguous():
            raise ValueError("frame bank and win_start must be contiguous")
        self._initial_state(state)
        pred, seq = self._outputs()
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_forward_bank(self._h, _ptr(frames), frames.shape[0], _ptr(win_start), _ptr(pred),
                                                  _ptr(seq), self._stream()), "nint_forward_bank")
        self._keep = (frames, win_start)    # the backward kernels read both again
        self._tkeep = None
        self.generation += 1
        return pred, seq

    def _grad_buffers(self, out):
        gw: List[torch.Tensor] = []
        gb: List[torch.Tensor] = []
        if out is not None:
            gw, gb, ghw, ghb = out
            cin = self.C
            for l, (hc, k) in enumerate(zip(self.hidden, self.ksize)):
                self._check_dev(gw[l], "grad weight", (4 * hc, cin + hc, k, k))
                self._check_dev(gb[l], "grad bias", (4 * hc,))
                cin = hc
            self._check_dev(ghw, "grad head weight", (1, self.hidden[-1], 1, 1))
            self._check_dev(ghb, "grad head bias", (1,))
            if not all(t.is_contiguous() for t in [*gw, *gb, ghw, ghb]):
                raise ValueError("gradient outputs must be contiguous")
        else:
            cin = self.C
            for hc, k in zip(self.hidden, self.ksize):
                gw.append(torch.empty((4 * hc, cin + hc, k, k), dtype=torch.float32, device=self.device))
                gb.append(torch.empty((4 * hc,), dtype=torch.float32, device=self.device))
                cin = hc
            ghw = torch.empty((1, self.hidden[-1], 1, 1), dtype=torch.float32, device=self.device)
            ghb = torch.empty((1,), dtype=torch.float32, device=self.device)
        return gw, gb, ghw, ghb

    def backward(self, dpred: Optional[torch.Tensor], dseq: Optional[torch.Tensor] = None, out=None, on_ready=None,
                 dh_T=None, dc_T=None):
        """Returns ([grad_weight_l], [grad_bias_l], grad_head_weight, grad_head_bias).  `out`: optional
        (gw list, gb list, ghw, ghb) of preallocated contiguous fp32 tensors the gradients are written into
        (e.g. views of one flat all-reduce buffer).  `on_ready(i)`: called as soon as the kernels producing a
        gradient bucket are queued on the current stream -- i = L for the head, then i = L-1 .. 0 for the layers.
        dh_T / dc_T: optional per-layer dL/dh_T, dL/dc_T [B,Hc_l,H,W] of the final state (entries may be None; plans
        made with state_grad=True); backward_initial_state() then gives dL/dh0, dL/dc0.
        BPTT turns the saved gates into their gradients in place: one backward per forward."""
        if dseq is not None:
            dseq = dseq.detach().contiguous().clone() if dpred is not None else dseq.detach().contiguous()
            self._check_dev(dseq, "dseq", (self.B, self.T, self.H, self.W))
            if dpred is not None:   # pred is seq[:, -1]: fold its gradient in
                dseq[:, -1] += dpred.detach().reshape(self.B, self.H, self.W)
                dpred = None
        if dpred is not None:
            dpred = dpred.detach().contiguous()
            self._check_dev(dpred, "dpred", (self.B, 1, self.H, self.W))
        dh_T, dc_T = self._state_table(dh_T, "dh_T"), self._state_table(dc_T, "dc_T")
        gw, gb, ghw, ghb = self._grad_buffers(out)
        self.generation += 1        # the saved activations are consumed: a second backward of the same forward must fail
        state_in = dh_T is not None or dc_T is not None
        with _lib.on_device(self.device):
            if on_ready is None and not state_in:
                arr_w = (ctypes.c_void_p * self.L)(*[t.data_ptr() for t in gw])
                arr_b = (ctypes.c_void_p * self.L)(*[t.data_ptr() for t in gb])
                _lib.check(self.lib.nint_backward(self._h, _ptr(dpred), _ptr(dseq), arr_w, arr_b, _ptr(ghw), _ptr(ghb),
                                                  self._stream()), "nint_backward")
                return gw, gb, ghw, ghb
            # staged: the caller hears about every finished gradient bucket (the head's after BPTT, then one layer at a
            # time, top layer first) while the following wgrad kernels are still queued -- nint.h nint_backward_bptt/_wgrad
            if state_in:
                _lib.check(self.lib.nint_backward_bptt_state(self._h, _ptr(dpred), _ptr(dseq), self._ptr_table(dh_T),
                                                             self._ptr_table(dc_T), _ptr(ghw), _ptr(ghb), self._stream()),
                           "nint_backward_bptt_state")
            else:
                _lib.check(self.lib.nint_backward_bptt(self._h, _ptr(dpred), _ptr(dseq), _ptr(ghw), _ptr(ghb),
                                                       self._stream()), "nint_backward_bptt")
            notify = on_ready or (lambda i: None)
            notify(self.L)
            for l in range(self.L - 1, -1, -1):
                _lib.check(self.lib.nint_backward_wgrad(self._h, l, _ptr(gw[l]), _ptr(gb[l]), self._stream()),
                           "nint_backward_wgrad")
                notify(l)
        return gw, gb, ghw, ghb

    def _state_table(self, ts, name):
        """per-layer state gradients -> contiguous tensors (None where absent), or None when none is given"""
        if ts is None or all(t is None for t in ts):
            return None
        if len(ts) != self.L:
            raise ValueError(f"{name} has {len(ts)} layers, expected {self.L}")
        out = []
        for l, t in enumerate(ts):
            if t is not None:
                self._check_dev(t, f"{name}[{l}]", self._state_shape(l))
                t = t.detach().contiguous()
            out.append(t)
        return out

    def _ptr_table(self, ts):
        return None if ts is None else (ctypes.c_void_p * self.L)(*[None if t is None else t.data_ptr() for t in ts])

    def backward_initial_state(self):
        """([dL/dh0_l], [dL/dc0_l]) fp32 [B,Hc_l,H,W] of the last backward (plans made with state_grad=True); call after
        `backward`."""
        new = lambda l: torch.empty(self._state_shape(l), dtype=torch.float32, device=self.device)
        dh0 = [new(l) for l in range(self.L)]
        dc0 = [new(l) for l in range(self.L)]
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_backward_initial_state(self._h, self._ptr_table(dh0), self._ptr_table(dc0),
                                                            self._stream()), "nint_backward_initial_state")
        return dh0, dc0

    def backward_input(self) -> torch.Tensor:
        """dx [B,T,C,H,W] of the last backward (plans made with input_grad=True); call after `backward`."""
        dx = torch.empty((self.B, self.T, self.C, self.H, self.W), dtype=torch.float32, device=self.device)
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_backward_input(self._h, _ptr(dx), self._stream()), "nint_backward_input")
        return dx

    def backward_input_bank(self, dframes: torch.Tensor):
        """Adds dL/dx of the last backward into `dframes` [N,C,H,W] fp32, the gradient of the N frames of the bank the
        last forward read (forward_bank): dframes[win_start[b] + t] += dx[b, t], in increasing t, then b (plans made
        with input_grad=True; call after `backward`)."""
        if self._keep is None:
            raise RuntimeError("backward_input_bank: the last forward did not read a frame bank (forward_bank)")
        self._check_dev(dframes, "dframes", (self._keep[0].shape[0], self.C, self.H, self.W))
        if not dframes.is_contiguous():
            raise ValueError("dframes must be contiguous")
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_backward_input_bank(self._h, _ptr(dframes), self._stream()), "nint_backward_input_bank")

    # ---- tangent-linear model (plans made with training=True, tangent=True)
    def _tangent_outputs(self, dh0, dc0):
        dh0, dc0 = self._state_table(dh0, "dh0"), self._state_table(dc0, "dc0")
        dpred, dseq = self._outputs()
        new = lambda l: torch.empty(self._state_shape(l), dtype=torch.float32, device=self.device)
        dh_T = [new(l) for l in range(self.L)]
        dc_T = [new(l) for l in range(self.L)]
        return dh0, dc0, dpred, dseq, dh_T, dc_T

    def set_param_tangent(self, layers=None, head=None):
        """Makes dtheta the parameter direction of the following forward_tangent[_bank] calls (plans made with
        param_tangent=True): layers = per layer (dW [4Hc, Cin+Hc, k, k], db [4Hc] or None) or None, head = (dw
        [1,Hc_last,1,1], db [1] or None) or None, shapes as set_weights / set_head; a missing entry is zero.  Replaces the
        whole previous direction.  One forward serves many directions:

            plan.forward(x)
            for layers, head in directions:
                plan.set_param_tangent(layers, head)
                dpred, dseq, dstate = plan.forward_tangent(dx, dh0, dc0)    # J (dx, dh0, dc0, dtheta)
            plan.clear_param_tangent()
            plan.backward(dpred_seed)                                       # one ordinary backward at the end
        """
        self.clear_param_tangent()
        if layers is not None and len(layers) != self.L:
            raise ValueError(f"layers has {len(layers)} entries, expected {self.L}")
        checked = []
        cin = self.C
        for l, entry in enumerate(layers or [None] * self.L):
            hc, k = self.hidden[l], self.ksize[l]
            if entry is not None:
                dw, db = entry
                self._check_dev(dw, f"weight tangent [{l}]", (4 * hc, cin + hc, k, k))
                if db is not None:
                    self._check_dev(db, f"bias tangent [{l}]", (4 * hc,))
                checked.append((l, dw.detach().contiguous(), None if db is None else db.detach().contiguous()))
            cin = hc
        if head is not None:
            hw, hb = head
            self._check_dev(hw, "head weight tangent", (1, self.hidden[-1], 1, 1))
            if hb is not None:
                self._check_dev(hb, "head bias tangent", (1,))
            head = (hw.detach().contiguous(), None if hb is None else hb.detach().contiguous())
        with _lib.on_device(self.device):
            for l, dw, db in checked:
                _lib.check(self.lib.nint_plan_set_weight_tangent(self._h, l, _ptr(dw), _ptr(db), self._stream()),
                           "nint_plan_set_weight_tangent")
            if head is not None:
                _lib.check(self.lib.nint_plan_set_head_tangent(self._h, _ptr(head[0]), _ptr(head[1]), self._stream()),
                           "nint_plan_set_head_tangent")

    def clear_param_tangent(self):
        """Zero parameter direction: forward_tangent is J (dx, dh0, dc0) at fixed parameters again."""
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_plan_clear_param_tangent(self._h, self._stream()), "nint_plan_clear_param_tangent")

    def forward_tangent(self, dx: Optional[torch.Tensor] = None, dh0=None, dc0=None):
        """J v of the last `forward` for v = (dx [B,T,C,H,W], per-layer dh0 / dc0 [B,Hc_l,H,W]; None = zero), plus the
        parameter direction set by set_param_tangent (param_tangent plans; else at fixed parameters): returns (dpred [B,1,H,W], dseq [B,T,H,W] or None, [(dh_T, dc_T) per layer]).  The forward's saved
        activations are only read: more tangents, and then one `backward`, of the same forward may follow."""
        if dx is not None:
            self._check_dev(dx, "dx", (self.B, self.T, self.C, self.H, self.W), dtypes=(torch.float32, torch.bfloat16))
            if dx.dtype == torch.bfloat16 and self.precision != "bf16":
                raise TypeError("bf16 tangents need precision='bf16'")
            dx = dx.detach().contiguous()
        dh0, dc0, dpred, dseq, dh_T, dc_T = self._tangent_outputs(dh0, dc0)
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_forward_tangent(self._h, _ptr(dx),
                                                     _lib.X_BF16 if dx is not None and dx.dtype == torch.bfloat16 else _lib.X_FP32,
                                                     self._ptr_table(dh0), self._ptr_table(dc0), _ptr(dpred), _ptr(dseq),
                                                     self._ptr_table(dh_T), self._ptr_table(dc_T), self._stream()),
                       "nint_forward_tangent")
        return dpred, dseq, list(zip(dh_T, dc_T))

    def forward_tangent_bank(self, dframes: torch.Tensor, dh0=None, dc0=None):
        """forward_tangent after `forward_bank`: dframes [N,H,W,c_pad] are the tangent frames in the bank's layout with
        the constant-1 lane 0 (FrameBank.tangent / tangent_from_fields), N the bank's; the windows are those of the
        forward.  The plan keeps a reference to dframes until the next forward: backward_second_order_params reads
        them again."""
        if self._keep is None:
            raise RuntimeError("forward_tangent_bank: the last forward did not read a frame bank (forward_bank)")
        frames = self._keep[0]
        if tuple(dframes.shape) != tuple(frames.shape):
            raise ValueError(f"tangent frames have shape {tuple(dframes.shape)}, expected {tuple(frames.shape)}")
        self._check_dev(dframes, "tangent frames", dtypes=(frames.dtype,))
        if not dframes.is_contiguous():
            raise ValueError("tangent frames must be contiguous")
        dh0, dc0, dpred, dseq, dh_T, dc_T = self._tangent_outputs(dh0, dc0)
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_forward_tangent_bank(self._h, _ptr(dframes), dframes.shape[0], self._ptr_table(dh0),
                                                          self._ptr_table(dc0), _ptr(dpred), _ptr(dseq),
                                                          self._ptr_table(dh_T), self._ptr_table(dc_T), self._stream()),
                       "nint_forward_tangent_bank")
        self._tkeep = dframes    # backward_second_order_params' wgrad reads them again through the plan's tensor maps
        return dpred, dseq, list(zip(dh_T, dc_T))

    # ---- second-order adjoint (plans made with training=True, second_order=True)
    def _head_seed(self, u, name):
        """u: dL/dpred [B,1,H,W], or (dpred, dseq) with dseq [B,T,H,W] (return_sequence plans; either may be None) ->
        (dpred, dseq) for the library, dpred folded into dseq[:, T-1] when both are given (pred is the last step)"""
        dpred, dseq = tuple(u) if isinstance(u, (tuple, list)) else (u, None)
        if dseq is not None:
            self._check_dev(dseq, f"{name} (sequence)", (self.B, self.T, self.H, self.W))
            dseq = dseq.detach().contiguous().clone() if dpred is not None else dseq.detach().contiguous()
        if dpred is not None:
            self._check_dev(dpred, name, (self.B, 1, self.H, self.W))
            if dseq is not None:
                dseq[:, -1] += dpred.detach().reshape(self.B, self.H, self.W)
                dpred = None
            else:
                dpred = dpred.detach().contiguous()
        return dpred, dseq

    def _second_order(self, fn, u, du, targets, state):
        dpred, dseq = self._head_seed(u, "u")
        ddpred, ddseq = self._head_seed(du, "du")
        new = lambda l: torch.empty(self._state_shape(l), dtype=torch.float32, device=self.device)
        st = [[new(l) for l in range(self.L)] for _ in range(4)] if state else [None] * 4
        with _lib.on_device(self.device):
            _lib.check(fn(self._h, _ptr(dpred), _ptr(dseq), _ptr(ddpred), _ptr(ddseq), _ptr(targets[0]), _ptr(targets[1]),
                          *[self._ptr_table(t) for t in st], self._stream()), fn.__name__)
        return (list(zip(st[0], st[1])), list(zip(st[2], st[3]))) if state else (None, None)

    def backward_second_order(self, u, du, state: bool = False):
        """Gradient and Hessian-vector product of a loss L of the last `forward`'s outputs w.r.t. its input and initial
        state, at fixed parameters, in the direction of the last `forward_tangent` of that forward (forward-over-reverse).
        u = dL/dout and du = its tangent d2L/dout2 . dout, each dpred [B,1,H,W] or (dpred, dseq [B,T,H,W]) like the
        plan's outputs (None entries are zero).  Returns (dx, ddx, dstate, ddstate): dx = grad_x L and ddx = (H v)_x
        [B,T,C,H,W] fp32; with state=True, dstate / ddstate = [(dh0, dc0) per layer] of the gradient / of H v, else None.
        The saved activations are only read: one forward can serve many (forward_tangent, backward_second_order) pairs,
        e.g. the Hessian-vector products of a Newton-CG or Lanczos loop, and then one `backward`."""
        new = lambda: torch.empty((self.B, self.T, self.C, self.H, self.W), dtype=torch.float32, device=self.device)
        dx, ddx = new(), new()
        dst, ddst = self._second_order(self.lib.nint_backward_second_order, u, du, (dx, ddx), state)
        return dx, ddx, dst, ddst

    def backward_second_order_bank(self, u, du, dframes: torch.Tensor, ddframes: torch.Tensor, state: bool = False):
        """backward_second_order after `forward_bank` / `forward_tangent_bank`: the gradient and H v w.r.t. the frames
        are ADDED into dframes / ddframes [N,C,H,W] fp32 (frame win_start[b] + t gets sample b's step t, in decreasing t
        -- the pass runs backwards in time -- then increasing b).  Returns (dstate, ddstate) as backward_second_order."""
        if self._keep is None:
            raise RuntimeError("backward_second_order_bank: the last forward did not read a frame bank (forward_bank)")
        for t, name in ((dframes, "dframes"), (ddframes, "ddframes")):
            self._check_dev(t, name, (self._keep[0].shape[0], self.C, self.H, self.W))
            if not t.is_contiguous():
                raise ValueError(f"{name} must be contiguous")
        return self._second_order(self.lib.nint_backward_second_order_bank, u, du, (dframes, ddframes), state)

    def backward_second_order_params(self, grad: bool = True):
        """Parameter outputs of the last backward_second_order[_bank] (plans made with second_order=True and
        param_tangent=True): (grads, hvps), each a list in ConvLSTM._params() order -- per layer weight, bias, then the
        head's weight and bias -- with grads = dL/dtheta (None when grad=False: its wgrad launches are skipped) and hvps =
        the theta block of H v for the joint direction (dx, dh0, dc0, dtheta) of the tangent pass the second-order pass
        followed.  One forward serves many directions:

            plan.forward(x)
            for direction in directions:
                plan.set_param_tangent(*model.param_direction(direction))
                dpred, dseq, _ = plan.forward_tangent()
                u, du = ...                                   # loss gradient and its tangent on (dpred, dseq)
                plan.backward_second_order(u, du)
                _, hv = plan.backward_second_order_params(grad=False)
            plan.backward(dpred_seed)                         # one ordinary backward at the end
        """
        new = lambda s: torch.empty(s, dtype=torch.float32, device=self.device)
        shapes, cin = [], self.C
        for hc, k in zip(self.hidden, self.ksize):
            shapes += [(4 * hc, cin + hc, k, k), (4 * hc,)]
            cin = hc
        shapes += [(1, self.hidden[-1], 1, 1), (1,)]
        g = [new(s) for s in shapes] if grad else None
        h = [new(s) for s in shapes]
        table = lambda ts, j: None if ts is None else (ctypes.c_void_p * self.L)(*[ts[2 * l + j].data_ptr()
                                                                                 for l in range(self.L)])
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_backward_second_order_params(
                self._h, table(g, 0), table(g, 1), table(h, 0), table(h, 1), _ptr(g[-2] if g else None),
                _ptr(g[-1] if g else None), _ptr(h[-2]), _ptr(h[-1]), self._stream()), "nint_backward_second_order_params")
        return g, h

    # ---- ConvLSTMCell as a differentiable unit (plans with T = 1, L = 1)
    def cell_forward(self, x, h, c):
        shape = (self.B, self.hidden[0], self.H, self.W)
        self._check_dev(x, "x", (self.B, self.C, self.H, self.W))
        self._check_dev(h, "h", shape)
        self._check_dev(c, "c", shape)
        h_out = torch.empty(shape, dtype=torch.float32, device=self.device)
        c_out = torch.empty(shape, dtype=torch.float32, device=self.device)
        self._keep = None
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_cell_forward(self._h, _ptr(x.detach().contiguous()), _ptr(h.detach().contiguous()),
                                                  _ptr(c.detach().contiguous()), _ptr(h_out), _ptr(c_out), self._stream()),
                       "nint_cell_forward")
        self.generation += 1
        return h_out, c_out

    def cell_backward(self, dh_out, dc_out, need_dx=True, need_state=True, need_params=True):
        """(dx, dh, dc, grad_weight, grad_bias) of the last cell_forward; unneeded outputs are None."""
        shape = (self.B, self.hidden[0], self.H, self.W)
        hc, k = self.hidden[0], self.ksize[0]
        for t, n in ((dh_out, "dh_out"), (dc_out, "dc_out")):
            if t is not None:
                self._check_dev(t, n, shape)
        new = lambda s: torch.empty(s, dtype=torch.float32, device=self.device)
        dx = new((self.B, self.C, self.H, self.W)) if need_dx else None
        dh = new(shape) if need_state else None
        dc = new(shape) if need_state else None
        gw = new((4 * hc, self.C + hc, k, k)) if need_params else None
        gb = new((4 * hc,)) if need_params else None
        self.generation += 1
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_cell_backward(self._h, _ptr(None if dh_out is None else dh_out.detach().contiguous()),
                                                   _ptr(None if dc_out is None else dc_out.detach().contiguous()),
                                                   _ptr(dx), _ptr(dh), _ptr(dc), _ptr(gw), _ptr(gb), self._stream()),
                       "nint_cell_backward")
        return dx, dh, dc, gw, gb

    # ---- measurement
    KERNEL_CLASSES = ("gate_conv_fwd", "dgrad_gate_bwd", "wgrad", "other")

    def profile(self, enable: bool):
        _lib.check(self.lib.nint_plan_profile(self._h, int(enable)), "nint_plan_profile")

    def profile_read(self):
        """{class: (device ms, launches)} since the last read (waits for the recorded events)."""
        ms = (ctypes.c_double * 4)()
        n = (ctypes.c_longlong * 4)()
        _lib.check(self.lib.nint_plan_profile_read(self._h, ms, n), "nint_plan_profile_read")
        return {k: (ms[i], n[i]) for i, k in enumerate(self.KERNEL_CLASSES)}

    def debug_raw_gates(self, x: torch.Tensor) -> torch.Tensor:
        """Gate pre-activations (no bias) of layer 0 at t=0, returned as [B,4*Hc,H,W] in the
        reference's channel order (test hook for the implicit-GEMM machinery)."""
        self._check_dev(x, "x", (self.B, self.T, self.C, self.H, self.W))
        hc = self.hidden[0]
        if hc % 16 or (hc > 64 and hc % 64):
            raise ValueError("debug_raw_gates: hidden size must not need padding")
        out = torch.empty((self.B, self.H, self.W, 4 * hc), dtype=torch.float32, device=self.device)
        with _lib.on_device(self.device):
            _lib.check(self.lib.nint_debug_raw_gates(self._h, _ptr(x.contiguous()), _ptr(out), self._stream()),
                       "nint_debug_raw_gates")
        perm = torch.tensor([self.lib.nint_gate_column(q, hc) for q in range(4 * hc)], device=self.device)
        nat = torch.empty_like(out)
        nat[..., perm] = out
        nat = nat.permute(0, 3, 1, 2).contiguous()
        # the packed forward weights of the sigmoid gates (i, f, o) carry a factor 0.5 (the epilogue's sigmoid expects
        # halved pre-activations: exact, a power of two); undo it for the comparison with a plain convolution
        for gate in (0, 1, 3):
            nat[:, gate * hc:(gate + 1) * hc] *= 2.0
        return nat
