"""CPU: the parameter-space tangent without a GPU -- the fp64 restatement of the tangent pass with a parameter direction
(oracle/param_tangent_oracle.py) against torch.func.jvp of the reference loop with the parameters as an argument, and
against central differences; the C ABI's new flag and entry points; and the workspace: plans without the flag keep their
sizes, plans with it reserve the direction's weight panels and biases."""
import ctypes

import pytest
import torch

from nasa_niswan_b200 import _lib
from oracle import convlstm_oracle as O
from oracle.param_tangent_oracle import jvp_restatement
from oracle.state_oracle import convlstm_forward_state


def _setup(seed=0, B=2, T=4, C=3, H=9, W=11, hidden=(12, 5), ks=(3, 5), with_state=True):
    params = {k: v.double() for k, v in O.init_params(C, list(hidden), list(ks), seed=seed).items()}
    g = torch.Generator().manual_seed(seed + 1)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    x = r(B, T, C, H, W)
    state = [(r(B, hc, H, W) * 0.5, r(B, hc, H, W) * 0.5) for hc in hidden] if with_state else None
    dx = r(B, T, C, H, W)
    dstate = [(r(B, hc, H, W), r(B, hc, H, W)) for hc in hidden] if with_state else None
    dparams = {k: r(*v.shape) * 0.1 for k, v in params.items()}
    return params, len(hidden), x, state, dx, dstate, dparams


def _func_jvp(params, L, x, state, dx, dstate, dparams, return_sequence):
    """torch.func.jvp of the reference loop over (params, x, h0s, c0s)"""
    B, _, _, H, W = x.shape
    zero = [(torch.zeros(B, params[f"layers.{l}.conv.bias"].shape[0] // 4, H, W, dtype=x.dtype),) * 2
            for l in range(L)]
    state, dstate = state or zero, dstate or zero

    def f(p, x, hs, cs):
        return convlstm_forward_state(x, p, L, list(zip(hs, cs)), return_sequence=return_sequence)

    primals = (params, x, tuple(h for h, _ in state), tuple(c for _, c in state))
    tangents = (dparams, dx, tuple(h for h, _ in dstate), tuple(c for _, c in dstate))
    return torch.func.jvp(f, primals, tangents)


def _flat(obj):
    if isinstance(obj, torch.Tensor):
        return [obj]
    return [t for o in obj for t in _flat(o)]


def _close(a, b, tol):
    for u, v in zip(_flat(a), _flat(b), strict=True):
        assert float((u - v).abs().max()) <= tol * max(1.0, float(v.abs().max())), float((u - v).abs().max())


@pytest.mark.parametrize("return_sequence", [False, True])
@pytest.mark.parametrize("with_state", [False, True])
def test_joint_jvp_matches_torch_func(with_state, return_sequence):
    params, L, x, state, dx, dstate, dparams = _setup(with_state=with_state)
    ref_out, ref_dout = _func_jvp(params, L, x, state, dx, dstate, dparams, return_sequence)
    out, dout = jvp_restatement(x, params, L, state, dx, dstate, dparams, return_sequence)
    _close(out, ref_out, 1e-12)
    _close(dout, ref_dout, 1e-10)


def test_parameter_only_direction_and_partial_dicts():
    params, L, x, _, _, _, dparams = _setup(with_state=False)
    part = {"layers.1.conv.weight": dparams["layers.1.conv.weight"], "conv.bias": dparams["conv.bias"]}
    full = {k: (part[k] if k in part else torch.zeros_like(v)) for k, v in params.items()}
    _, ref = _func_jvp(params, L, x, None, torch.zeros_like(x), None, full, False)
    _, got = jvp_restatement(x, params, L, dparams=part)
    _close(got, ref, 1e-10)
    # linear in the direction
    _, got2 = jvp_restatement(x, params, L, dparams={k: 2 * v for k, v in part.items()})
    _close(got2, tuple(_flat(2 * t for t in _flat(got))), 1e-12)


def test_central_differences():
    params, L, x, state, dx, dstate, dparams = _setup(with_state=True)
    eps = 1e-5
    shift = lambda s: {k: params[k] + s * dparams[k] for k in params}
    move = lambda s: [(h + s * dh, c + s * dc) for (h, c), (dh, dc) in zip(state, dstate)]
    fp, _ = convlstm_forward_state(x + eps * dx, shift(eps), L, move(eps))
    fm, _ = convlstm_forward_state(x - eps * dx, shift(-eps), L, move(-eps))
    _, (dout, _) = jvp_restatement(x, params, L, state, dx, dstate, dparams)
    fd = (fp - fm) / (2 * eps)
    assert float((fd - dout).abs().max()) <= 1e-7 * float(dout.abs().max())


def test_abi_exports_the_parameter_tangent_entry_points():
    lib = _lib.load()
    for name in ("nint_plan_set_weight_tangent", "nint_plan_set_head_tangent", "nint_plan_clear_param_tangent"):
        assert hasattr(lib, name) and name in _lib.EXPORTS
    assert _lib.FLAG_PARAM_TANGENT == 32


def _ws(B, T, H, W, C, hidden, ks, dtype, training, flags):
    lib = _lib.load()
    cfg = _lib.NintConfig()
    cfg.batch, cfg.seq_len, cfg.height, cfg.width, cfg.in_channels = B, T, H, W, C
    cfg.num_layers = len(hidden)
    for i, (hc, k) in enumerate(zip(hidden, ks)):
        cfg.hidden[i], cfg.ksize[i] = hc, k
    cfg.dtype, cfg.training, cfg.return_sequence, cfg.flags = dtype, training, 0, flags
    h = ctypes.c_void_p()
    assert lib.nint_plan_create(ctypes.byref(cfg), ctypes.byref(h)) == 0, lib.nint_last_error()
    n = lib.nint_plan_workspace_bytes(h)
    lib.nint_plan_destroy(h)
    return n


def test_the_flag_reserves_the_direction_on_top_of_the_tangent_buffers():
    B, T, H, W, C, hidden, ks = 4, 5, 90, 144, 21, [64, 20], [3, 5]
    for dtype, esize in ((0, 2), (1, 4)):
        tangent = _ws(B, T, H, W, C, hidden, ks, dtype, 1, _lib.FLAG_TANGENT)
        extra = _ws(B, T, H, W, C, hidden, ks, dtype, 1, _lib.FLAG_PARAM_TANGENT) - tangent
        # per layer the packed panels of dW (x part 32 lanes, h part 64 / 32 lanes, 4 * hc rows, k * k taps) and the
        # q-order bias; the head's dw and db
        need = (9 * (32 + 64) * 4 * 64 + 25 * (64 + 32) * 4 * 32) * esize + (4 * 64 + 4 * 32) * 4 + 32 * 4 + 4
        assert need <= extra < need + 16 * 1024
