"""CPU: the second-order adjoint without a GPU -- the fp64 restatement of the recursion (oracle/hvp_oracle.py) against
torch.func's forward-over-reverse Hessian-vector product of the reference loop, its symmetry and its agreement with
central differences of the gradient; the C ABI's new flag and entry points; and the workspace: plans without the flag
keep their sizes, plans with it reserve the per-step tangent history and the pass's buffers."""
import ctypes

import pytest
import torch

from nasa_niswan_b200 import _lib
from oracle import convlstm_oracle as O
from oracle.hvp_oracle import hvp_restatement
from oracle.state_oracle import convlstm_forward_state


def _loss(return_sequence, crop=(1, 8, 2, 10), seed=7, shape=(2, 9, 11), T=4):
    """MSE + L1 on a crop (the training loss: curvature from the MSE), on pred and, with return_sequence, on seq"""
    g = torch.Generator().manual_seed(seed)
    B, H, W = shape
    y = torch.randn(B, 1, H, W, generator=g, dtype=torch.float64)
    ys = torch.randn(B, T, H, W, generator=g, dtype=torch.float64)
    y0, y1, x0, x1 = crop

    def term(p, t):
        d = (p - t)[..., y0:y1, x0:x1]
        return (d * d).mean() + d.abs().mean()

    if return_sequence:
        return lambda out: term(out[0], y) + 0.5 * term(out[1], ys)
    return lambda out: term(out, y)


def _setup(seed=0, B=2, T=4, C=3, H=9, W=11, hidden=(12, 5), ks=(3, 5), with_state=True, with_dstate=True):
    params = {k: v.double() for k, v in O.init_params(C, list(hidden), list(ks), seed=seed).items()}
    g = torch.Generator().manual_seed(seed + 1)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    x = r(B, T, C, H, W)
    state = [(r(B, hc, H, W) * 0.5, r(B, hc, H, W) * 0.5) for hc in hidden] if with_state else None
    dx = r(B, T, C, H, W)
    dstate = [(r(B, hc, H, W), r(B, hc, H, W)) for hc in hidden] if with_dstate else None
    return params, len(hidden), x, state, dx, dstate


def _zeros_like_state(x, params, L):
    B, _, _, H, W = x.shape
    return [(torch.zeros(B, params[f"layers.{l}.conv.bias"].shape[0] // 4, H, W, dtype=x.dtype),) * 2 for l in range(L)]


def _func_hvp(params, L, loss_fn, x, state, dx, dstate, return_sequence):
    """torch.func.jvp(torch.func.grad(L o f)) of the reference loop: (grad, hvp) over (x, h0s, c0s)"""
    zero = _zeros_like_state(x, params, L)
    state = state or zero
    dstate = dstate or zero

    def lf(x, hs, cs):
        out, _ = convlstm_forward_state(x, params, L, list(zip(hs, cs)), return_sequence=return_sequence)
        return loss_fn(out)
    primals = (x, tuple(h for h, _ in state), tuple(c for _, c in state))
    tangents = (dx, tuple(h for h, _ in dstate), tuple(c for _, c in dstate))
    return torch.func.jvp(torch.func.grad(lf, argnums=(0, 1, 2)), primals, tangents)


def _flat(res):
    x, pairs = res
    return [x] + ([t for p in pairs for t in p] if pairs is not None else [])


def _ref_flat(res):
    x, hs, cs = res
    return [x] + [t for h, c in zip(hs, cs) for t in (h, c)]


CASES = {
    "input_only": dict(with_state=False, with_dstate=False),
    "state_no_state_direction": dict(with_state=True, with_dstate=False),
    "state_and_state_direction": dict(with_state=True, with_dstate=True),
    "zero_state_with_state_direction": dict(with_state=False, with_dstate=True),
}


@pytest.mark.parametrize("return_sequence", [False, True], ids=["pred", "return_sequence"])
@pytest.mark.parametrize("case", list(CASES))
def test_restatement_equals_torch_func_hvp(case, return_sequence):
    """two layers, k 3 / 5, hidden 12 (not a multiple of 16) and 5"""
    params, L, x, state, dx, dstate = _setup(**CASES[case])
    loss_fn = _loss(return_sequence)
    loss, grad, hv = hvp_restatement(x, params, L, loss_fn, state, dx, dstate, return_sequence)
    g_ref, h_ref = _func_hvp(params, L, loss_fn, x, state, dx, dstate, return_sequence)
    out, _ = convlstm_forward_state(x, params, L, state, return_sequence=return_sequence)
    assert abs(float(loss) - float(loss_fn(out))) <= 1e-12 * abs(float(loss))
    # without a given state the restatement reports the (well-defined) gradient w.r.t. the zero state too
    for a, b in zip(_flat(grad), _ref_flat(g_ref)):
        assert O.max_abs_normalised(a, b) <= 1e-10
    for a, b in zip(_flat(hv), _ref_flat(h_ref)):
        assert O.max_abs_normalised(a, b) <= 1e-10


def _dot(a, b):
    return sum(float((p * q).sum()) for p, q in zip(a, b))


def test_restatement_hessian_is_symmetric():
    params, L, x, state, v, dv = _setup(seed=4)
    g = torch.Generator().manual_seed(40)
    w = torch.randn(x.shape, generator=g, dtype=torch.float64)
    dw = [(torch.randn(h.shape, generator=g, dtype=torch.float64), torch.randn(c.shape, generator=g, dtype=torch.float64))
          for h, c in state]
    loss_fn = _loss(True)
    hv = _flat(hvp_restatement(x, params, L, loss_fn, state, v, dv, True)[2])
    hw = _flat(hvp_restatement(x, params, L, loss_fn, state, w, dw, True)[2])
    vv = [v] + [t for p in dv for t in p]
    ww = [w] + [t for p in dw for t in p]
    lhs, rhs = _dot(ww, hv), _dot(hw, vv)
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), abs(rhs))


def test_restatement_matches_central_differences_of_the_gradient():
    """a smooth loss (MSE alone: L1's kink would spoil the difference quotient)"""
    params, L, x, state, dx, dstate = _setup(seed=5)
    y = torch.randn(2, 1, 9, 11, generator=torch.Generator().manual_seed(50), dtype=torch.float64)
    loss_fn = lambda out: ((out - y) ** 2).mean() + (out ** 3).mean()
    hv = _flat(hvp_restatement(x, params, L, loss_fn, state, dx, dstate)[2])
    eps = 1e-5

    def grad_at(s):
        st = [(h + s * dh, c + s * dc) for (h, c), (dh, dc) in zip(state, dstate)]
        return _flat(hvp_restatement(x + s * dx, params, L, loss_fn, st, dx, dstate)[1])
    for h, p, m in zip(hv, grad_at(eps), grad_at(-eps)):
        assert O.max_abs_normalised(h, (p - m) / (2 * eps)) < 1e-7


def test_abi_exports_the_second_order_entry_points():
    lib = _lib.load()
    for name in ("nint_backward_second_order", "nint_backward_second_order_bank"):
        assert hasattr(lib, name) and name in _lib.EXPORTS
    assert _lib.FLAG_SECOND_ORDER == 16


def _ws(B, T, H, W, C, hidden, ks, dtype, training, return_sequence, flags):
    lib = _lib.load()
    cfg = _lib.NintConfig()
    cfg.batch, cfg.seq_len, cfg.height, cfg.width, cfg.in_channels = B, T, H, W, C
    cfg.num_layers = len(hidden)
    for i, (hc, k) in enumerate(zip(hidden, ks)):
        cfg.hidden[i], cfg.ksize[i] = hc, k
    cfg.dtype, cfg.training, cfg.return_sequence, cfg.flags = dtype, training, return_sequence, flags
    h = ctypes.c_void_p()
    assert lib.nint_plan_create(ctypes.byref(cfg), ctypes.byref(h)) == 0, lib.nint_last_error()
    n = lib.nint_plan_workspace_bytes(h)
    lib.nint_plan_destroy(h)
    return n


# workspace bytes of plans without the second-order flag, as the library computed them before the flag existed (the
# configurations of the tangent flag's CPU tests, with and without that flag)
PINNED = [
    ((32, 12, 90, 144, 21, [64], [3], 0, 1, 0, 0), 5044623360),               # BASELINE cfg 2, bf16 training
    ((32, 12, 90, 144, 21, [64], [3], 0, 1, 0, 6), 5363275776),               # + input and state gradients
    ((2, 6, 100, 154, 5, [64, 32, 16], [5, 3, 3], 1, 1, 1, 7), 778169344),    # shipped model, tf32, every flag
    ((2, 4, 20, 24, 5, [20, 48, 64], [5, 3, 3], 0, 1, 1, 0), 14523392),       # padded hidden sizes, return_sequence
    ((4, 5, 90, 144, 21, [64], [3], 1, 0, 0, 0), 73879552),                   # tf32 inference
]


@pytest.mark.parametrize("cfg,nbytes", PINNED)
def test_flagless_workspace_sizes_are_unchanged(cfg, nbytes):
    assert _ws(*cfg) == nbytes


def test_tangent_only_workspace_is_unchanged_by_the_new_flag():
    """the tangent flag alone reserves exactly what it reserved before (its CPU test's accounting)"""
    B, T, H, W, C, hidden = 4, 5, 90, 144, 21, [64, 20]
    npix = B * H * W
    for dtype, esize in ((0, 2), (1, 4)):
        base = _ws(B, T, H, W, C, hidden, [3, 3], dtype, 1, 0, 0)
        extra = _ws(B, T, H, W, C, hidden, [3, 3], dtype, 1, 0, _lib.FLAG_TANGENT) - base
        need = T * npix * 32 * esize + 2 * npix * (64 + 32) * esize + npix * (64 + 32) * 4 + npix * 4 * 64 * 4
        assert need <= extra < need + 64 * 1024


def test_the_flag_reserves_the_second_order_buffers():
    B, T, H, W, C, hidden, ks = 4, 5, 90, 144, 21, [64, 20], [3, 3]
    npix = B * H * W
    hcs = [64, 32]                    # hidden 20 runs as 32 channels
    for dtype, esize in ((0, 2), (1, 4)):
        tangent = _ws(B, T, H, W, C, hidden, ks, dtype, 1, 0, _lib.FLAG_TANGENT)
        extra = _ws(B, T, H, W, C, hidden, ks, dtype, 1, 0, _lib.FLAG_SECOND_ORDER) - tangent
        ce = 64 // esize
        need = (sum(T * npix * 4 * hc * 4 for hc in hcs)            # tangent gate GEMM dump of every step
                + sum(T * npix * hc * 4 for hc in hcs)              # dc of every step (T + 1 slots for 1)
                - npix * 4 * 64 * 4                                 # ... in place of the single dump
                + sum(2 * npix * 4 * hc * esize for hc in hcs)      # dgates and their tangents
                + sum(2 * npix * hc * 4 for hc in hcs)              # running dc and its tangent
                + 2 * npix * 64 * 4                                 # dgrad dump (max(cin_rows 32, hc 64) columns)
                + 9 * (4 * 64 // ce) * 32 * 64)                     # layer 0's packed dx dgrad weights
        assert need <= extra < need + 64 * 1024
        # inference plans keep no saved gates: the flag reserves nothing there
        assert _ws(B, T, H, W, C, hidden, ks, dtype, 0, 0, _lib.FLAG_SECOND_ORDER) == \
            _ws(B, T, H, W, C, hidden, ks, dtype, 0, 0, 0)
