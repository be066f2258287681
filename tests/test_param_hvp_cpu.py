"""CPU: Hessian-vector products over the parameters jointly with the inputs and the initial state, without a GPU --
the fp64 restatement (oracle/param_hvp_oracle.py) against torch.func.jvp(torch.func.grad(L o f)) of the reference loop
over (theta, x, h0, c0), its symmetry and central differences of the gradient; the ABI's params call; the workspace of
plans with both flags."""
import ctypes

import pytest
import torch

from nasa_niswan_b200 import _lib
from oracle import convlstm_oracle as O
from oracle.param_hvp_oracle import param_hvp_restatement
from oracle.state_oracle import convlstm_forward_state


def _loss(return_sequence, crop=(1, 8, 2, 10), seed=7, shape=(2, 9, 11), T=4):
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


def _func(params, L, loss_fn, x, state, dx, dstate, dparams, return_sequence):
    B, _, _, H, W = x.shape
    zero = [(torch.zeros(B, params[f"layers.{l}.conv.bias"].shape[0] // 4, H, W, dtype=x.dtype),) * 2
            for l in range(L)]
    state, dstate = state or zero, dstate or zero

    def lf(p, x, hs, cs):
        out, _ = convlstm_forward_state(x, p, L, list(zip(hs, cs)), return_sequence=return_sequence)
        return loss_fn(out)
    primals = (params, x, tuple(h for h, _ in state), tuple(c for _, c in state))
    tangents = (dparams, dx, tuple(h for h, _ in dstate), tuple(c for _, c in dstate))
    return torch.func.jvp(torch.func.grad(lf, argnums=(0, 1, 2, 3)), primals, tangents)


def _check(ours, ref, L, with_state, tol):
    gx, gst, gp = ours
    rp, rx, rh, rc = ref
    err = lambda a, b: float((a - b).abs().max()) / max(1.0, float(b.abs().max()))
    assert err(gx, rx) <= tol
    for k, v in rp.items():
        assert err(gp[k], v) <= tol, k
    if with_state:
        for l in range(L):
            assert err(gst[l][0], rh[l]) <= tol and err(gst[l][1], rc[l]) <= tol


@pytest.mark.parametrize("return_sequence", [False, True])
@pytest.mark.parametrize("with_state", [False, True])
def test_joint_hvp_matches_torch_func(with_state, return_sequence):
    params, L, x, state, dx, dstate, dparams = _setup(with_state=with_state)
    loss_fn = _loss(return_sequence)
    g_ref, h_ref = _func(params, L, loss_fn, x, state, dx, dstate, dparams, return_sequence)
    _, g, h = param_hvp_restatement(x, params, L, loss_fn, state, dx, dstate, dparams, return_sequence)
    _check(g, g_ref, L, with_state, 1e-10)
    _check(h, h_ref, L, with_state, 1e-10)


def test_parameter_only_direction():
    params, L, x, _, _, _, dparams = _setup(with_state=False)
    loss_fn = _loss(False)
    _, h_ref = _func(params, L, loss_fn, x, None, torch.zeros_like(x), None, dparams, False)
    _, _, h = param_hvp_restatement(x, params, L, loss_fn, dparams=dparams)
    _check(h, h_ref, L, False, 1e-10)


def _dot(v, w):
    return sum(float((a * b).sum()) for a, b in zip(v, w))


def test_symmetry():
    """<v1, H v2> = <v2, H v1> over the joint space (theta, x, h0, c0)"""
    params, L, x, state, dx1, ds1, dp1 = _setup(seed=0)
    _, _, _, _, dx2, ds2, dp2 = _setup(seed=5)
    loss_fn = _loss(True)
    flat = lambda dx, ds, dp: [dx, *[t for pair in ds for t in pair], *[dp[k] for k in sorted(dp)]]
    hflat = lambda h: [h[0], *[t for pair in h[1] for t in pair], *[h[2][k] for k in sorted(h[2])]]
    _, _, h1 = param_hvp_restatement(x, params, L, loss_fn, state, dx1, ds1, dp1, True)
    _, _, h2 = param_hvp_restatement(x, params, L, loss_fn, state, dx2, ds2, dp2, True)
    a, b = _dot(flat(dx2, ds2, dp2), hflat(h1)), _dot(flat(dx1, ds1, dp1), hflat(h2))
    assert abs(a - b) <= 1e-12 * max(abs(a), abs(b))


def test_central_differences_of_the_parameter_gradient():
    """with a loss smooth at the point (MSE only), H v = (grad(z + e v) - grad(z - e v)) / 2e"""
    params, L, x, state, dx, dstate, dparams = _setup(with_state=True)
    y = torch.randn(2, 1, 9, 11, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    loss_fn = lambda out: ((out - y) ** 2).mean()
    eps = 1e-5

    def grad_at(s):
        p = {k: params[k] + s * dparams[k] for k in params}
        st = [(h + s * a, c + s * b) for (h, c), (a, b) in zip(state, dstate)]
        return param_hvp_restatement(x + s * dx, p, L, loss_fn, st)[1][2]
    gp, gm = grad_at(eps), grad_at(-eps)
    _, _, h = param_hvp_restatement(x, params, L, loss_fn, state, dx, dstate, dparams)
    for k in params:
        fd = (gp[k] - gm[k]) / (2 * eps)
        assert float((fd - h[2][k]).abs().max()) <= 1e-6 * max(1.0, float(h[2][k].abs().max())), k


def test_abi_exports_the_params_call():
    lib = _lib.load()
    assert hasattr(lib, "nint_backward_second_order_params") and "nint_backward_second_order_params" in _lib.EXPORTS


def _ws(flags, B=4, T=5, H=90, W=144, C=21, hidden=(64, 20), ks=(3, 5), dtype=0):
    lib = _lib.load()
    cfg = _lib.NintConfig()
    cfg.batch, cfg.seq_len, cfg.height, cfg.width, cfg.in_channels = B, T, H, W, C
    cfg.num_layers = len(hidden)
    for i, (hc, k) in enumerate(zip(hidden, ks)):
        cfg.hidden[i], cfg.ksize[i] = hc, k
    cfg.dtype, cfg.training, cfg.return_sequence, cfg.flags = dtype, 1, 0, flags
    h = ctypes.c_void_p()
    assert lib.nint_plan_create(ctypes.byref(cfg), ctypes.byref(h)) == 0, lib.nint_last_error()
    n = lib.nint_plan_workspace_bytes(h)
    lib.nint_plan_destroy(h)
    return n


def test_both_flags_reserve_the_histories():
    B, T, H, W = 4, 5, 90, 144
    npix = B * H * W
    for dtype, esize in ((0, 2), (1, 4)):
        so = _ws(_lib.FLAG_SECOND_ORDER, dtype=dtype)
        pt = _ws(_lib.FLAG_PARAM_TANGENT, dtype=dtype) - _ws(_lib.FLAG_TANGENT, dtype=dtype)
        both = _ws(_lib.FLAG_SECOND_ORDER | _lib.FLAG_PARAM_TANGENT, dtype=dtype) - so - pt
        # dh history: T+1 slots instead of 2 (hc_pad 64 / 32); (a, da) history: 2T slots instead of 2 (4hc 256 / 128);
        # dW's dgrad panels: taps * 4hc * (cin_rows + hc)
        need = ((T - 1) * npix * (64 + 32) + (2 * T - 2) * npix * (256 + 128)) * esize \
            + (9 * 256 * (32 + 64) + 25 * 128 * (64 + 32)) * esize
        assert need <= both < need + 64 * 1024
