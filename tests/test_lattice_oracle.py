"""CPU: the integer-lattice cases of test_gpu_exact.py are exact by construction (no GPU, no libnint.so needed).

For every case the GPU file runs: the fp64 reference equals the same reference evaluated in fp32 with the pixels and
time steps of every gradient sum in another order (so the result does not depend on the accumulation order); every
sum stays within 2^20 grid steps (the exactness headroom, oracle/lattice.py); nonzero terms reach every corner, the
last ragged tile row and column, every tap, every channel chunk, every gate row and every image; and planted defects
of the kinds an exact comparison is meant to catch change the result."""
import functools

import pytest
import torch

from oracle import lattice as Lt

CASES = dict(Lt.suite_cases())


@functools.lru_cache(maxsize=None)
def _ref(cid):
    stats = {}
    return Lt.reference(CASES[cid], stats=stats), stats


def _asserted(case, out):
    """the outputs the GPU tests assert: h' of a cell step is exact only in its mode-3 channels"""
    out = dict(out)
    if case["kind"] == "B":
        out["h"] = out["h"][:, case["h_mask"]]
    return out


@pytest.mark.parametrize("cid", list(CASES))
def test_fp32_in_another_order_equals_fp64(cid):
    case = CASES[cid]
    ref = _asserted(case, _ref(cid)[0])
    for order in (1, 2):
        got = _asserted(case, Lt.reference(case, torch.float32, order=order))
        for k in ref:
            assert torch.equal(got[k].double(), ref[k]), (k, order)


@pytest.mark.parametrize("cid", list(CASES))
def test_headroom(cid):
    hr = _ref(cid)[1]["headroom"]
    worst = max(hr, key=hr.get)
    assert hr[worst] <= 2.0 ** Lt.HEADROOM_BITS, (worst, hr[worst])


@pytest.mark.parametrize("cid", list(CASES))
def test_coverage(cid):
    cov = Lt.summarize_coverage(CASES[cid], _ref(cid)[1]["cov"])
    assert all(cov.values()), [k for k, v in cov.items() if not v]


def _first_images(case, n):
    """a whole-model case cut to its first n images (same grid, tiles, halos and weights)"""
    out = dict(case, B=n, x=case["x"][:n], dpred=case["dpred"][:n])
    if case["dseq"] is not None:
        out["dseq"] = case["dseq"][:n]
    return out


@pytest.mark.parametrize("cid", list(CASES))
def test_planted_defects_change_the_exact_result(cid):
    case = CASES[cid]
    if cid.endswith("cfg2_b32"):
        # at B=32 one evaluation of the reference takes about 10 s: the defects are planted into its first 4 images
        case = _first_images(case, 4)
        ref = _asserted(case, Lt.reference(case))
    else:
        ref = _asserted(case, _ref(cid)[0])
    for d in Lt.defects_for(case):
        bad = _asserted(case, Lt.reference(case, defect=d))
        assert any(not torch.equal(bad[k], ref[k]) for k in ref), f"{d} leaves every asserted output unchanged"


def test_every_defect_is_planted_somewhere():
    planted = {d for case in CASES.values() for d in Lt.defects_for(case)}
    assert planted == set(Lt.DEFECTS)


@pytest.mark.parametrize("cid", [c for c in CASES if not c.endswith("cfg2_b32")])
def test_construction_sits_on_the_exact_points(cid):
    """what the constructions promise: A is dense; B's pre-activations are the bias and its live channels get no dx;
    C stays in the zero state (pred = head bias) and only the g rows of dgates carry gradient"""
    case = CASES[cid]
    out = _ref(cid)[0]
    if case["kind"] == "A":
        assert bool((out["gates"] != 0).float().mean() > 0.5)
    elif case["kind"] == "B":
        C = case["C"]
        assert bool((out["dx"][:, Lt.live_channels(C)] == 0).all()) and bool((out["dx"] != 0).any())
        hm = case["h_mask"]
        assert bool((out["h"][:, hm].abs() == 0.5).all())           # o = 1/2, tanh(+-24) = +-1
        mode2 = (torch.arange(case["hidden"][0]) % 3 + 1) == 2
        assert torch.equal(out["c"][:, mode2], case["c0"][:, mode2] / 2 + 0.5)
        assert bool((out["gw"] != 0).any()) and bool((out["dh"] != 0).any())
    else:
        assert bool((out["pred"] == case["hb"]).all())
        L, hid = len(case["hidden"]), case["hidden"]
        for l in range(L):
            gb = out[f"gb{l}"].view(4, hid[l])
            assert bool((gb[[0, 1, 3]] == 0).all()) and bool((gb[2] != 0).any())
        assert bool((out["gw0"] != 0).any()) and bool((out["dx"] != 0).any())
        assert bool((out["dx"][:, :, Lt.live_channels(case["C"])] == 0).all())
