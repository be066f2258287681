"""CPU: the C-ABI library loads and exports what include/nint.h declares; host-side geometry
logic (tile choice, gate column order, plan validation, workspace accounting); the nn.Module
surface matches the reference's state_dict contract.  No compute calls (no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from nasa_niswan_b200 import ConvLSTM, ConvLSTMCell, _lib
from oracle.golden import load_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "nint.h")).read()
    declared = set(re.findall(r"\b(nint_[a-z_0-9]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in nint.h but not exported by libnint.so"
    assert declared == set(_lib.EXPORTS)
    assert lib.nint_version() >= 100


def test_pick_tile():
    # every grid is covered by 8 x 16 pixel tiles (UMMA M = 128); ragged edges are TMA out-of-bounds work
    for H, W in [(90, 144), (100, 154), (180, 288), (11, 13), (20, 24), (1, 1), (3, 500)]:
        assert _lib.pick_tile(H, W) == (8, 16)


@pytest.mark.parametrize("hc", [16, 32, 64, 128, 256])
def test_gate_column_is_a_permutation(hc):
    lib = _lib.load()
    cols = [lib.nint_gate_column(q, hc) for q in range(4 * hc)]
    assert sorted(cols) == list(range(4 * hc))
    # q-order: inside every 64-column span the four gates (model.py:221 order i,f,g,o) of a 16-channel group
    # sit 16 columns apart
    for q0 in range(0, 4 * hc, 64):
        for c16 in range(16):
            n = [cols[q0 + g * 16 + c16] for g in range(4)]
            assert [v // hc for v in n] == [0, 1, 2, 3] and len({v % hc for v in n}) == 1
        chans = sorted(cols[q0 + c16] % hc for c16 in range(16))
        assert chans == list(range(chans[0], chans[0] + 16)) and chans[0] % 16 == 0


def _cfg(**kw):
    cfg = _lib.NintConfig()
    d = dict(batch=2, seq_len=3, height=20, width=24, in_channels=21, num_layers=1, dtype=0, training=1,
             return_sequence=0)
    d.update(kw)
    hidden, ksize = d.pop("hidden", [32]), d.pop("ksize", [3])
    for k, v in d.items():
        setattr(cfg, k, v)
    for i, (h, k) in enumerate(zip(hidden, ksize)):
        cfg.hidden[i], cfg.ksize[i] = h, k
    return cfg


def _create(cfg):
    lib = _lib.load()
    h = ctypes.c_void_p()
    rc = lib.nint_plan_create(ctypes.byref(cfg), ctypes.byref(h))
    return rc, h, lib


def test_plan_validation_and_workspace_accounting():
    rc, h, lib = _create(_cfg())
    assert rc == 0
    train_bytes = lib.nint_plan_workspace_bytes(h)
    lib.nint_plan_destroy(h)
    rc, h, lib = _create(_cfg(training=0))
    infer_bytes = lib.nint_plan_workspace_bytes(h)
    lib.nint_plan_destroy(h)
    npix = 2 * 20 * 24
    # training keeps T+1 h/c slots and T gate slots; inference a 2-slot h ring and one c slot
    assert train_bytes > infer_bytes
    assert train_bytes >= 3 * npix * 32 * 2 + 4 * npix * 32 * 2 + 4 * npix * 32 * 4 + 3 * npix * 128 * 2
    assert infer_bytes >= 3 * npix * 32 * 2 + 2 * npix * 32 * 2 + npix * 32 * 4
    for bad in [dict(hidden=[0]), dict(hidden=[257]), dict(ksize=[4]), dict(num_layers=0), dict(batch=0),
                dict(dtype=7), dict(hidden=[512]), dict(ksize=[17])]:
        rc, h, lib = _create(_cfg(**bad))
        assert rc != 0 and lib.nint_last_error(), bad


def test_product_build_refuses_the_kernel_experiment_knobs(monkeypatch):
    # NINT_DEBUG_FLAGS (skip the epilogue's memory work, issue no MMAs, timeline stamps ...) are compiled into the
    # experiment build only (build.py --knobs -> libnint_knobs.so); the product library says so instead of ignoring them.
    # Bit 9 (512: no bias folding) is host-side and stays available
    monkeypatch.setenv("NINT_DEBUG_FLAGS", "2")
    rc, h, lib = _create(_cfg())
    assert rc != 0 and b"experiment build" in lib.nint_last_error()
    monkeypatch.setenv("NINT_DEBUG_FLAGS", "512")
    rc, h, lib = _create(_cfg())
    assert rc == 0
    lib.nint_plan_destroy(h)
    from nasa_niswan_b200 import build
    assert build.LIB_KNOBS.endswith("libnint_knobs.so") and build.LIB != build.LIB_KNOBS


def test_any_hidden_size_is_accepted_by_padding():
    # model.py:207 takes any int (the notebooks use ConvLSTM(5, 10, 3, 2)-style sizes): hidden sizes run padded to the
    # kernels' granularity (16; 64 above 64), so the workspace of hidden 10 equals that of hidden 16, 70 that of 128
    def ws(hidden):
        rc, h, lib = _create(_cfg(hidden=hidden, ksize=[3] * len(hidden), num_layers=len(hidden)))
        assert rc == 0, lib.nint_last_error()
        n = lib.nint_plan_workspace_bytes(h)
        lib.nint_plan_destroy(h)
        return n
    assert ws([10]) == ws([16]) and ws([24]) == ws([32]) and ws([70]) == ws([128]) and ws([96]) == ws([128])
    assert ws([10, 3]) == ws([16, 16])
    assert ws([16]) < ws([32]) < ws([64]) < ws([128])


def test_deterministic_and_input_grad_plans_reserve_their_buffers():
    base = _cfg(hidden=[64], batch=4, seq_len=5, height=90, width=144)
    det = _cfg(hidden=[64], batch=4, seq_len=5, height=90, width=144, flags=_lib.FLAG_DETERMINISTIC)
    dx = _cfg(hidden=[64], batch=4, seq_len=5, height=90, width=144, flags=_lib.FLAG_INPUT_GRAD)
    sizes = []
    for cfg in (base, det, dx):
        rc, h, lib = _create(cfg)
        assert rc == 0, lib.nint_last_error()
        sizes.append(lib.nint_plan_workspace_bytes(h))
        c_pad, ones, eb = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        assert lib.nint_plan_input_layout(h, ctypes.byref(c_pad), ctypes.byref(ones), ctypes.byref(eb)) == 0
        assert (c_pad.value, ones.value, eb.value) == (32, 21, 2)      # 21 channels -> 32 lanes, lane 21 carries 1.0
        lib.nint_plan_destroy(h)
    slice_bytes = 9 * 256 * 96 * 4                                     # [taps][4hc][x 32 + h 64 columns] fp32
    assert sizes[1] - sizes[0] >= 30 * slice_bytes                     # one partial-sum slice per split-K share
    assert sizes[2] - sizes[0] >= 4 * 90 * 144 * (64 + 64) * 4         # dgrad dump + upstream dh staging


def test_compute_without_binding_fails_loudly():
    rc, h, lib = _create(_cfg())
    assert rc == 0
    assert lib.nint_forward(h, None, None, None, None) != 0
    assert b"not bound" in lib.nint_last_error()
    lib.nint_plan_destroy(h)


def test_module_surface_matches_reference_contract(golden_dir):
    # param-count known answer test.ipynb:4698-4699 and state_dict names (utils.py:27,39)
    net = ConvLSTM(5, [64, 32, 16], [5, 3, 3], 3)
    assert [p.numel() for p in net.parameters()] == [441600, 256, 110592, 128, 27648, 64, 16, 1]
    z = load_case(golden_dir, "lstm_3layer_k533")
    ref_sd = {k[6:]: z[k] for k in z if k.startswith("param/")}
    net = ConvLSTM(5, [32, 16, 16], [5, 3, 3], 3)
    sd = net.state_dict()
    assert list(sd.keys()) == list(ref_sd.keys())
    assert all(tuple(sd[k].shape) == ref_sd[k].shape for k in sd)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in ref_sd.items()})     # strict load works
    assert net.layers[0].hidden_channels == 32 and net.num_layers == 3
    with pytest.raises(AssertionError):
        ConvLSTM(5, [64, 32], [5, 3, 3], 3)                                       # model.py:237


def test_default_init_matches_reference_rng_stream(golden_dir):
    # same seed -> same parameters as the reference constructor (golden generated with seed 0)
    z = load_case(golden_dir, "lstm_c21_h32_k3")
    torch.manual_seed(0)
    net = ConvLSTM(21, [32], [3], 1)
    for k, v in net.state_dict().items():
        assert np.array_equal(v.numpy(), z["param/" + k]), k


def test_no_cpu_fallback():
    net = ConvLSTM(3, [16], [3], 1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(torch.zeros(1, 2, 3, 8, 8))
    cell = ConvLSTMCell(3, 16, 3)
    with pytest.raises((RuntimeError, NotImplementedError)):
        with torch.no_grad():
            cell(torch.zeros(1, 3, 8, 8), (torch.zeros(1, 16, 8, 8), torch.zeros(1, 16, 8, 8)))


def test_checkpoint_format_matches_reference(tmp_path):
    """utils.py:23-50: same dict keys, same lr override rules (CPU: any nn.Module + torch optimizer)"""
    import torch
    from nasa_niswan_b200.utils import load_checkpoint, save_checkpoint
    net = torch.nn.Conv2d(3, 4, 3)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, betas=(0.5, 0.999))
    net(torch.randn(1, 3, 8, 8)).sum().backward()
    opt.step()
    f = tmp_path / "generator.pth.tar"
    save_checkpoint(net, opt, str(f), learning_rate=5e-4, epoch=10)
    raw = torch.load(str(f), weights_only=False)
    assert set(raw) == {"model_state_dict", "optimizer_state_dict", "learning_rate", "epoch"}
    net2 = torch.nn.Conv2d(3, 4, 3)
    opt2 = torch.optim.Adam(net2.parameters(), lr=1e-3, betas=(0.5, 0.999))
    load_checkpoint(str(f), net2, opt2)
    assert all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), net2.state_dict().values()))
    assert opt2.param_groups[0]["lr"] == 5e-4            # utils.py:47-49: the stored learning rate wins
    load_checkpoint(str(f), net2, opt2, lr=1e-2)
    assert opt2.param_groups[0]["lr"] == 1e-2            # utils.py:43-45: an explicit lr overrides it


def test_torch_library_ops_are_registered_cuda_only():
    """SURVEY 8b: the hot path is reachable as torch.library ops; they have no CPU kernel (no fallback)"""
    import nasa_niswan_b200  # noqa: F401  (registers the ops)
    assert str(torch.ops.nint.convlstm_forward.default._schema) == \
        "nint::convlstm_forward(Tensor x, Tensor[] params, SymInt plan_id) -> (Tensor, Tensor)"
    assert str(torch.ops.nint.convlstm_backward.default._schema) == \
        "nint::convlstm_backward(Tensor dpred, Tensor? dseq, SymInt plan_id, SymInt generation, bool need_dx) -> Tensor[]"
    assert str(torch.ops.nint.convlstm_forward_bank.default._schema) == \
        "nint::convlstm_forward_bank(Tensor frames, Tensor win_start, Tensor[] params, SymInt plan_id) -> (Tensor, Tensor)"
    assert "nint::cell_forward" in str(torch.ops.nint.cell_forward.default._schema)
    assert "nint::cell_backward" in str(torch.ops.nint.cell_backward.default._schema)
    with pytest.raises(NotImplementedError, match="CPU"):
        torch.ops.nint.convlstm_forward(torch.zeros(1, 1, 1, 8, 8), [torch.zeros(1)], 1)


def test_module_survives_deepcopy_and_pickle():
    """ADVICE r1: plans (ctypes handles + workspaces) are derived state; copying / pickling the module must work and
    yield an empty plan cache (copy.deepcopy, torch.save(model), swa_utils.AveragedModel all do this)."""
    import copy
    import io
    net = ConvLSTM(5, [16], [3], 1)
    net._plans._plans["fake"] = ctypes.c_void_p(1)            # what a live plan holds: deepcopy of this raises
    net.layers[0]._plans._all.append(ctypes.c_void_p(2))
    twin = copy.deepcopy(net)
    assert len(twin._plans._plans) == 0 and len(twin.layers[0]._plans._all) == 0
    assert all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), twin.state_dict().values()))
    buf = io.BytesIO()
    torch.save(net, buf)
    buf.seek(0)
    back = torch.load(buf, weights_only=False)
    assert len(back._plans._plans) == 0 and back.layers[0].hidden_channels == 16
    torch.optim.swa_utils.AveragedModel(net)


def test_model_shim_reexports_upstream_names(tmp_path, monkeypatch):
    """SURVEY 8b: a replacement model.py keeps `from model import Generator, UNet, ConvLSTM, initialize_weights`
    (train.py:19) resolving -- ConvLSTM from here, the rest from upstream's renamed file."""
    import importlib.util
    import sys
    (tmp_path / "model_reference.py").write_text(
        "class Generator: pass\nclass UNet: pass\nclass Discriminator: pass\ndef initialize_weights(m): return 'init'\n")
    monkeypatch.syspath_prepend(str(tmp_path))
    sys.modules.pop("model_reference", None)
    spec = importlib.util.spec_from_file_location("model_shim", os.path.join(ROOT, "integration", "model.py"))
    shim = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(shim)
    assert shim.ConvLSTM is ConvLSTM and shim.ConvLSTMCell is ConvLSTMCell
    assert shim.Generator.__name__ == "Generator" and shim.initialize_weights(None) == "init"
    with pytest.raises(ImportError, match="reference"):
        shim.Encoder()                                        # not in the fake upstream: importable, raises when used
    sys.modules.pop("model_reference", None)


def test_val_loop_keeps_the_reference_signature():
    import inspect
    from nasa_niswan_b200.utils import val_loop, seed
    assert list(inspect.signature(val_loop).parameters)[:3] == ["args", "dataloader", "model"]   # utils.py:52
    prev = torch.backends.cudnn.deterministic
    seed(0)                                                   # utils.py:77-88
    assert torch.backends.cudnn.deterministic and not torch.backends.cudnn.benchmark
    from nasa_niswan_b200.model import _deterministic_default
    assert _deterministic_default()
    torch.backends.cudnn.deterministic = prev


def test_frame_bank_layout_rule_matches_the_library():
    """preprocess.input_layout (what FrameBank builds) and nint_plan_input_layout (what the TMA descriptors expect) are
    the same rule: channels padded to 32 lanes, first padding lane = the ones lane, none when C is a multiple of 32"""
    from nasa_niswan_b200.preprocess import input_layout
    for C in (1, 5, 8, 21, 31, 32, 33, 40, 64):
        rc, h, lib = _create(_cfg(in_channels=C, training=0))
        assert rc == 0, lib.nint_last_error()
        c_pad, ones, eb = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        assert lib.nint_plan_input_layout(h, ctypes.byref(c_pad), ctypes.byref(ones), ctypes.byref(eb)) == 0
        lib.nint_plan_destroy(h)
        assert (c_pad.value, ones.value) == input_layout(C), C
    rc, h, lib = _create(_cfg(dtype=1, training=0))
    lib.nint_plan_input_layout(h, None, None, ctypes.byref(eb))
    lib.nint_plan_destroy(h)
    assert eb.value == 4                                            # tf32 plans keep fp32 storage


def test_host_side_helpers_degrade_without_a_gpu():
    from nasa_niswan_b200.parallel import bind_to_gpu_numa_node, shard_batch
    if not torch.cuda.is_available():
        assert bind_to_gpu_numa_node("cuda:0") is None              # topology unreadable: nothing is changed
    assert [shard_batch(256, r, 8) for r in (0, 7)] == [(0, 32), (224, 256)]     # BASELINE cfg 3 at 8 ranks
    assert [shard_batch(256, r, 2)[1] - shard_batch(256, r, 2)[0] for r in (0, 1)] == [128, 128]
