"""Cost of frame-bank input gradients.  Two geometries, both read through a FrameBank built by from_fields:
BASELINE cfg 2 (B=32, T=12, 20 levels + emission = 21 channels, 80x134 -> 90x144, 21 -> 64, 3x3, bf16) and the shipped
model (B=8, T=48, 4 levels + emission, 90x144 -> 100x154, [64, 32, 16], [5, 3, 3], bf16).

  1. ms per training step (forward_windows + backward) without and with bank.grad, CUDA events around --steps steps,
     the two alternated --rounds times in the same process.
  2. device time per launch of the accumulation kernel (accum_frames_kernel, one per step t of a backward) and of the
     preprocessing adjoint (fuse_adjoint_kernel) over a record of --frames frames, from torch.profiler in a run of its
     own, with achieved bytes/s on the kernels' algorithmic bytes against the measured device-to-device copy bandwidth.
Prints one JSON line with the card name and power limit; --out also writes it to a file.

    python tools/bank_grad_time.py --steps 20 --rounds 3 --out bank_grad_time.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from nasa_niswan_b200 import ConvLSTM  # noqa: E402
from nasa_niswan_b200.preprocess import FrameBank  # noqa: E402

# name: (B, T, levels, H, W, Hp, Wp, hidden, ks)
GEOMS = {"cfg2": (32, 12, 20, 80, 134, 90, 144, [64], [3]),
         "shipped": (8, 48, 4, 90, 144, 100, 154, [64, 32, 16], [5, 3, 3])}


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def copy_bandwidth(nbytes=2 << 30, reps=20):
    """device-to-device copy: read + write bytes per second"""
    src = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda").fill_(1.0)
    dst = torch.empty_like(src)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    e1.synchronize()
    return 2 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3)


def setup(name, n_frames):
    B, T, L, H, W, Hp, Wp, hidden, ks = GEOMS[name]
    g = torch.Generator(device="cuda").manual_seed(0)
    lev = torch.randn(n_frames, L, H, W, device="cuda", generator=g)
    emis = torch.randn(n_frames, H, W, device="cuda", generator=g).abs()
    mean, std = torch.zeros(L + 1, device="cuda"), torch.ones(L + 1, device="cuda")
    bank = FrameBank.from_fields(lev, emis, mean, std, (Hp, Wp), "reference_rnn", precision="bf16")
    torch.manual_seed(0)
    net = ConvLSTM(L + 1, hidden, ks, len(hidden), precision="bf16").cuda()
    starts = torch.randperm(n_frames - T + 1, device="cuda")[:B].to(torch.int32)   # distinct starts
    dpred = torch.randn(B, 1, Hp, Wp, device="cuda", generator=g)
    return bank, net, starts, T, dpred


def step(bank, net, starts, T, dpred):
    net.forward_windows(bank, starts, T).backward(dpred)


def time_steps(bank, net, starts, T, dpred, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step(bank, net, starts, T, dpred)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def kernel_us(fn, names):
    """mean device time per launch (us) of the kernels whose names contain each of `names`"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for n in names:
        tot, cnt = 0.0, 0
        for e in prof.key_averages():
            if n in e.key:
                tot += getattr(e, "device_time_total", None) or e.cuda_time_total
                cnt += e.count
        out[n] = (tot / cnt if cnt else float("nan"), cnt)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frames", type=int, default=384)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: these are GPU times")
    res = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    bw = copy_bandwidth()
    res["copy_bandwidth_TBps"] = round(bw / 1e12, 3)
    for name in GEOMS:
        B, T, L, H, W, Hp, Wp, hidden, ks = GEOMS[name]
        C = L + 1
        bank, net, starts, T, dpred = setup(name, a.frames)
        plain, grad = [], []
        for r in range(a.rounds):
            for with_grad in (False, True):
                bank.requires_grad_(with_grad)
                if r == 0:
                    for _ in range(a.warmup):
                        step(bank, net, starts, T, dpred)
                ms = time_steps(bank, net, starts, T, dpred, a.steps)
                (grad if with_grad else plain).append(ms)
        bank.requires_grad_()
        k = kernel_us(lambda: step(bank, net, starts, T, dpred), ["accum_frames_kernel"])["accum_frames_kernel"]
        ncols = (C + 31) // 32 * 32                            # width of the dgrad dump (the padded input channels)
        acc_bytes = B * Hp * Wp * (ncols + 2 * C) * 4             # raw dump read, frames read and written
        adj = kernel_us(lambda: bank.field_grads(), ["fuse_adjoint_kernel"])["fuse_adjoint_kernel"]
        adj_bytes = a.frames * C * (Hp * Wp + H * W) * 4
        res[name] = {
            "step_ms_without_bank_grad": [round(v, 3) for v in plain],
            "step_ms_with_bank_grad": [round(v, 3) for v in grad],
            "accum_us_per_launch": round(k[0], 2), "accum_launches_per_step": k[1],
            "accum_MB_per_launch": round(acc_bytes / 1e6, 1),
            "accum_TBps": round(acc_bytes / (k[0] * 1e-6) / 1e12, 3),
            "adjoint_frames": a.frames, "adjoint_us": round(adj[0], 1), "adjoint_MB": round(adj_bytes / 1e6, 1),
            "adjoint_TBps": round(adj_bytes / (adj[0] * 1e-6) / 1e12, 3),
        }
        del bank, net
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
