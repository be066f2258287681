"""Cost and accuracy of the tangent-linear model (ConvLSTM.jvp / Plan.forward_tangent).  Two geometries, bf16:
BASELINE cfg 2 (B=32, T=12, 21 channels, 90x144, 21 -> 64, 3x3) and the shipped model (B=8, T=48, 5 channels, 100x154,
[64, 32, 16], [5, 3, 3]).

  1. ms per forward alone and per forward + one tangent pass (same training plan), CUDA events around --steps calls,
     alternated --rounds times in the same process.
  2. device time per launch of the tangent gate GEMM (the conv kernel with its raw dump) and of tangent_cell_kernel,
     from torch.profiler over one tangent pass in a run of its own, next to the forward's conv kernel; achieved bytes/s
     of tangent_cell_kernel on its algorithmic bytes against the measured device-to-device copy bandwidth.
  3. wall time of utils.tangent_sweep against utils.sensitivity_sweep (every feature, --batches batches).
  4. (cfg 2 only) how far sensitivity_sweep's bf16 finite differences (+5 %) and the bf16 tangent sit from the fp32
     oracle's JVP (torch.func.jvp on the CPU) of the same windows, for --features features, max|a-b|/max|b| and
     relative L2 over the cropped field; and the fp32 oracle's own +5 % finite difference against its JVP (the
     nonlinearity a finite difference carries at that size).
Prints one JSON line with the card name and power limit; --out also writes it to a file.

    python tools/tangent_time.py --steps 20 --rounds 3 --out tangent_time.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from nasa_niswan_b200 import ConvLSTM, utils  # noqa: E402

# name: (B, T, C, H, W, hidden, ks)
GEOMS = {"cfg2": (32, 12, 21, 90, 144, [64], [3]),
         "shipped": (8, 48, 5, 100, 154, [64, 32, 16], [5, 3, 3])}
CROP = (5, 95, 5, 139)


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


def time_ms(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def kernel_us(fn, names):
    """mean device time per launch (us) and launch count of the kernels whose names contain each of `names`"""
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


def cell_bytes(B, H, W, hidden, esize):
    """algorithmic bytes of the tangent cell kernels of one step: raw dump (fp32) and gates read, c_{t-1}, c_t read,
    dc read and written, dh written -- per layer"""
    return sum(B * H * W * (4 * hc * 4 + 4 * hc * esize + 4 * hc * 4 + hc * esize) for hc in hidden)


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def accuracy(net, features, perturbation=0.05):
    """bf16 finite differences and bf16 tangent against the fp32 oracle's JVP, on two cfg 2 windows"""
    from oracle import convlstm_oracle as O
    from oracle.state_oracle import convlstm_forward_state
    B, T, C, H, W, hidden, ks = GEOMS["cfg2"]
    g = torch.Generator().manual_seed(1)
    X = torch.randn(2, T, C, H, W, generator=g)
    params = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    loader = [(X, None)]
    fd = utils.sensitivity_sweep(loader, net, C, perturbation, crop=CROP) - \
        utils.sensitivity_sweep(loader, net, C, 0.0, crop=CROP)
    lin = utils.tangent_sweep(loader, net, C, perturbation, crop=CROP)
    c = lambda p: p[:, 0, CROP[0]:CROP[1], CROP[2]:CROP[3]]
    f = lambda x: c(convlstm_forward_state(x, params, len(hidden))[0])
    out = {}
    for i in features:
        v = torch.zeros_like(X)
        v[:, :, i] = X[:, :, i] * perturbation
        with torch.no_grad():
            base, ref = torch.func.jvp(f, (X,), (v,))
            ofd = f(X + v) - base
        err = lambda a: {"max_abs_norm": float(O.max_abs_normalised(a, ref)), "rel_l2": float(O.rel_l2(a, ref))}
        out[f"feature_{i}"] = {"bf16_finite_difference": err(fd[i]), "bf16_tangent": err(lin[i]),
                               "fp32_oracle_finite_difference": err(ofd), "jvp_max_abs": float(ref.abs().max())}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batches", type=int, default=2)
    ap.add_argument("--features", default="0,10,20")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: these are GPU times")
    res = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    bw = copy_bandwidth()
    res["copy_bandwidth_TBps"] = round(bw / 1e12, 3)
    for name, (B, T, C, H, W, hidden, ks) in GEOMS.items():
        torch.manual_seed(0)
        net = ConvLSTM(C, hidden, ks, len(hidden), precision="bf16").cuda()
        g = torch.Generator(device="cuda").manual_seed(0)
        x = torch.randn(B, T, C, H, W, device="cuda", generator=g)
        dx = torch.randn(B, T, C, H, W, device="cuda", generator=g)
        plan = net.plan_for(x, True, tangent=True)
        fwd = lambda: plan.forward(x)
        both = lambda: (plan.forward(x), plan.forward_tangent(dx))
        plain, tang = [], []
        for r in range(a.rounds):
            for fn, acc in ((fwd, plain), (both, tang)):
                if r == 0:
                    for _ in range(a.warmup):
                        fn()
                acc.append(time_ms(fn, a.steps))
        fk = kernel_us(fwd, ["conv_halo_kernel"])["conv_halo_kernel"]
        plan.forward(x)
        tk = kernel_us(lambda: plan.forward_tangent(dx), ["conv_halo_kernel", "tangent_cell_kernel"])
        steps = T * len(hidden)
        cb = cell_bytes(B, H, W, hidden, 2) / len(hidden)     # mean bytes per cell-kernel launch
        loader = [(torch.randn(B, T, C, H, W, generator=torch.Generator().manual_seed(b)), None)
                  for b in range(a.batches)]
        sweep_s = wall(lambda: utils.sensitivity_sweep(loader, net, C, crop=CROP))
        tsweep_s = wall(lambda: utils.tangent_sweep(loader, net, C, crop=CROP))
        res[name] = {
            "forward_ms": [round(v, 3) for v in plain], "forward_plus_tangent_ms": [round(v, 3) for v in tang],
            "forward_conv_us_per_launch": round(fk[0], 2), "forward_conv_launches": fk[1],
            "tangent_gemm_us_per_launch": round(tk["conv_halo_kernel"][0], 2),
            "tangent_gemm_launches": tk["conv_halo_kernel"][1],
            "tangent_cell_us_per_launch": round(tk["tangent_cell_kernel"][0], 2),
            "tangent_cell_launches": tk["tangent_cell_kernel"][1], "tangent_cell_MB_per_launch": round(cb / 1e6, 1),
            "tangent_cell_TBps": round(cb / (tk["tangent_cell_kernel"][0] * 1e-6) / 1e12, 3),
            "cell_steps": steps,
            "sweep_features": C, "sweep_batches": a.batches,
            "sensitivity_sweep_s": round(sweep_s, 3), "tangent_sweep_s": round(tsweep_s, 3),
        }
        if name == "cfg2":
            res[name]["accuracy_vs_fp32_oracle_jvp"] = accuracy(net, [int(i) for i in a.features.split(",")])
        del net, plan
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
