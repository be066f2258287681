"""Headline benchmark: ConvLSTM training samples/s on the BASELINE geometry (90x144 grid, 20 levels
+ BCB emission = 21 channels, hidden 64, T=12), one process per GPU.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # CPU arm: the oracle port on the host cores
    python bench.py ... --dump-outputs DIR    # also write what the last timed step computed as DIR/<name>.npy

A step = forward + MSE+L1 loss + BPTT + gradient all-reduce + Adam (train.py:96-110) on one batch of
synthetic N(0,1) data of the named shape.  Prints ONE JSON line (rank 0):

  value            K steps with the batch resident in HBM (CUDA events, max over ranks)
  sustained        the same over >= 2 s (the GPU power-caps within a second; short runs flatter it)
  e2e              the same metric through Trainer.step on HOST batches: pinned bf16 windows copied every step
                   (double-buffered), loss read back every step
  e2e_variants     host_window_fp32 (the reference's own staging dtype, train.py:92), host_window_bf16 (= e2e),
                   frame_bank (record resident in HBM, a step uploads B window indices; dataset.py:551-637)
  roofline         the dominant kernel against the measured HBM / tensor peak; kernels: every class, vs burst AND sustained
  gpu_eager_baseline   the same step written with stock PyTorch ops (cuDNN, eager pointwise, autograd, fused Adam) on
                   this GPU: the library kernels to beat
  configs          the other BASELINE.json configurations at their own sizes (N=1 only)
  cpu_baseline     the oracle port on this box's host cores (N=1 only)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True                             # the benchmark leaves the source tree as it found it
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

C_IN, HIDDEN, H, W = 21, 64, 90, 144


def conv_flops(batch, T, k, cin=C_IN, hc=HIDDEN, hw=H * W):
    """Algorithmic (necessary) conv FLOPs per launch class for one training step (SURVEY.md 8d):
    h_{-1}=0 -> no h segment at t=0; no dx for layer 0; padding channels are not counted."""
    n = 4 * hc
    f_x = 2.0 * hw * n * cin * k * k * batch
    f_h = 2.0 * hw * n * hc * k * k * batch
    fwd = T * f_x + (T - 1) * f_h
    return {"gate_conv_fwd": fwd, "dgrad_gate_bwd": (T - 1) * f_h, "wgrad": fwd}


def model_train_flops(batch, T, cin, hidden, ks, hw):
    """necessary conv FLOPs of one training step of a stacked model (fwd + dgrad + wgrad, SURVEY.md 8d)"""
    total, c = 0.0, cin
    for l, (hc, k) in enumerate(zip(hidden, ks)):
        f_x = 2.0 * hw * 4 * hc * c * k * k * batch
        f_h = 2.0 * hw * 4 * hc * hc * k * k * batch
        fwd = T * f_x + (T - 1) * f_h
        total += 2 * fwd + (T - 1) * f_h + (T * f_x if l > 0 else 0.0)
        c = hc
    return total


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons, watts = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
            except (ValueError, IndexError):
                continue
            try:
                watts.append(float(r[2]))
            except (ValueError, IndexError):
                pass
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        watts.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w": watts[len(watts) // 2] if watts else None}


def cpu_oracle_run(batch, T, k, steps, warmup, threads):
    """The CPU arm: oracle port of the reference path (oracle/convlstm_oracle.py), fwd+loss+bwd."""
    from oracle import convlstm_oracle as O
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    params = O.init_params(C_IN, [HIDDEN], [k], seed=0)
    x, y = torch.randn(batch, T, C_IN, H, W), torch.randn(batch, H, W)
    for _ in range(warmup):
        O.forward_backward(x, y, params, 1)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.forward_backward(x, y, params, 1)
    dt = (time.perf_counter() - t0) / steps
    return batch / dt, dt * 1e3


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = len(os.sched_getaffinity(0))
    batch = 2
    sps, ms = cpu_oracle_run(batch, args.seq_len, args.ksize, max(1, min(args.steps, 5)), min(args.warmup, 1), threads)
    sample = f"oracle port (torch CPU fp32), batch {batch} x T={args.seq_len} fwd+loss+bwd per step, {threads} threads"
    print(json.dumps({
        "impl": "reference", "metric": "train samples/sec", "value": round(sps, 4), "unit": "samples/s",
        "n_gpus": args.gpus, "steps": max(1, min(args.steps, 5)), "warmup": min(args.warmup, 1),
        "ms_per_step": round(ms, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"ConvLSTM train step, 90x144x(20 levels+BCB)=21ch, hidden 64, k{args.ksize}, "
                               f"T={args.seq_len}; CPU sample batch {batch}"},
        "cpu_baseline": {"value": round(sps, 4), "unit": "samples/s", "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": round(sps, 4), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------------------------------
def dump_outputs(out_dir, model, loss):
    """What Trainer.step, the timed path, hands its caller after the last timed step: the loss it returns, the
    parameters it updated in place and the gradients it wrote into their .grad (all fp32, 0.8 MB each for parameters and
    gradients at hidden 64, k3).  Inputs and initial weights come from fixed seeds, so two builds can be compared array
    by array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss}
    for name, p in model.named_parameters():
        arrays["param." + name] = p
        arrays["grad." + name] = p.grad
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
    return sorted(arrays)


def cuda_timed(fn, n, dev):
    """ms per call of fn over n calls (CUDA events on the current stream, synchronised on both sides)"""
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / n


def gpu_eager_baseline(B, T, k, dev, steps=3):
    """The same training step with stock PyTorch ops on this GPU (nn.Conv2d -> cuDNN, eager pointwise kernels,
    autograd, fused Adam, bf16 autocast): what the reference's model.py executes on a B200 (SURVEY.md 8d "library kernel
    to beat").  Self-contained: neither the reference (absent on the GPU box) nor oracle/ is imported."""
    import torch.nn as nn
    import torch.nn.functional as F

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.conv = nn.Conv2d(C_IN + HIDDEN, 4 * HIDDEN, k, padding=k // 2)
            self.head = nn.Conv2d(HIDDEN, 1, 1)

        def forward(self, x):
            h = torch.zeros(x.shape[0], HIDDEN, H, W, device=x.device)
            c = torch.zeros_like(h)
            for t in range(x.shape[1]):
                i, f, g, o = torch.split(self.conv(torch.cat([x[:, t], h], 1)), HIDDEN, 1)
                c = c * torch.sigmoid(f) + torch.sigmoid(i) * torch.tanh(g)
                h = torch.sigmoid(o) * torch.tanh(c)
            return self.head(h)

    torch.manual_seed(0)
    net = Net().to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, betas=(0.5, 0.999), fused=True)
    x, y = torch.randn(B, T, C_IN, H, W, device=dev), torch.randn(B, H, W, device=dev)
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.deterministic = False             # cuDNN's fastest algorithms: the library kernels to beat

    def step():
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            p = net(x).squeeze(1).float()
        (F.mse_loss(p, y) + F.l1_loss(p, y)).backward()
        opt.step()
    for _ in range(2):
        step()
    ms = cuda_timed(step, steps, dev)
    del net, opt, x, y
    torch.cuda.empty_cache()
    return {"ms_per_step": round(ms, 2), "value": round(B / ms * 1e3, 1), "unit": "samples/s", "steps": steps,
            "how": f"torch {torch.__version__} eager + cuDNN {torch.backends.cudnn.version()}, bf16 autocast, fused Adam, "
                   f"same shapes (B={B}, T={T}, k{k})"}


def other_configs(dev):
    """BASELINE.json configs 1, 4, 5, cfg 2 with 5x5 kernels, the reference's shipped recipe (launcher.sh:13-30) and the
    only timing the reference publishes (test.ipynb:4585-4586: forward of ConvLSTM(5,[64,32,16],[5,3,3],3) on
    (1,48,5,100,154), 38.7 ms on an A100) -- each at its own size, bf16, this GPU."""
    from nasa_niswan_b200 import ConvLSTM
    from nasa_niswan_b200.parallel import Trainer
    out = {}

    def train(name, B, T, C, Hh, Ww, hidden, ks, crop=None, n=3, note=None):
        torch.manual_seed(0)
        net = ConvLSTM(C, hidden, ks, len(hidden), precision="bf16").to(dev)
        tr = Trainer(net, lr=1e-3, betas=(0.5, 0.999), crop=crop)
        x = torch.randn(B, T, C, Hh, Ww, device=dev)
        yh, yw = (crop[1] - crop[0], crop[3] - crop[2]) if crop else (Hh, Ww)
        y = torch.randn(B, yh, yw, device=dev)
        for _ in range(2):
            tr.step(x, y)
        ms = cuda_timed(lambda: tr.step(x, y), n, dev)
        tf = model_train_flops(B, T, C, hidden, ks, Hh * Ww) / (ms * 1e-3) / 1e12
        out[name] = {"ms_per_step": round(ms, 3), "samples_per_s": round(B / ms * 1e3, 1), "conv_tflops": round(tf, 1),
                     "shape": f"B={B} T={T} C={C} {Hh}x{Ww} hidden {hidden} k {ks}" + (f"; {note}" if note else "")}
        del net, tr, x, y
        torch.cuda.empty_cache()

    train("cfg1_b2_t4", 2, 4, C_IN, H, W, [HIDDEN], [3], n=10, note="BASELINE cfg 1 geometry (the CPU case) on the GPU")
    train("cfg2_k5", 32, 12, C_IN, H, W, [HIDDEN], [5], note="cfg 2 with the reference's real layer-0 kernel size")
    train("cfg5", 8, 12, C_IN, 180, 288, [128, 128, 128], [5, 5, 5], n=2, note="BASELINE cfg 5, B=8 per GPU")
    train("shipped_model", 8, 48, 5, 100, 154, [64, 32, 16], [5, 3, 3], crop=(5, 95, 5, 149), n=2,
          note="launcher.sh:13-30 recipe (batch 8, T=48, crop train.py:102)")
    with torch.no_grad():
        torch.manual_seed(0)
        net = ConvLSTM(C_IN, [HIDDEN], [3], 1, precision="bf16").to(dev)
        x = torch.randn(64, 120, C_IN, H, W, device=dev)
        net(x)
        ms = cuda_timed(lambda: net(x), 3, dev)
        f_full = 2.0 * H * W * 4 * HIDDEN * (C_IN + HIDDEN) * 9 * 64
        out["cfg4_rollout"] = {"ms_per_rollout": round(ms, 2), "us_per_step": round(ms / 120 * 1e3, 1),
                               "samples_per_s": round(64 / ms * 1e3, 1),
                               "conv_tflops": round((120 * f_full - 2.0 * H * W * 256 * HIDDEN * 9 * 64) / (ms * 1e-3) / 1e12, 1),
                               "shape": "B=64 T=120 inference, state resident in HBM (BASELINE cfg 4)"}
        del net, x
        torch.cuda.empty_cache()
        # batch-1 regimes of the reference: val_loop / test.ipynb (utils.py:52-75) and the published %%timeit cell
        net = ConvLSTM(5, [64, 32, 16], [5, 3, 3], 3, precision="bf16").to(dev)
        xh = torch.randn(1, 48, 5, 100, 154).pin_memory()
        xd = xh.to(dev)
        net(xd)
        ms_dev = cuda_timed(lambda: net(xd), 10, dev)
        t0 = time.perf_counter()
        for _ in range(10):
            net(xh.to(dev, non_blocking=True))       # the notebook cell times randn + .cuda() + forward; here H2D + forward
        torch.cuda.synchronize(dev)
        ms_e2e = (time.perf_counter() - t0) * 100.0
        out["published_forward_b1"] = {"ms_device": round(ms_dev, 3), "ms_with_h2d_wall": round(ms_e2e, 3),
                                       "reference_ms_a100": 38.7, "speedup_vs_published": round(38.7 / ms_e2e, 1),
                                       "shape": "ConvLSTM(5,[64,32,16],[5,3,3],3) forward on (1,48,5,100,154): test.ipynb:4585-4586"}
        del net, xd
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="per-GPU batch (weak scaling)")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="fixed GLOBAL batch split over the ranks (strong scaling; 256 = BASELINE cfg 3: 128/64/32 per rank at 2/4/8)")
    ap.add_argument("--seq-len", type=int, default=12)
    ap.add_argument("--ksize", type=int, default=3)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sustained run, eager baseline, e2e variants and configs block")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, parameters and gradients of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from nasa_niswan_b200 import ConvLSTM, _lib
    from nasa_niswan_b200.parallel import HostFeeder, Trainer, bind_to_gpu_numa_node, shard_batch
    from nasa_niswan_b200.preprocess import FrameBank

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(dev)                       # pinned staging buffers land next to this GPU's PCIe root
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W_, K_ = max(3, args.warmup), args.steps
    T, k = args.seq_len, args.ksize
    if args.global_batch:
        b0, b1 = shard_batch(args.global_batch, rank, world)
        B, global_batch, scaling = b1 - b0, args.global_batch, "strong"
    else:
        B, global_batch, scaling = args.batch, args.batch * world, "weak"

    torch.manual_seed(0)                                   # identical init on every rank (utils.py:77-88)
    # the reference trains under seed() (train.py:32 -> utils.py:87: cudnn.deterministic), which selects the fixed-order
    # gradient reductions here: every run of the same arguments computes the same bits (--dump-outputs), instead of
    # fp32-atomic sums whose order differences Adam carries from step to step
    torch.backends.cudnn.deterministic = True
    model = ConvLSTM(C_IN, [HIDDEN], [k], 1, precision=args.precision).to(dev)
    trainer = Trainer(model, lr=1e-3, betas=(0.5, 0.999))
    torch.manual_seed(1 + rank)
    x = torch.randn(B, T, C_IN, H, W, device=dev)          # 418 MB at B=32: larger than the 126 MB L2
    y = torch.randn(B, H, W, device=dev)
    lib = _lib.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---------------- device-resident throughput (`value`)
    for _ in range(W_):
        trainer.step(x, y)
    plan = model.plan_for(x, True)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    plan.profile(True)
    n0 = lib.nint_launch_count(-1)
    cls0 = [lib.nint_launch_count(c) for c in range(4)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K_):
        loss = trainer.step(x, y)
    e1.record()
    barrier()
    launches = lib.nint_launch_count(-1) - n0
    cls_launches = dict(zip(("gate_conv_fwd", "dgrad_gate_bwd", "wgrad", "other"),
                            [lib.nint_launch_count(c) - v for c, v in enumerate(cls0)]))
    prof = plan.profile_read()
    plan.profile(False)
    clocks = sampler.stop() if rank == 0 else None
    ms_step = max_over_ranks(e0.elapsed_time(e1)) / K_
    value = global_batch / (ms_step * 1e-3)
    dumped = None
    if args.dump_outputs and rank == 0:                    # before the runs below train the same model further
        dumped = {"dir": os.path.abspath(args.dump_outputs), "arrays": dump_outputs(args.dump_outputs, model, loss)}

    # ---------------- the same over >= 2 s: the power cap bites after ~1 s, short runs read 3-8 % high
    sustained = None
    if not args.no_extras:
        n_long = max(K_, int(args.sustained_seconds * 1e3 / ms_step) + 1)
        barrier()
        e0.record()
        for _ in range(n_long):
            trainer.step(x, y)
        e1.record()
        barrier()
        ms_long = max_over_ranks(e0.elapsed_time(e1)) / n_long
        sustained = {"value": round(global_batch / (ms_long * 1e-3), 2), "unit": "samples/s", "steps": n_long,
                     "ms_per_step": round(ms_long, 3), "seconds": round(ms_long * n_long * 1e-3, 2)}

    # ---------------- end to end through the public API with host buffers (`e2e`)
    # every step copies its own inputs from pinned host memory (train.py:92-93) and reads its loss back
    # (train.py:113); the copy of batch i+1 overlaps the training of batch i (HostFeeder: what a data loader does)
    e2e_steps = max(3, K_ // 2)
    feeder = HostFeeder(dev)

    def e2e_run(put, step, steps):
        for _ in range(2):
            slot = put()
            float(step(feeder.get(slot)))
            feeder.release(slot)
        barrier()
        e0.record()
        slot = put()
        for i in range(steps):
            args_dev = feeder.get(slot)
            loss_dev = step(args_dev)
            feeder.release(slot)
            if i + 1 < steps:
                slot = put()                                # H2D of the next batch while this one trains
            float(loss_dev)                                 # train.py:113 loss.item(): D2H + sync
        e1.record()
        barrier()
        return global_batch / (max_over_ranks(e0.elapsed_time(e1)) / steps * 1e-3)

    variants = {}
    yh = y.cpu().pin_memory()
    xh16 = x.to(torch.bfloat16).cpu().pin_memory() if args.precision == "bf16" else None
    xh32 = x.cpu().pin_memory() if (xh16 is None or not args.no_extras) else None
    del x, y
    if xh16 is not None:
        v = e2e_run(lambda: feeder.put(xh16, yh), lambda a: trainer.step(*a), e2e_steps)
        variants["host_window_bf16"] = {"value": round(v, 2), "h2d_bytes_per_step": xh16.numel() * 2 + yh.numel() * 4,
                                        "d2h_bytes_per_step": 4, "steps": e2e_steps,
                                        "how": "pinned bf16 windows [B,T,C,H,W] + fp32 targets copied every step (double-buffered "
                                               "on a copy stream), Trainer.step, loss read back every step; bf16 staging gives "
                                               "bit-identical results to fp32 staging (the model rounds x to bf16 anyway)"}
    if xh32 is not None:
        v = e2e_run(lambda: feeder.put(xh32, yh), lambda a: trainer.step(*a), e2e_steps)
        variants["host_window_fp32"] = {"value": round(v, 2), "h2d_bytes_per_step": xh32.numel() * 4 + yh.numel() * 4,
                                        "d2h_bytes_per_step": 4, "steps": e2e_steps,
                                        "how": "the reference's staging dtype (train.py:92: fp32 X.cuda())"}
    headline = "host_window_bf16" if xh16 is not None else "host_window_fp32"
    bank_resident = None
    if not args.no_extras:
        # frame bank: the record lives in HBM once (dataset.py:551-637 keeps it in RAM), a step uploads B window indices
        n_frames = 512
        torch.manual_seed(7 + rank)
        bank = FrameBank.from_frames(torch.randn(n_frames, C_IN, H, W, device=dev), args.precision,
                                     targets=torch.randn(n_frames, H, W, device=dev))
        gen = torch.Generator().manual_seed(rank)
        idx_batches = [torch.randint(0, n_frames - T + 1, (B,), generator=gen, dtype=torch.int32).pin_memory() for _ in range(8)]
        idx_dev = [t.to(dev) for t in idx_batches]
        it = iter(range(10 ** 9))
        for i in range(3):
            trainer.step_windows(bank, idx_dev[i], T)
        barrier()
        e0.record()
        for i in range(K_):
            trainer.step_windows(bank, idx_dev[i % 8], T)
        e1.record()
        barrier()
        ms_bank = max_over_ranks(e0.elapsed_time(e1)) / K_
        bank_resident = {"value": round(global_batch / (ms_bank * 1e-3), 2), "unit": "samples/s", "steps": K_,
                         "ms_per_step": round(ms_bank, 3),
                         "how": "as `value`, with the batch given as window indices into the HBM-resident frame bank: no "
                                "per-step input packing pass (the TMA descriptors read the bank)"}
        v = e2e_run(lambda: feeder.put(idx_batches[next(it) % 8]), lambda a: trainer.step_windows(bank, a[0], T), e2e_steps)
        variants["frame_bank"] = {"value": round(v, 2), "h2d_bytes_per_step": B * 4, "d2h_bytes_per_step": 4, "steps": e2e_steps,
                                  "resident_bytes": bank.frames.numel() * bank.frames.element_size() + bank.targets.numel() * 4,
                                  "how": f"{n_frames}-frame record resident in HBM in the operand layout (uploaded and packed once, "
                                         "outside the timed region); every step copies B int32 window starts from pinned host "
                                         "memory, reads inputs and targets through them, and reads the loss back"}
        del bank

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak_sus = peaks.get("bf16_tflops_sustained", 1400.0)   # kernels timed inside a long step
        peak_burst = peaks.get("bf16_tflops", 1590.0)
        peak_src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md: 1.59 PF burst, 1.4 PF sustained, 6.65 TB/s)"
        if args.precision == "tf32":
            peak_sus, peak_burst, peak_src = peak_sus / 2, peak_burst / 2, peak_src + " / 2 (tf32 nominal half rate)"
        flops = conv_flops(B, T, k)
        kernels = {}
        # n counts TIME STEPS: a time-fused conv launch (all steps of a layer but the first as one persistent launch,
        # DESIGN.md 5.1) counts once per step it covers, so "launches_per_step" / "avg_launch_us" keep meaning "per
        # (layer, time step)" = per launch of the one-launch-per-step schedule; "kernel_launches_per_step" is the
        # number of kernels actually launched
        for name in ("gate_conv_fwd", "dgrad_gate_bwd", "wgrad"):
            ms, n = prof[name]
            if n:
                tf = flops[name] * K_ / (ms * 1e-3) / 1e12
                kernels[name] = {"launches_per_step": n / K_, "kernel_launches_per_step": cls_launches[name] / K_,
                                 "ms_per_step": round(ms / K_, 4),
                                 "avg_launch_us": round(ms / n * 1e3, 2), "tflops": round(tf, 1),
                                 "frac": round(tf / peak_sus, 4), "frac_burst": round(tf / peak_burst, 4)}
        ms_o, n_o = prof["other"]
        dominant = max(kernels, key=lambda n_: kernels[n_]["ms_per_step"])
        conv_ms = sum(v["ms_per_step"] for v in kernels.values())
        # the fused dgrad + gate-backward kernel is HBM-bound (DESIGN.md 5.2).  Algorithmic bytes per pixel of one launch
        # (bf16 gates / fp32 state, hidden 64): gates_t r 512 + dgates_t w 512 + dc w 256 in every launch; the dgrad
        # operand dgates_{t+1} r 512, c_{t-1} r 256 and dc r 256 in T-1 of the T launches (nothing flows into the last
        # step, nothing precedes the first); c_t is recomputed, not read.  Average over the T launches of a step.
        esz = 2 if args.precision == "bf16" else 4
        gates_b, state_b = 4 * HIDDEN * esz, HIDDEN * 4
        bwd_bytes = int(B * H * W * (2 * gates_b + state_b + (gates_b + 2 * state_b) * (T - 1) / T))
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        if "dgrad_gate_bwd" in kernels:
            kb = kernels["dgrad_gate_bwd"]
            per_launch = bwd_bytes * (T / kb["launches_per_step"])     # sub-batch-major schedules launch more, smaller kernels
            kb["hbm_gbs"] = round(per_launch / (kb["avg_launch_us"] * 1e-6) / 1e9, 1)
            kb["hbm_frac"] = round(kb["hbm_gbs"] / hbm_peak, 4)
            kb["bytes_per_launch"] = int(per_launch)
        traffic = None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full captures
            traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(dominant)
        except (OSError, ValueError):
            pass
        if dominant == "dgrad_gate_bwd":
            roof = {"bound": "hbm", "kernel": dominant, "achieved": kernels[dominant]["hbm_gbs"], "peak": hbm_peak,
                    "unit": "GB/s", "frac": kernels[dominant]["hbm_frac"], "traffic": traffic,
                    "peak_source": peak_src + " hbm_gbs", "bytes_per_launch": kernels[dominant]["bytes_per_launch"]}
        else:
            roof = {"bound": "tensor", "kernel": dominant, "achieved": kernels[dominant]["tflops"], "peak": peak_sus,
                    "unit": "TFLOP/s", "frac": kernels[dominant]["frac"], "frac_burst": kernels[dominant]["frac_burst"],
                    "traffic": traffic, "peak_source": peak_src + " bf16_tflops_sustained (kernel timed inside a long step)",
                    "flops_per_launch": flops[dominant] / (kernels[dominant]["launches_per_step"])}
        total_tf = sum(flops.values()) / (conv_ms * 1e-3) / 1e12
        e2e = dict(variants[headline])
        e2e["unit"] = "samples/s"
        e2e["variant"] = headline
        out = {
            "metric": "train samples/sec", "value": round(value, 2), "unit": "samples/s", "n_gpus": world,
            "steps": K_, "warmup": W_, "ms_per_step": round(ms_step, 3), "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": {"workload": f"ConvLSTM train step (fwd+MSE/L1+BPTT+allreduce+Adam), 90x144 grid, 20 levels + BCB "
                                   f"= 21 ch, hidden 64, k{k}, T={T}, batch {B}/GPU (global {global_batch})",
                       "parallelism": f"dp{world}", "l2_policy": "inputs (418 MB/step at B=32) larger than the 126 MB L2",
                       "loss_at_end": round(float(loss), 5), "numa_node": numa, "deterministic": True,
                       "sub_batch": int(os.environ.get("NINT_SUB_BATCH", "0") or 0),
                       "pdl": int(os.environ.get("NINT_PDL", "0") or 0),
                       "time_fused_launches": os.environ.get("NINT_FUSE_STEPS", "auto (BPTT launches fused when short)")},
            "e2e": e2e,
            "e2e_variants": variants,
            "sustained": sustained,
            "frame_bank_resident": bank_resident,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "kernels": kernels,
            "dumped_outputs": dumped,
            "gate_conv_fwd_bwd": {"tflops": round(total_tf, 1), "frac": round(total_tf / peak_sus, 4),
                                  "frac_burst": round(total_tf / peak_burst, 4), "peak_sustained": peak_sus,
                                  "peak_burst": peak_burst, "target": "60 % of bf16 dense peak (BASELINE.md: <= 5.13 ms of conv time at cfg 2)",
                                  "conv_ms_per_step": round(conv_ms, 3), "other_ms_per_step": round(ms_step - conv_ms, 3),
                                  "other_kernels_ms_per_step": round(ms_o / K_, 3), "other_launches_per_step": n_o / K_},
        }
        if world == 1 and not args.no_extras:
            del trainer, model, plan
            torch.cuda.empty_cache()
            out["gpu_eager_baseline"] = gpu_eager_baseline(B, T, k, dev)
            out["gpu_eager_baseline"]["speedup"] = round(out["gpu_eager_baseline"]["ms_per_step"] / ms_step, 2)
            out["configs"] = other_configs(dev)
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)               # the CPU arm gets every host core again
            threads = len(os.sched_getaffinity(0))
            sps, ms = cpu_oracle_run(2, T, k, 3, 1, threads)
            out["cpu_baseline"] = {"value": round(sps, 4), "unit": "samples/s", "cores": threads, "kind": "port",
                                   "sample": f"oracle port (torch CPU fp32) fwd+loss+bwd, batch 2 x T={T}, 3 timed steps "
                                             f"of {ms:.0f} ms, {threads} threads"}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
