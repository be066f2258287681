"""Cost of the stateful path: ms per training step at BASELINE cfg 2 (B=32, T=12, 21 -> 64 channels, 3x3, 90x144,
bf16) with and without an explicit initial state, CUDA events around --steps steps of each, the two alternated
--rounds times.  The stateful step starts from a nonzero (h0, c0) that requires grad and puts h_T and c_T in the loss,
so it adds the t=0 h segment of the gate convolution, the state pack / unpack kernels, the dL/dh_T and dL/dc_T staging
and the dh0 dgrad; it prints both times, the card name and its power limit as one JSON line.

    python tools/state_step_time.py --steps 50 --rounds 3
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
from nasa_niswan_b200 import ConvLSTM  # noqa: E402


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--seq-len", type=int, default=12)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: the step times are GPU times")
    dev = torch.device("cuda", 0)
    B, T, C, H, W, hc = a.batch, a.seq_len, 21, 90, 144, 64
    torch.manual_seed(0)
    net = ConvLSTM(C, [hc], [3], 1, precision="bf16").to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    x = torch.randn(B, T, C, H, W, device=dev)
    y = torch.randn(B, H, W, device=dev)
    h0 = (torch.randn(B, hc, H, W, device=dev) * 0.5).requires_grad_(True)
    c0 = (torch.randn(B, hc, H, W, device=dev) * 0.5).requires_grad_(True)

    def step(stateful):
        opt.zero_grad(set_to_none=True)
        if stateful:
            pred, ((h, c),) = net(x, hidden_state=[(h0, c0)], return_state=True)
            extra = 1e-3 * (h.square().mean() + c.square().mean())
        else:
            pred, extra = net(x), 0.0
        loss = F.mse_loss(pred.squeeze(1), y) + F.l1_loss(pred.squeeze(1), y) + extra
        loss.backward()
        opt.step()

    def timed(stateful):
        for _ in range(a.warmup):
            step(stateful)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            step(stateful)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / a.steps

    times = {"stateless": [], "stateful": []}
    for _ in range(a.rounds):
        for mode in ("stateless", "stateful"):
            times[mode].append(round(timed(mode == "stateful"), 4))
    best = {k: min(v) for k, v in times.items()}
    print(json.dumps({"shape": f"B={B} T={T} 21->64 3x3 90x144 bf16", "ms_per_step": times,
                      "stateful_over_stateless": round(best["stateful"] / best["stateless"], 4),
                      "device": torch.cuda.get_device_name(dev), "power_limit": power_limit()}))


if __name__ == "__main__":
    main()
