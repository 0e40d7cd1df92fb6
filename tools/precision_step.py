"""Step time of a bench.py workload (default changeformer_v6_256_b32, config C5: ChangeFormerV6, 32 pairs of 256 x 256, chunk 32)
at bf16 and on the precision path ("tf32": split-bf16 operands), measured in one process on one GPU.  The net, batch and chunk
are bench.py's (WORKLOADS, build_net).

    python tools/precision_step.py [--workload changeformer_v6_256_b32] [--reps 3] [--window 2.0] [--profile-dir DIR]

* the card's name, power limit and max SM clock (nvidia-smi, read-only query);
* the two precisions alternate, each repeated --reps times; a timed window is >= --window seconds of back-to-back steps on
  device-resident inputs between two CUDA events after a synchronise (C5's inputs are 2 x 25 MB: the working set is the plan's
  ~GB of activations, far beyond the 126 MB L2);
* per-op device time of one step of each precision (the plan's own CUDA events around every launch), summed by op kind;
* a separate torch.profiler pass over tf32 steps: per-kernel device time of the split kernels (template argument `true`) and
  of the conv kernel.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from stcd_b200 import lowering as L, synth  # noqa: E402


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


def window(net, a, b, seconds: float, est_ms: float) -> float:
    """pairs/s over >= `seconds` of back-to-back steps."""
    n = max(3, int(seconds * 1e3 / est_ms) + 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        net(a, b)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    assert ms >= seconds * 1e3 * 0.9, f"window too short: {ms:.0f} ms"
    return n * a.shape[0] / (ms / 1e3)


def op_kind(prog, name: str) -> str:
    op = next(o for o in prog.ops if o.name == name)
    if isinstance(op, L.ConvSpec):
        return "conv (K-partitioned)" if (".part" in op.name or (op.res or "").endswith(".part0")) else "conv"
    return type(op).__name__


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="changeformer_v6_256_b32", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--window", type=float, default=2.0)
    ap.add_argument("--profile-dir", default=None, help="also export the profiler trace there")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (no CPU timing)")
    print(card())
    print(torch.cuda.get_device_name(0))
    wl = bench.WORKLOADS[args.workload]
    print(f"{args.workload}: {wl['desc']}")
    net = bench.build_net(wl).cuda()
    net.chunk_pairs = wl.get("chunk", net.default_chunk_pairs)
    x1, x2 = synth.image_pairs(wl["batch"], wl["h"], wl["w"])
    a, b = x1.cuda(), x2.cuda()
    est = {}
    for prec in ("bf16", "tf32"):                       # warm-up: plans, modules, clocks
        net.precision = prec
        for _ in range(3):
            net(a, b)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            net(a, b)
        e1.record()
        e1.synchronize()
        est[prec] = e0.elapsed_time(e1) / 5
    rates = defaultdict(list)
    for rep in range(args.reps):
        for prec in ("bf16", "tf32"):
            net.precision = prec
            rates[prec].append(window(net, a, b, args.window, est[prec]))
            print(f"rep {rep} {prec}: {rates[prec][-1]:.1f} pairs/s")
    med = {p: sorted(v)[len(v) // 2] for p, v in rates.items()}
    spread = {p: (max(v) - min(v)) / med[p] for p, v in rates.items()}
    print(f"{args.workload} bf16: {med['bf16']:.1f} pairs/s (spread {100 * spread['bf16']:.1f} %), tf32: {med['tf32']:.1f} pairs/s "
          f"(spread {100 * spread['tf32']:.1f} %); tf32 step / bf16 step = {med['bf16'] / med['tf32']:.2f}x")

    # per-op device time of one step (the plan's CUDA events around every launch), by op kind
    kinds = {}
    for prec in ("bf16", "tf32"):
        net.precision = prec
        plan = net.plan_for(a)
        rows = plan.profile(a, b)
        agg = defaultdict(float)
        for name, ms, _ in rows:
            agg[op_kind(plan.prog, name)] += ms
        kinds[prec] = agg
    print("per-op-kind device ms per step (bf16 | tf32 | ratio):")
    for k in sorted(set(kinds["bf16"]) | set(kinds["tf32"]), key=lambda k: -kinds["tf32"].get(k, 0)):
        b16, t32 = kinds["bf16"].get(k, 0.0), kinds["tf32"].get(k, 0.0)
        print(f"  {k:24s} {b16:8.2f} | {t32:8.2f} | {t32 / b16 if b16 else float('nan'):5.2f}")
    print(f"  {'total':24s} {sum(kinds['bf16'].values()):8.2f} | {sum(kinds['tf32'].values()):8.2f}")

    # torch.profiler, a separate pass: device time per kernel over tf32 steps
    from torch.profiler import ProfilerActivity, profile
    net.precision = "tf32"
    steps = 3
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            net(a, b)
        torch.cuda.synchronize()
    if args.profile_dir:
        os.makedirs(args.profile_dir, exist_ok=True)
        prof.export_chrome_trace(os.path.join(args.profile_dir, "precision_step_tf32.json"))
    print(f"torch.profiler, tf32, per step ({steps} steps): kernel | calls | device ms")
    for ev in sorted(prof.key_averages(), key=lambda e: -e.device_time_total):
        if "<true>" in ev.key or ", true>" in ev.key or "conv_ws_kernel" in ev.key:
            print(f"  {ev.key[:110]:110s} {ev.count // steps:5d} {ev.device_time_total / 1e3 / steps:9.3f}")


if __name__ == "__main__":
    main()
