#!/usr/bin/env python
"""bench.py — image-pairs/s of the bi-temporal change-detection hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path over one batch of synthetic image pairs on every rank:
``net_G(x1, x2)`` (libstcd_b200) + the evaluator's fused binarise/confusion-matrix kernel, then
the int64[4] all-reduce of the matrix (the path's only collective).  Prints ONE JSON line (rank 0).

* ``value``     pairs/s over all ranks, inputs resident in HBM, CUDA-event timed, max over ranks.
* ``e2e``       the same through the public API with pinned HOST buffers: H2D of the step's pairs
                and labels, forward, metric, D2H of the uint8 change maps and the matrix.
* ``roofline``  the dominant kernel (by device time, from a per-launch CUDA-event pass) against
                the measured peak in MEASURED_PEAKS.json.
* ``cpu_baseline``  the oracle's fp32 CPU forward (torch.nn.functional restatement of the
                reference, oracle/nets.py) on this box's host cores, bounded sample, rank 0, N=1.
``--impl reference`` times that CPU path alone with all host threads and prints the same line.
``--dump-outputs DIR`` writes the last timed step's logits, change map and confusion matrix as .npy files; inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.
The default workloads SNUNet 256^2 and SegCD 1024^2 also time the other one, in an ``also`` object of the same line:
``--steps`` timed steps after a fixed 3 warm-up steps, whatever ``--warmup`` says.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# workload -> (net kind, ctor args, synth gain, H, W, per-GPU batch, binarise kind, config string)
WORKLOADS = {
    "snunet_256_b64": dict(net="SNUNet_ECAM", n_class=2, h=256, w=256, batch=64, kind="argmax", chunk=64,
                           desc="C2: SNUNet-CD (ECAM) 256x256 RGB pairs, batch 64 per GPU, bf16"),
    "siamunet_diff_256": dict(net="SiamUnet_diff", n_class=2, h=256, w=256, batch=8, kind="argmax",
                              desc="C1: SiamUnet_diff 256x256 RGB pairs, batch 8 per GPU"),
    "siamunet_diff_256_b64": dict(net="SiamUnet_diff", n_class=2, h=256, w=256, batch=64, kind="argmax",
                                  desc="SiamUnet_diff 256x256 RGB pairs, batch 64 per GPU"),
    "siamunet_conc_256": dict(net="SiamUnet_conc", n_class=2, h=256, w=256, batch=8, kind="argmax",
                              desc="SiamUnet_conc 256x256 RGB pairs, batch 8 per GPU"),
    "segcd_r34_1024_b16": dict(net="SegCD", n_class=1, h=1024, w=1024, batch=16, kind="sigmoid", chunk=16, input_sets=2, e2e_input="u8",
                               desc="C3: smp SegCD (Unet, ResNet-34 Siamese encoder) 1024x1024 RGB pair tiles, batch 16 per GPU, "
                                    "bf16, + confusion-matrix F1/IoU on sigmoid(change) > 0.5"),
    "segcd_r50_1024_b16": dict(net="SegCD", encoder="resnet50", n_class=1, h=1024, w=1024, batch=16, kind="sigmoid", chunk=8,
                               input_sets=2, e2e_input="u8",
                               desc="smp SegCD with the ResNet-50 encoder train_stcd.py:638 selects, 1024x1024 RGB pair tiles, "
                                    "batch 16 per GPU, bf16, + confusion matrix on sigmoid(change) > 0.5"),
    "changegnn_v1_256_b32": dict(net="ChangeGNNV1", n_class=2, h=256, w=256, batch=32, kind="argmax", chunk=32,
                                 desc="C4: ChangeGNNV1 (pyramid ViG Grapher encoder: dense kNN k=9 + max-relative graph conv, "
                                      "multi-scale difference decoder) 256x256 RGB pairs, batch 32 per GPU, bf16"),
    "changeformer_v6_256_b32": dict(net="ChangeFormerV6", n_class=2, h=256, w=256, batch=32, kind="argmax", chunk=32,
                                    desc="C5: ChangeFormerV6 (MiT transformer encoder + difference decoder) 256x256 RGB pairs, "
                                         "batch 32 per GPU, bf16"),
    "dtcdscn_256_b32": dict(net="CDNet_model", n_class=2, h=256, w=256, batch=32, kind="argmax", chunk=32,
                            desc="DTCDSCN (CDNet34: Siamese SE-ResNet-34, dilated centre block, SCSE decoder on feature differences) "
                                 "256x256 RGB pairs, batch 32 per GPU, bf16"),
    "bit_dd8_256_b32": dict(net="BASE_Transformer", n_class=2, h=256, w=256, batch=32, kind="argmax", chunk=32,
                            desc="BIT base_transformer_pos_s4_dd8 (ResNet-18 stages 1-3, 4 semantic tokens, 1 encoder + 8 decoder layers) "
                                 "256x256 RGB pairs, batch 32 per GPU, bf16 convs + fp32 token path"),
    "changegnn_v2_256_b32": dict(net="ChangeGNNV2", n_class=2, h=256, w=256, batch=32, kind="argmax", chunk=32,
                                 desc="ChangeGNNV2 (pyramid ViG encoder, HFFM + VFFM decoder) 256x256 RGB pairs, batch 32 per GPU, bf16"),
    "gnn_256_b32": dict(net="VIG_V20_2", n_class=2, h=256, w=256, batch=32, kind="argmax", chunk=32,
                        desc="VIG_V20_2 (registry key GNN: pyramid ViG encoder, conv_diff_V20 + csam_V20 + AFF decoder) 256x256 RGB pairs, batch 32 per GPU, bf16"),
    "changeformer_v2_256_b32": dict(net="ChangeFormerV2", n_class=2, h=256, w=256, batch=32, kind="argmax", chunk=32,
                                    desc="ChangeFormerV2 (Tenc MiT encoder depths 3-4-6-3, |fx1 - fx2|, TDec) 256x256 RGB pairs, batch 32 per GPU, bf16"),
    "changeformer_v3_256_b32": dict(net="ChangeFormerV3", n_class=2, h=256, w=256, batch=32, kind="argmax", chunk=32,
                                    desc="ChangeFormerV3 (Tenc MiT encoder, TDecV2 with a PixelShuffle(4) head) 256x256 RGB pairs, batch 32 per GPU, bf16"),
    "changeformer_v1_256_b32": dict(net="ChangeFormerV1", n_class=2, h=256, w=256, batch=32, kind="argmax", chunk=32,
                                    desc="ChangeFormerV1 (Tenc MiT encoder, |fx1 - fx2|, convprojection_base) 256x256 RGB pairs, batch 32 per GPU, bf16"),
    "ifnet_256_b16": dict(net="DSIFN", n_class=1, h=256, w=256, batch=16, kind="sigmoid", chunk=16,
                          desc="IFNet / DSIFN (shared VGG16 features, channel + spatial attention difference decoder) 256x256 RGB pairs, "
                               "batch 16 per GPU, bf16, change = sigmoid(out) > 0.5"),
    "segcd_r34_256_b64": dict(net="SegCD", n_class=1, h=256, w=256, batch=64, kind="sigmoid", chunk=16,
                              desc="smp SegCD (Unet, ResNet-34 Siamese encoder) 256x256 RGB pairs, batch 64 per GPU, bf16"),
}
DEFAULT_WORKLOAD = "snunet_256_b64"


def build_net(wl):
    from stcd_b200 import synth
    from stcd_b200.networks import CLASSES
    if wl["net"] == "SegCD":
        return synth.prepare_(CLASSES["SegCD"](wl.get("encoder", "resnet34"), classes=wl["n_class"]).eval(), "SegCD")
    if wl["net"] == "DSIFN":
        return synth.prepare_(CLASSES["DSIFN"]().eval(), "DSIFN")
    if wl["net"] == "BASE_Transformer":
        net = CLASSES["BASE_Transformer"](3, wl["n_class"], with_pos="learned", resnet_stages_num=4, token_len=4, enc_depth=1, dec_depth=8)
        return synth.prepare_(net.eval(), "BASE_Transformer")
    if wl["net"] in ("VIG_V20_2", "ChangeFormerV1", "ChangeFormerV2", "ChangeFormerV3"):
        return synth.prepare_(CLASSES[wl["net"]]().eval(), wl["net"])
    if wl["net"] in ("ChangeGNNV1", "ChangeFormerV6", "ChangeGNNV2"):
        return synth.prepare_(CLASSES[wl["net"]](3, wl["n_class"], embed_dim=256).eval(), wl["net"])
    return synth.prepare_(CLASSES[wl["net"]](3, wl["n_class"]).eval(), wl["net"])


def oracle_forward(wl, sd, x1, x2):
    from oracle import nets
    if wl["net"] == "SiamUnet_diff":
        return nets.siamunet_forward(sd, x1, x2, "diff")
    if wl["net"] == "SiamUnet_conc":
        return nets.siamunet_forward(sd, x1, x2, "conc")
    if wl["net"] == "SNUNet_ECAM":
        return nets.snunet_forward(sd, x1, x2)
    if wl["net"] == "SegCD":
        return nets.segcd_forward(sd, x1, x2)
    if wl["net"] == "ChangeGNNV1":
        return nets.changegnn_forward(sd, x1, x2)
    if wl["net"] == "ChangeFormerV6":
        return nets.changeformer_forward(sd, x1, x2)
    if wl["net"] == "CDNet_model":
        return nets.dtcdscn_forward(sd, x1, x2)
    if wl["net"] == "BASE_Transformer":
        return nets.bit_forward(sd, x1, x2, stages=4)
    if wl["net"] == "DSIFN":
        return nets.dsifn_forward(sd, x1, x2)
    if wl["net"] == "ChangeGNNV2":
        return nets.changegnn_v2_forward(sd, x1, x2, "cross")
    if wl["net"] == "VIG_V20_2":
        return nets.vig_v20_forward(sd, x1, x2)
    if wl["net"] in ("ChangeFormerV1", "ChangeFormerV2", "ChangeFormerV3"):
        return getattr(nets, "changeformer_v%s_forward" % wl["net"][-1])(sd, x1, x2)
    raise KeyError(wl["net"])


def flops_per_pair(net, wl) -> float:
    return 2.0 * net.lower(wl["h"], wl["w"]).macs_per_pair()


# ------------------------------------------------------------------------------------------ helpers
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


DUMP_BYTES = 60 << 20           # what --dump-outputs writes in all: under 64 MB with the .npy headers


def dump_outputs(out_dir, arrays):
    """Write each tensor of ``arrays`` as ``out_dir/<name>.npy``: int64 counts as float64, everything else as float32.
    Arrays under 1 MiB are written whole.  When the larger ones together exceed what is left of DUMP_BYTES, each keeps
    the same share of its elements, drawn with a fixed seed and written flattened in index order, so the files of two
    builds run with the same arguments compare element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    host = {k: (t.double() if t.dtype == torch.int64 else t.float()).cpu().numpy() for k, t in arrays.items()}
    small = sum(a.nbytes for a in host.values() if a.nbytes < 1 << 20)
    large = sum(a.nbytes for a in host.values() if a.nbytes >= 1 << 20)
    keep = max(0.0, min(1.0, (DUMP_BYTES - small) / max(large, 1)))
    for name, a in host.items():
        if keep < 1.0 and a.nbytes >= 1 << 20:
            idx = np.sort(np.random.default_rng(0).choice(a.size, int(a.size * keep), replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md).  The sampler process is
    started well before the region (nvidia-smi takes a few hundred ms to produce its first line); every row is
    stamped on arrival and `summary()` keeps the rows that fall inside the region [t0, t1] (for a region shorter
    than two sampling periods: the rows nearest to it, taken under the same load during warm-up / e2e)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def __enter__(self):          # timed region begins
        if self.proc is None:
            self.start()
        self.t0 = time.time()
        return self

    def __exit__(self, *a):       # timed region ends
        self.t1 = time.time()

    def stop(self):
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
            self.proc = None

    def summary(self):
        self.stop()
        t0, t1 = self.t0 or 0.0, self.t1 or float("inf")
        inside = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.06]
        near = inside or [r for (t, r) in self.rows if t0 - 1.0 <= t <= t1 + 1.0]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in near:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "samples_inside_timed_region": len(inside)}


def cpu_baseline(wl, seconds_target: float = 15.0, threads: int | None = None):
    """The oracle's CPU forward + numpy confusion matrix on a bounded sample of the workload."""
    from oracle import metric as ometric
    from stcd_b200 import synth
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    net = build_net(wl)
    sd = net.state_dict()
    n = 2 if wl["h"] * wl["w"] < 512 * 512 else 1
    x1, x2 = synth.image_pairs(n, wl["h"], wl["w"])
    lab = synth.labels(n, wl["h"], wl["w"]).numpy()

    def step():
        with torch.no_grad():
            y = oracle_forward(wl, sd, x1, x2)
        y = y[-1] if isinstance(y, (list, tuple)) else y
        ometric.confusion_matrix(ometric.binarise(y.numpy(), wl["kind"]), lab)

    t0 = time.perf_counter()
    step()                                   # warm-up (also sizes the sample)
    t_one = time.perf_counter() - t0
    reps = max(1, min(20, int(seconds_target / max(t_one, 1e-3))))
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2]
    return {"value": n / med, "unit": "pairs/s", "cores": threads, "kind": "port",
            "sample": f"{reps} x {n} pairs of {wl['h']}x{wl['w']} (median), oracle/nets.py fp32 torch CPU + numpy bincount"}


# ------------------------------------------------------------------------------------------ arms
def reference_forward(wl, net):
    """The UNMODIFIED reference module for this workload, fed with our net's state_dict (identical names), when
    /root/reference is present (build container; oracle/refimport.py); else None -> the oracle port is timed."""
    try:
        from oracle import refimport
        if not refimport.available():
            return None
        where = {"SNUNet_ECAM": ("models.SNUNet", "SNUNet_ECAM", (3, wl["n_class"])),
                 "SiamUnet_diff": ("models.SiamUnet_diff", "SiamUnet_diff", (3, wl["n_class"])),
                 "SiamUnet_conc": ("models.SiamUnet_conc", "SiamUnet_conc", (3, wl["n_class"])),
                 "SegCD": ("segmentation_models_pytorch", "SegCD", (wl.get("encoder", "resnet34"), 5, None))}.get(wl["net"])
        if where is None:
            return None
        ref = getattr(refimport.ref_module(where[0]), where[1])(*where[2]).eval()
        ref.load_state_dict(net.state_dict())
        return ref
    except Exception as e:      # any import trouble: fall back to the port, say so
        print(f"bench.py: reference import failed ({e!r}); timing the oracle port", file=sys.stderr)
        return None


def run_reference(args, wl, rank, world):
    """The reference arm: the reference's own CPU forward + its bincount evaluator on this box's host cores, all
    threads, on a BOUNDED sample of the workload per step (``config.pairs_per_step`` pairs of the workload's size --
    the full batch of 64 would take minutes per step on a CPU)."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    from oracle import metric as ometric
    from stcd_b200 import synth
    net = build_net(wl)
    sd = net.state_dict()
    ref = reference_forward(wl, net)
    n = 2 if wl["h"] * wl["w"] < 512 * 512 else 1   # bounded sample per step
    x1, x2 = synth.image_pairs(n, wl["h"], wl["w"])
    lab = synth.labels(n, wl["h"], wl["w"]).numpy()

    def step():
        with torch.no_grad():
            y = ref(x1, x2) if ref is not None else oracle_forward(wl, sd, x1, x2)
        y = y[-1] if isinstance(y, (list, tuple)) else y
        ometric.confusion_matrix(ometric.binarise(y.numpy(), wl["kind"]), lab)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = n * args.steps / dt
    kind = "reference" if ref is not None else "port"
    sample = (f"{n} pairs of {wl['h']}x{wl['w']} per step, {args.steps} steps; "
              + ("unmodified reference module from /root/reference" if ref is not None else "oracle/nets.py port (no /root/reference on this box)")
              + " + numpy bincount evaluator")
    print(json.dumps({
        "impl": "reference", "metric": "image-pairs/sec", "value": v, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "batch_per_gpu": wl["batch"], "h": wl["h"], "w": wl["w"],
                   "pairs_per_step": n,
                   "note": f"bounded sample: each timed step is {n} pair(s) of the workload's size, not the full batch"},
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def pin_to_gpu_numa(local_rank: int):
    """Bind this rank's threads (and, by first touch, the pinned host buffers it allocates afterwards) to the NUMA node
    its GPU hangs off, so eight ranks' H2D copies do not all cross the same socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local_rank)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:              # nvml prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"numa_node": None}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:                           # no sysfs / nvml in this container: run unpinned
        return {"numa_node": None, "why": repr(e)[:80]}


def run_ours(args, wl, rank, world, local_rank):
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — stcd_b200 has no CPU path (use --impl reference for the CPU arm)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa = pin_to_gpu_numa(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    out = measure(args, args.workload, wl, rank, world, local_rank, dev, full=True)
    # BASELINE.json's metric names both sizes ("at 256^2 and 1024^2"): the other headline configuration rides
    # along as a compact object (same --steps, no CPU leg) so one default run reports both
    other = {"snunet_256_b64": "segcd_r34_1024_b16", "segcd_r34_1024_b16": "snunet_256_b64"}.get(args.workload)
    if other and not args.no_also:
        import copy
        a2 = copy.copy(args)
        wl2 = WORKLOADS[other]
        a2.workload, a2.chunk, a2.input_sets = other, wl2.get("chunk", 32), wl2.get("input_sets", 4)
        a2.warmup, a2.no_cpu_baseline = 3, True
        torch.cuda.empty_cache()
        o2 = measure(a2, other, wl2, rank, world, local_rank, dev, full=False)
        if out is not None and o2 is not None:
            out["also"] = {k: o2[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "config",
                                              "e2e", "e2e_u8", "gpu_launches", "roofline") if k in o2}
            if "e2e_f32" in o2:
                out["also"]["e2e_f32"] = o2["e2e_f32"]
    if out is not None:
        out["host"] = {"cores": os.cpu_count(), "rank0_affinity": numa}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def measure(args, wl_name, wl, rank, world, local_rank, dev, full=True):
    """One workload on this rank's GPU: returns the JSON object on rank 0, None elsewhere."""
    import torch.distributed as dist
    from stcd_b200 import synth
    from stcd_b200.metric import SegmentationMetric

    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    B, H, W = wl["batch"], wl["h"], wl["w"]
    net = build_net(wl).to(dev)
    net.chunk_pairs = args.chunk
    fl_pair = flops_per_pair(net, wl)
    metric = SegmentationMetric(2, dev)
    n_sets = args.input_sets                 # rotate distinct batches: working set > L2 (126 MB)
    hx1, hx2, hlab = [], [], []
    for s in range(n_sets):
        a, b = synth.image_pairs(B, H, W, seed=synth.DATA_SEED + 100 * rank + s)
        hx1.append(a.pin_memory())
        hx2.append(b.pin_memory())
        hlab.append(synth.labels(B, H, W, seed=synth.DATA_SEED + 7 + 100 * rank + s).to(torch.uint8).pin_memory())
    dx1 = [t.to(dev) for t in hx1]
    dx2 = [t.to(dev) for t in hx2]
    dlab = [t.to(dev) for t in hlab]
    plan = net.plan_for(dx1[0])
    logits = [torch.empty(s, dtype=torch.float32, device=dev) for s in plan.out_shapes(B)]
    pred = torch.empty(B, H, W, dtype=torch.uint8, device=dev)
    hpred = torch.empty(B, H, W, dtype=torch.uint8).pin_memory()
    hcm = torch.empty(4, dtype=torch.int64).pin_memory()

    def step(i):
        s = i % n_sets
        plan.forward(dx1[s], dx2[s], outs=logits)
        metric.addLogits(logits[-1], dlab[s], kind=wl["kind"], pred_out=pred)

    # the path's only collective: the int64 matrix is summed over the ranks ONCE per evaluation, like the reference
    # reads its matrix once after the loop (train_stcd.py:488-492) -- inside the timed region, after the last step
    step.finish = metric.allreduce

    # End to end through the public API (net(x1, x2) + SegmentationMetric.addLogits) with HOST buffers.  Like a
    # DataLoader(pin_memory=True) + non_blocking prefetcher, the H2D copy of step i+1 rides a copy stream while
    # step i computes; every step's inputs cross PCIe inside the timed region and every step's change map and
    # confusion matrix are read back.
    copy_stream = torch.cuda.Stream(dev)

    def make_e2e(host_a, host_b, fwd):
        slots = [dict(a=torch.empty_like(host_a[0], device=dev), b=torch.empty_like(host_b[0], device=dev),
                      lab=torch.empty_like(dlab[0]), ready=torch.cuda.Event(), free=torch.cuda.Event()) for _ in range(2)]
        state = {"next": None}

        def issue_h2d(i):
            s, slot = i % n_sets, slots[i % 2]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(slot["free"])          # the compute that last read this slot is done
                slot["a"].copy_(host_a[s], non_blocking=True)
                slot["b"].copy_(host_b[s], non_blocking=True)
                slot["lab"].copy_(hlab[s], non_blocking=True)
                slot["ready"].record(copy_stream)

        def step_fn(i):
            if state["next"] != i:
                issue_h2d(i)
            issue_h2d(i + 1)
            state["next"] = i + 1
            slot = slots[i % 2]
            cur = torch.cuda.current_stream(dev)
            cur.wait_event(slot["ready"])
            y = fwd(slot["a"], slot["b"])
            y = y[-1] if isinstance(y, (list, tuple)) else y
            metric.addLogits(y, slot["lab"], kind=wl["kind"], pred_out=pred)
            slot["free"].record(cur)
            hpred.copy_(pred, non_blocking=True)
            hcm.copy_(metric.confusion_counts().reshape(-1), non_blocking=True)

        def finish():
            metric.allreduce()
            hcm.copy_(metric.confusion_counts().reshape(-1), non_blocking=True)

        step_fn.reset = lambda: state.update(next=None)   # the timed region starts with nothing prefetched
        step_fn.finish = finish
        return step_fn

    step_e2e = make_e2e(hx1, hx2, net)
    # the same with the decoded uint8 HWC images the reference's loader starts from (data/dataset.py:196-203):
    # ToTensor + Normalize run in the input-pack kernel, a quarter of the PCIe bytes (SURVEY.md §8(f)-1)
    gu = torch.Generator().manual_seed(77 + rank)
    if True:
        hu1 = [torch.randint(0, 256, (B, H, W, 3), generator=gu, dtype=torch.uint8).pin_memory() for _ in range(n_sets)]
        hu2 = [torch.randint(0, 256, (B, H, W, 3), generator=gu, dtype=torch.uint8).pin_memory() for _ in range(n_sets)]
        step_e2e_u8 = make_e2e(hu1, hu2, net.forward_uint8)

    def timed(fn, steps, warmup, sampler=None):
        for i in range(warmup):
            fn(i)
        if hasattr(fn, "reset"):
            fn.reset()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler is not None:
            sampler.__enter__()
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        if hasattr(fn, "finish"):
            fn.finish()
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        if sampler is not None:
            sampler.__exit__()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    ms_total = timed(step, args.steps, args.warmup, sampler)
    if full and rank == 0 and args.dump_outputs:
        # the last timed step's logits and change map (the e2e passes below overwrite these buffers) and that step's own
        # confusion matrix: the evaluator kernel run again on its logits and labels into a fresh accumulator, since
        # `metric` holds the sum over the warm-up and timed steps
        last = SegmentationMetric(2, dev)
        last.addLogits(logits[-1], dlab[(args.warmup + args.steps - 1) % n_sets], kind=wl["kind"])
        outs = {("logits" if len(logits) == 1 else f"logits{i}"): t for i, t in enumerate(logits)}
        outs.update(change_map=pred, confusion_matrix=last.confusion_counts())
        dump_outputs(args.dump_outputs, outs)
    metric.reset()
    ms_e2e = timed(step_e2e, args.steps, max(1, args.warmup // 2))
    metric.reset()
    ms_e2e_u8 = timed(step_e2e_u8, args.steps, max(3, args.warmup // 2))
    value = world * B * args.steps / (ms_total / 1e3)
    e2e = world * B * args.steps / (ms_e2e / 1e3)
    e2e_u8 = world * B * args.steps / (ms_e2e_u8 / 1e3)

    # consistency check of the evaluator inside the run: counts sum to the pixels seen
    torch.cuda.synchronize(dev)

    if rank == 0:
        peaks = measured_peaks()
        # ---- dominant kernel: per-launch CUDA-event pass (same inputs, after the timed region)
        prof = plan.profile(dx1[0], dx2[0])
        prof = [p for p in prof if p[1] > 0]
        total_ms = sum(p[1] for p in prof)
        top = max(prof, key=lambda p: p[1])
        # the top op's two roofs: tensor (reference-equivalent FLOPs) and HBM (algorithmic bytes, DESIGN.md §4);
        # the one that would take longer at peak is the bound the kernel is reported against
        from stcd_b200 import lowering as L
        op_by_name = {o.name: o for o in plan.prog.ops}
        top_op = op_by_name[top[0]]
        top_bytes = L.op_bytes_per_pair(plan.prog, top_op) * B
        top_flops = 2.0 * top[2]
        top_s = top[1] * 1e-3
        t_tensor = top_flops / (peaks["tf_burst"] * 1e12)
        t_hbm = top_bytes / (peaks["hbm"] * 1e9)
        kname = ("conv_ws_kernel" if isinstance(top_op, L.ConvSpec) else type(top_op).__name__) + f"[{top[0]}]"
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")      # per-op DRAM bytes from the round's ncu tables
        if os.path.exists(tpath):
            tr = json.load(open(tpath)).get(wl_name, {}).get(top[0])
            if tr:                                   # ncu --set full: dram bytes read + written, per pair -> per launch
                traffic = int(tr["dram_bytes_per_pair"] * min(args.chunk, B))
        launches = max(1, -(-B // args.chunk))        # the profile pass sums the op over its launches (chunks)
        if t_tensor >= t_hbm:
            ach = top_flops / top_s / 1e12
            roof = {"bound": "tensor", "achieved": round(ach, 2), "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                    "frac": round(ach / peaks["tf_burst"], 4)}
        else:
            ach = top_bytes / top_s / 1e9
            roof = {"bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": round(ach / peaks["hbm"], 4)}
        step_tf = fl_pair * B / (ms_total / args.steps * 1e-3) / 1e12
        roof.update({"traffic": traffic, "kernel": kname, "kernel_share_of_step": round(top[1] / total_ms, 4),
                     "launches_per_step": launches, "algorithmic_bytes_per_launch": int(top_bytes / launches),
                     "algorithmic_flops_per_launch": int(top_flops / launches),
                     "avg_launch_ms": round(top[1] / launches, 4),
                     "peak_source": f"{peaks['src']} ({'bf16 burst' if t_tensor >= t_hbm else 'copy bandwidth'}; kernel timed alone with CUDA events)",
                     "whole_step": {"achieved": round(step_tf, 2), "peak": peaks["tf_sust"],
                                    "frac": round(step_tf / peaks["tf_sust"], 4), "unit": "TFLOP/s",
                                    "flops_per_pair": fl_pair}})
        out = {
            "metric": "image-pairs/sec", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": wl["desc"], "batch_per_gpu": B, "global_batch": B * world, "h": H, "w": W,
                       "parallelism": f"dp{world}", "chunk_pairs": args.chunk,
                       "l2": f"{n_sets} distinct input batches rotated; activations per step exceed the 126 MB L2"},
            "e2e": {"value": e2e, "unit": "pairs/s",
                    "h2d_bytes_per_step": int(2 * B * 3 * H * W * 4 + B * H * W),
                    "d2h_bytes_per_step": int(B * H * W + 32),
                    "input": "fp32 NCHW host tensors (what the reference's loader hands to net_G: data/dataset.py:196-203)"},
            "e2e_u8": {"value": e2e_u8, "unit": "pairs/s", "h2d_bytes_per_step": int(2 * B * 3 * H * W + B * H * W),
                       "d2h_bytes_per_step": int(B * H * W + 32),
                       "input": "uint8 HWC host images (the decoded RGB the reference's loader STARTS from)",
                       "note": "net.forward_uint8: uint8 HWC host images, ToTensor+Normalize fused into the input-pack kernel"},
            "gpu_launches": int((plan.launches(B) + 1) * args.steps),
            "clocks": sampler.summary() if sampler else None,
            "roofline": roof,
            "per_op_ms": [[n, round(ms, 4)] for n, ms, _ in prof],
        }
        if wl.get("e2e_input") == "u8":
            # 1024x1024 tiles: fp32 pairs are 25 MB each -- eight ranks' H2D copies (3.4 GB per step) saturate the host side
            # (round 1: e2e efficiency 0.47 at 8 GPUs).  The end-to-end path for these workloads is the uint8 loader fusion
            # (a quarter of the PCIe bytes, bit-identical logits: tests/test_gpu_uint8.py); the fp32 figure stays as e2e_f32.
            out["e2e_f32"], out["e2e"] = out["e2e"], out["e2e_u8"]
        if not full:
            out.pop("per_op_ms")
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(wl)
        return out
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--chunk", type=int, default=0, help="image pairs per pass through the layer stack (0: the workload's default)")
    ap.add_argument("--input-sets", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the compact run of the other headline configuration")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's outputs to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    wl = WORKLOADS[args.workload]
    args.chunk = args.chunk or wl.get("chunk", 32)
    args.input_sets = args.input_sets or wl.get("input_sets", 4)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
    else:
        if args.gpus > 1 and world == 1:
            raise SystemExit("bench.py: launch N>1 with torch.distributed.run (one rank per GPU)")
        run_ours(args, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
