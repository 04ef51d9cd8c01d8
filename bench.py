#!/usr/bin/env python
"""Headline benchmark: ViT-B/16 @ 224 bf16 forward throughput (images/s) of the B200-native encoder path.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU forward (oracle port) on host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's output as DIR/*.npy

A step = one forward of the model over one batch of synthetic images (BASELINE.json configs[1]: ViT-B/16 augreg 224,
197 tokens, GLOBAL batch 1024, random-init weights). With N GPUs the batch is sharded (1024 / N images per GPU,
"scaling": "strong" — the configuration BASELINE.json / SURVEY §8(d) name); `--scaling weak` keeps 1024 images per GPU
instead, and a short weak-scaled measurement is reported beside the strong one when N > 1.
Prints ONE JSON line (rank 0). See DESIGN.md §Measurement.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
RESULT_OUT = sys.stdout  # replaced in __main__ by a duplicate of the original stdout
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (constructor, per-GPU batch, input shape, kind, n_heads for the oracle, pool, tokens per sample)
    "c2": dict(desc="ViT-B/16 augreg 224px (197 tokens), bf16", batch=1024, shape=(3, 224, 224), kind="vit",
               make=lambda pm: pm.ViT.from_google("B/16"), heads=12, pool="cls_token", L=197, layers=12, d=768, P=196, p=16),
    "c3": dict(desc="ViT-L/16 SigLIP 384px (576 tokens), bf16", batch=256, shape=(3, 384, 384), kind="vit",
               make=lambda pm: pm.ViT.from_google("L/16_siglip", img_size=384), heads=16, pool="mha", L=576, layers=24,
               d=1024, P=576, p=16),
    "c4": dict(desc="DINOv2 L/14 518px (1370 tokens), bf16", batch=128, shape=(3, 518, 518), kind="vit",
               make=lambda pm: pm.ViT.from_facebook("L/14_dinov2"), heads=16, pool="cls_token", L=1370, layers=24,
               d=1024, P=1369, p=14),
    "c5": dict(desc="Whisper large-v3 encoder (3000 mel frames -> 1500 tokens), bf16", batch=64, shape=(128, 3000),
               kind="whisper", make=lambda pm: pm.WhisperEncoder(32, 1280, 128), heads=20, pool=None, L=1500, layers=32,
               d=1280, P=0, p=0),
}


def flops_per_sample(c: dict) -> float:
    """Algorithmic FLOPs (SURVEY §8(d)): F_embed + layers * (24 L d^2 + 4 L^2 d); biases/LN/GELU/softmax excluded."""
    L, d = c["L"], c["d"]
    if c["kind"] == "vit":
        embed = 2.0 * c["P"] * (3 * c["p"] ** 2) * d
    else:
        embed = 2.0 * 3000 * 128 * 3 * d + 2.0 * 1500 * d * 3 * d
    return embed + c["layers"] * (24.0 * L * d * d + 4.0 * L * L * d)


def synthetic_weights_(model: torch.nn.Module, seed: int) -> None:
    """Random-init weights of the named architecture (no checkpoints offline): default nn init under manual_seed(0)
    plus seeded noise in the tensors the architecture zero/one-initialises (cls_token, pe, pos_embs, LayerNorm)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for k, v in model.state_dict().items():
            parts = k.split(".")
            is_norm = len(parts) >= 2 and "norm" in parts[-2]
            if k in ("cls_token", "pe", "pos_embs", "pooler.probe"):
                v.copy_(0.02 * torch.randn(v.shape, generator=g))
            elif is_norm and parts[-1] == "weight":
                v.copy_(1.0 + 0.1 * torch.randn(v.shape, generator=g))
            elif is_norm and parts[-1] == "bias":
                v.copy_(0.1 * torch.randn(v.shape, generator=g))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.lines: list[tuple[float, str]] = []  # (arrival time, csv line)
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self) -> None:
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0: float | None = None, t1: float | None = None) -> dict:
        """Median SM clock / reasons over the samples that arrived inside [t0, t1] (host times bracketing the timed
        region). The sampler is started before the warm-up steps; if the timed region is shorter than the sampling
        interval and holds no sample, the samples of warm-up + timed region are used and the line says so."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        window = "timed region"
        lines = [ln for ts, ln in self.lines if t0 is None or t0 <= ts <= (t1 if t1 is not None else ts)]
        if not lines:
            lines = [ln for _, ln in self.lines]
            window = "warm-up + timed region (the timed region is shorter than the sampling interval)"
        for line in lines:
            f = [t.strip() for t in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])), smax.append(float(f[1])), power.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


def measured_peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(source="measured", burst=p["bf16_tflops"], sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    hbm=p["hbm_gbs"])
    return dict(source="fallback", burst=1590.0, sustained=1400.0, hbm=6650.0)


def bind_to_gpu_numa_node(index: int) -> dict:
    """Pin this process (and therefore the pinned staging buffers it first-touches) to the CPUs of the NUMA node the
    GPU hangs off. Under torchrun the ranks otherwise land anywhere, and H2D copies from the far socket were the
    6-7 % end-to-end loss of the round-1 multi-GPU runs."""
    info: dict = {"numa_node": None, "cpus": None}
    try:
        pr = torch.cuda.get_device_properties(index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        info["pci"] = bdf
        if node < 0:
            return info
        cpus: set[int] = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info.update(numa_node=node, cpus=len(allowed))
    except (OSError, ValueError, AttributeError):
        pass
    return info


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, y: torch.Tensor, rank: int, world: int) -> None:
    """Writes `y`, the forward's output in the last timed step, as float32 .npy. Weights and images are seeded, so the
    same arguments give the same inputs on every run. Above 64 MB in all (e.g. the Whisper encoder's 64 x 1500 x 1280
    tokens) a fixed, seeded subset of the samples is written, in batch order; the same subset on every run."""
    import numpy as np

    limit = DUMP_BYTES // world
    keep = max(1, min(y.shape[0], limit // max(4 * y[0].numel(), 1)))
    if keep < y.shape[0]:
        idx = torch.randperm(y.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        y = y[idx.to(y.device)]
    os.makedirs(out_dir, exist_ok=True)
    name = "embeddings" if world == 1 else f"embeddings_rank{rank}"
    np.save(os.path.join(out_dir, f"{name}.npy"), y.float().cpu().numpy())


def committed_traffic(config: str, per_gpu_batch: int) -> dict | None:
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed `ncu --set full`
    capture of this configuration: profiles/r02/ncu_traffic.json, written by scripts/ncu_summary.py from the .ncu-rep
    of `scripts/gpu_ncu.sh`. None when there is no capture for this (config, batch)."""
    path = os.path.join(ROOT, "profiles", "r02", "ncu_traffic.json")
    if not os.path.exists(path):
        return None
    try:
        doc = json.load(open(path))
    except (OSError, ValueError):
        return None
    return doc.get(f"{config}_b{per_gpu_batch}")


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_forward_fn(cfg: dict, n_samples: int):
    """The reference's CPU path (fp32, all host threads) as restated by oracle/oracle_torch.py on the same config."""
    import pytorch_models_b200 as pm
    from oracle import oracle_torch  # the CPU arm is the one place bench.py may execute the oracle

    torch.manual_seed(0)
    model = cfg["make"](pm).eval()
    synthetic_weights_(model, 100)
    sd = {k: v.float() for k, v in model.state_dict().items()}
    torch.manual_seed(1)
    x = torch.randn(n_samples, *cfg["shape"])

    @torch.no_grad()
    def run():
        if cfg["kind"] == "vit":
            return oracle_torch.vit_forward(sd, x, cfg["heads"], cfg["pool"])
        return oracle_torch.whisper_encoder_forward(sd, x)

    return run


def cpu_sample_size(name: str) -> int:
    return {"c2": 32, "c3": 4, "c4": 2, "c5": 1}[name]


def time_cpu(cfg: dict, name: str, steps: int, warmup: int) -> tuple[float, int, int]:
    n = cpu_sample_size(name)
    run = cpu_forward_fn(cfg, n)
    for _ in range(warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = (time.perf_counter() - t0) / steps
    return dt, n, torch.get_num_threads()


def run_reference_arm(args, cfg: dict) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    dt, n, threads = time_cpu(cfg, args.config, args.steps, args.warmup)
    value = n / dt
    line = {
        "impl": "reference", "metric": "ViT-B/16 img/s bf16" if args.config == "c2" else f"{args.config} samples/s bf16",
        "value": value, "unit": "img/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": cfg["desc"], "arm": "reference CPU forward, fp32", "sample_images_per_step": n},
        "cpu_baseline": {"value": value, "unit": "img/s", "cores": threads, "kind": "port",
                         "sample": f"{n} images per step, fp32, torch CPU ops ({threads} threads), oracle/oracle_torch.py"},
        "e2e": {"value": value, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=RESULT_OUT, flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="GLOBAL batch (default: the config's, e.g. 1024 for c2)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: the global batch is sharded over the GPUs (default, BASELINE configs); "
                         "weak: every GPU takes the whole configured batch")
    ap.add_argument("--chunk", type=int, default=0,
                    help="images per H2D/compute pipeline chunk in the e2e leg (0 = the whole per-GPU batch)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="device-rate loop: replay the forward as one CUDA graph (graphs.GraphedForward). auto = when the "
                         "per-GPU batch is at most 256 images (the strong-scaled shards), where 64 stream launches "
                         "cost the GPU ~7 %% more than one graph launch")
    ap.add_argument("--prewarm", type=float, default=1.0,
                    help="seconds of untimed forwards before the W warm-up steps of the device-rate leg: short strong-"
                         "scaled runs (20 steps x 4.5 ms at 128 images per GPU) would otherwise be timed at the boost "
                         "clocks of a cold GPU while the legs after them run power-capped")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output of the last one as DIR/embeddings.npy (float32; "
                         "DIR/embeddings_rank<r>.npy per rank under torchrun) to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference_arm(args, cfg)
        return

    import torch.distributed as dist

    import pytorch_models_b200 as pm
    from pytorch_models_b200 import ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own banner / debug lines go to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    steps, warmup = args.steps, max(args.warmup, 3)
    global_cfg = args.batch or cfg["batch"]
    if args.scaling == "strong":
        if global_cfg % world:
            raise SystemExit(f"global batch {global_cfg} is not divisible by {world} GPUs")
        B = global_cfg // world
    else:
        B = global_cfg

    torch.manual_seed(0)
    model = cfg["make"](pm).eval()
    synthetic_weights_(model, 100)
    model = model.to(dev).bfloat16()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    use_graph = args.graph == "on" or (args.graph == "auto" and B <= 256)

    def device_rate(batch: int, n_steps: int, seed: int, sample_clocks: bool):
        """K forwards over a device-resident batch, CUDA events on the launching stream, barrier + synchronize on both
        sides, max over ranks. Returns (ms per step, launches, clocks, last output, the batch)."""
        torch.manual_seed(seed + rank)
        xd = torch.randn(batch, *cfg["shape"], device=dev).bfloat16()
        fwd = model
        if use_graph and batch == B:
            from pytorch_models_b200.graphs import GraphedForward

            fwd = GraphedForward(model, xd)  # public API: y = g(x) copies x in, replays, returns a copy of the output
        with torch.no_grad():
            t_pre = time.perf_counter()
            while sample_clocks and time.perf_counter() - t_pre < args.prewarm:  # reach the sustained clock regime
                for _ in range(4):
                    fwd(xd)
                torch.cuda.synchronize()
            sampler = ClockSampler(local) if (rank == 0 and sample_clocks) else None
            for _ in range(warmup):
                out = fwd(xd)
            barrier()
            l0 = ops.LAUNCHES
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_host0 = time.perf_counter()
            e0.record()
            for _ in range(n_steps):
                out = fwd(xd)
            e1.record()
            barrier()
            t_host1 = time.perf_counter()
            ms = max_over_ranks(e0.elapsed_time(e1)) / n_steps
            return ms, ops.LAUNCHES - l0, (sampler.stop(t_host0, t_host1) if sampler else None), out, xd

    # ---- device-resident throughput ("value")
    if os.environ.get("B200_PROFILE_STEP"):
        # ncu --profile-from-start off: capture exactly one warmed-up forward (scripts/gpu_ncu.sh)
        torch.manual_seed(1 + rank)
        xp = torch.randn(B, *cfg["shape"], device=dev).bfloat16()
        with torch.no_grad():
            for _ in range(warmup):
                model(xp)
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            model(xp)
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        del xp
    ms_step, launches, clocks, y, x_dev = device_rate(B, steps, 1, True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, y, rank, world)
    launches_per_step = launches // steps
    value = world * B / (ms_step * 1e-3)

    # ---- the same loop with CUDA events around EVERY launch of EVERY timed step (launching stream), bracketed as a
    # whole as well: the per-kernel sums must add up to the instrumented step, and the instrumented step must be close
    # to the plain one — otherwise the roofline below would describe a different regime than `value`.
    prof = None
    if rank == 0 or world > 1:
        with torch.no_grad():
            for _ in range(2):
                model(x_dev)
            barrier()
            rec = ops.profile(True)
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record()
            for _ in range(steps):
                model(x_dev)
            p1.record()
            torch.cuda.synchronize()
            ops.profile(False)
            barrier()
        if rank == 0:
            prof = dict(rec=rec, ms_step=p0.elapsed_time(p1) / steps)

    # ---- end to end: pinned host images -> H2D -> forward -> D2H embeddings, chunks pipelined over two streams
    def e2e_leg(host_dtype: torch.dtype) -> dict:
        chunk = min(args.chunk, B) if args.chunk > 0 else B
        n_chunks = (B + chunk - 1) // chunk
        torch.manual_seed(1 + rank)
        x_host = torch.randn(B, *cfg["shape"]).to(host_dtype).pin_memory()
        copy_stream, comp_stream = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        out_host = torch.empty(B, *y.shape[1:], dtype=torch.bfloat16).pin_memory()
        stage = [torch.empty(chunk, *cfg["shape"], device=dev, dtype=host_dtype) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]
        h2d_ev: list = []
        issued = [0]  # chunks issued so far: the two staging buffers alternate across step boundaries as well
        fwd = model
        if use_graph and B % chunk == 0:
            # the same public call as the device-rate leg at this shard size: y = g(x) copies the staged chunk into the
            # graph's input, replays the captured forward and returns a copy of its output
            from pytorch_models_b200.graphs import GraphedForward

            fwd = GraphedForward(model, stage[0])

        def step(timed: bool):
            for ci in range(n_chunks):
                lo, hi = ci * chunk, min(B, (ci + 1) * chunk)
                s = issued[0] % 2
                issued[0] += 1
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(freed[s])
                    if timed:
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record(copy_stream)
                    stage[s][: hi - lo].copy_(x_host[lo:hi], non_blocking=True)
                    if timed:
                        b.record(copy_stream)
                        h2d_ev.append((a, b))
                    ready[s].record(copy_stream)
                with torch.cuda.stream(comp_stream):
                    comp_stream.wait_event(ready[s])
                    out = fwd(stage[s][: hi - lo])  # fp32 images are converted inside the patch-embedding kernel
                    freed[s].record(comp_stream)
                    out_host[lo:hi].copy_(out, non_blocking=True)

        with torch.no_grad():
            for s in range(2):
                freed[s].record(comp_stream)
            for _ in range(warmup):
                step(False)
            barrier()
            t0 = torch.cuda.Event(enable_timing=True)
            t1 = torch.cuda.Event(enable_timing=True)
            t0.record(copy_stream)
            comp_stream.wait_event(t0)
            for _ in range(steps):
                step(True)
            copy_stream.wait_stream(comp_stream)
            t1.record(copy_stream)
            barrier()
            ms = max_over_ranks(t0.elapsed_time(t1)) / steps
        h2d_ms = sum(a.elapsed_time(b) for a, b in h2d_ev) / steps
        nbytes = x_host.numel() * x_host.element_size()
        return {"value": world * B / (ms * 1e-3), "unit": "img/s", "ms_per_step": ms,
                "host_dtype": str(host_dtype).replace("torch.", ""),
                "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": out_host.numel() * out_host.element_size(),
                "h2d_ms_per_step": h2d_ms, "h2d_gbs": nbytes / (h2d_ms * 1e-3) / 1e9 if h2d_ms > 0 else None,
                "frac_of_device_rate": (world * B / (ms * 1e-3)) / value,
                "launch": "CUDA-graph replay (graphs.GraphedForward)" if fwd is not model else "launch plan",
                "pipeline": f"{n_chunks} chunk(s) of {chunk} images per step on two staging buffers: the H2D copy of a "
                            "chunk overlaps the forward of the previous one (also across step boundaries); pinned "
                            f"buffers first-touched on NUMA node {numa.get('numa_node')}"}

    e2e = e2e_f32 = None
    if not args.no_e2e:
        e2e = e2e_leg(torch.bfloat16)
        e2e_f32 = e2e_leg(torch.float32)  # what the reference's callers hold (tests/image/test_vit.py:11)
        if os.environ.get("B200_BENCH_E2E_REPEAT"):  # experiment: does the order of the legs matter?
            again = e2e_leg(torch.bfloat16)
            if rank == 0:
                print(f"[e2e repeat] bf16 first {e2e['ms_per_step']:.3f} ms, fp32 {e2e_f32['ms_per_step']:.3f} ms, "
                      f"bf16 again {again['ms_per_step']:.3f} ms", file=sys.stderr, flush=True)

    # ---- N > 1: the optional NCCL all-gather of the embeddings, once, outside every timed region, checked bit for bit
    # against the same global batch run on one GPU (no cross-rank arithmetic exists, so it must be exact; SURVEY §8(e))
    gather_check = None
    if world > 1:
        from pytorch_models_b200.sharding import gather_embeddings, shard_batch

        n_chk = min(global_cfg, 8 * world)
        torch.manual_seed(12345)  # the same global batch on every rank
        xg = torch.randn(n_chk, *cfg["shape"]).bfloat16().to(dev)
        with torch.no_grad():
            mine = model(shard_batch(xg, rank, world))
            t0g = time.perf_counter()
            gathered = gather_embeddings(mine, total=n_chk)
            torch.cuda.synchronize()
            t_gather = time.perf_counter() - t0g
            whole = model(xg)
        same = torch.tensor([int(torch.equal(gathered, whole))], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        gather_check = {"backend": dist.get_backend(), "samples": n_chk, "bit_identical_on_all_ranks": bool(same.item()),
                        "bytes_per_rank": mine.numel() * mine.element_size(), "wall_ms_incl_launch": t_gather * 1e3}
        del xg

    # ---- weak-scaled companion figure (N > 1, strong run): every GPU takes the whole configured batch
    weak = None
    if world > 1 and args.scaling == "strong":
        del x_dev
        w_ms, _, _, _, xw = device_rate(global_cfg, max(3, steps // 2), 11, False)
        del xw
        weak = {"value": world * global_cfg / (w_ms * 1e-3), "unit": "img/s", "ms_per_step": w_ms,
                "per_gpu_batch": global_cfg, "global_batch": global_cfg * world, "steps": max(3, steps // 2)}

    # ---- rooflines from the in-region per-launch events
    roofline = roofline_attention = roofline_rows = None
    peaks = measured_peaks()
    if rank == 0 and prof is not None:
        by_kernel: dict[str, list[float]] = {}
        by_shape: dict[str, list[float]] = {}
        gemm_ms = gemm_flops = att_ms = att_flops = att_bytes = rows_ms = rows_bytes = 0.0
        att_n = rows_n = 0
        for name, meta, a, b in prof["rec"]:
            ms = a.elapsed_time(b)
            acc = by_kernel.setdefault(name, [0.0, 0])
            acc[0] += ms
            acc[1] += 1
            if name == "b200enc_linear":
                fl = 2.0 * meta["batches"] * meta["M"] * meta["N"] * meta["K"]
                gemm_ms += ms
                gemm_flops += fl
                key = f"N{meta['N']}_K{meta['K']}" + ("_ln" if meta["fold"] else "") + ("_gelu" if meta["gelu"] else "") + ("_res" if meta["res"] else "")
                sh = by_shape.setdefault(key, [0.0, 0.0, 0])
                sh[0] += ms
                sh[1] += fl
                sh[2] += 1
            elif name.startswith("b200enc_attention"):
                att_ms += ms
                att_n += 1
                att_flops += 4.0 * meta["B"] * meta["H"] * meta["Lq"] * meta["Lkv"] * 64
                att_bytes += 2.0 * meta["B"] * meta["H"] * 64 * (2 * meta["Lq"] + 2 * meta["Lkv"])  # q, out, k, v
            elif name in ("b200enc_layernorm", "b200enc_row_stats", "b200enc_patch_rows", "b200enc_mean_tokens"):
                rows_ms += ms
                rows_n += 1
                if name == "b200enc_layernorm":
                    rows_bytes += 4.0 * meta["rows"] * meta["d"]
                elif name == "b200enc_row_stats":
                    rows_bytes += 2.0 * meta["rows"] * meta["d"]
                elif name == "b200enc_mean_tokens":
                    rows_bytes += 2.0 * meta["B"] * (meta["L"] + 1) * meta["d"]
                else:
                    rows_bytes += meta["B"] * 3.0 * meta["H"] * meta["W"] * (4 if meta["f32"] else 2) + \
                        2.0 * meta["B"] * (meta["H"] // meta["p"]) * (meta["W"] // meta["p"]) * meta["kpad"]
        sum_ms = sum(v[0] for v in by_kernel.values()) / steps
        traffic = committed_traffic(args.config, B)
        n_gemm = by_kernel.get("b200enc_linear", [0.0, 0])[1]
        achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms else 0.0
        roofline = {
            "kernel": "gemm_bf16_kernel (b200enc_linear: QKV / out_proj / FC1 / FC2 / patch embed)",
            "bound": "tensor", "achieved": achieved, "peak": peaks["sustained"], "unit": "TFLOP/s",
            "frac": achieved / peaks["sustained"], "peak_source": f"{peaks['source']} (sustained cuBLAS bf16; burst {peaks['burst']})",
            "frac_of_burst": achieved / peaks["burst"],
            "traffic": None if traffic is None else traffic.get("gemm_mean_bytes_per_launch"),
            "traffic_source": None if traffic is None else traffic.get("source"),
            "timing": f"CUDA events around every launch of all {steps} timed steps of a second pass of the same loop "
                      "(launching stream, same buffers, sustained clocks)",
            "launches_per_step": n_gemm // steps, "avg_launch_ms": gemm_ms / max(n_gemm, 1),
            "share_of_step": gemm_ms / steps / prof["ms_step"],
            "by_shape": {k: {"launches_per_step": v[2] // steps, "avg_ms": round(v[0] / v[2], 4),
                             "tflops": round(v[1] / v[0] * 1e-9, 1)} for k, v in by_shape.items()},
            "step_breakdown_ms": {k: round(v[0] / steps, 3) for k, v in sorted(by_kernel.items(), key=lambda kv: -kv[1][0])},
            # consistency of the evidence: per-launch sums vs the bracketed instrumented loop vs the plain timed loop
            "sum_of_launches_ms_per_step": sum_ms, "instrumented_ms_per_step": prof["ms_step"],
            "launch_sum_over_instrumented_step": sum_ms / prof["ms_step"],
            "instrumented_over_plain_step": prof["ms_step"] / ms_step,
        }
        if att_n:
            hbm_bound = cfg["L"] <= 256  # SURVEY §8(d): attention is HBM-bound at L=197 (AI 98 F/B), tensor-bound for L >= 576
            a_tf = att_flops / (att_ms * 1e-3) / 1e12
            a_gb = att_bytes / (att_ms * 1e-3) / 1e9
            roofline_attention = {
                "kernel": "attention_kernel (b200enc_attention)", "bound": "hbm" if hbm_bound else "tensor",
                "achieved": a_gb if hbm_bound else a_tf, "peak": peaks["hbm"] if hbm_bound else peaks["sustained"],
                "unit": "GB/s" if hbm_bound else "TFLOP/s",
                "frac": (a_gb / peaks["hbm"]) if hbm_bound else (a_tf / peaks["sustained"]),
                "algorithmic": "bytes = 8*L*d per sample-layer (q, k, v, out); flops = 4*L^2*d",
                "tflops": a_tf, "gbs": a_gb, "launches_per_step": att_n // steps, "avg_launch_ms": att_ms / att_n,
                "share_of_step": att_ms / steps / prof["ms_step"],
                "traffic": None if traffic is None else traffic.get("attention_bytes_per_launch"),
            }
        if rows_n:
            r_gb = rows_bytes / (rows_ms * 1e-3) / 1e9
            roofline_rows = {"kernel": "row kernels (layernorm / row_stats / patch_rows / mean_tokens)", "bound": "hbm",
                             "achieved": r_gb, "peak": peaks["hbm"], "unit": "GB/s", "frac": r_gb / peaks["hbm"],
                             "launches_per_step": rows_n // steps, "ms_per_step": rows_ms / steps,
                             "share_of_step": rows_ms / steps / prof["ms_step"]}

    # ---- CPU baseline (rank 0, N = 1 only): the oracle port of the reference's CPU forward on a bounded sample
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        try:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))  # the CPU arm may use every host core
        except OSError:
            pass
        dt, n, threads = time_cpu(cfg, args.config, steps=2, warmup=1)
        cpu_baseline = {"value": n / dt, "unit": "img/s", "cores": threads, "kind": "port",
                        "sample": f"{n} images x 2 timed passes, fp32, torch CPU ops, oracle/oracle_torch.py"}

    if rank == 0:
        fl = flops_per_sample(cfg)
        line = {
            "metric": "ViT-B/16 img/s bf16" if args.config == "c2" else f"{args.config} samples/s bf16",
            "value": value, "unit": "img/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": cfg["desc"], "per_gpu_batch": B, "global_batch": B * world,
                       "parallelism": f"dp{world} (batch-sharded, no collective)", "weights": "random-init, seed 0",
                       "launch": ("one CUDA-graph replay per forward (graphs.GraphedForward; the per-launch profile "
                                  "uses single calls)") if use_graph else
                                 "launch plan: one b200enc_run_ops call per forward (plans.py)",
                       "l2": "inputs+activations per step >> 126 MB L2 (no flush needed)" if B >= 64 else
                             "per-step activations may fit the 126 MB L2 at this batch",
                       "prewarm": f"{args.prewarm:g} s of untimed forwards before the {warmup} warm-up steps (sustained clocks)",
                       "numa": numa},
            "tokens_per_s": value * cfg["L"],
            "model_tflops": value * fl / 1e12, "model_frac_of_burst_peak": value * fl / 1e12 / world / peaks["burst"],
            "model_frac_of_sustained_peak": value * fl / 1e12 / world / peaks["sustained"],
            "e2e": e2e, "e2e_fp32_host": e2e_f32, "weak_scaling": weak, "gather_check": gather_check,
            "gpu_launches": launches,
            "gpu_launches_per_step": launches_per_step, "clocks": clocks,
            "roofline": roofline, "roofline_attention": roofline_attention, "roofline_rows": roofline_rows,
            "cpu_baseline": cpu_baseline,
        }
        print(json.dumps(line), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    # stdout carries exactly ONE JSON line: everything else that might write to file descriptor 1 (NCCL's version
    # banner, library printf) is sent to stderr for the duration of the run
    sys.stdout.flush()
    RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    main()
