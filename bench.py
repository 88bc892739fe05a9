#!/usr/bin/env python
"""bench.py — images/sec of the full TokenHMR forward (BASELINE.json metric) on N B200s of one box.

    python bench.py --gpus 1 --steps 20 --warmup 5              # our engine (default)
    torchrun --nproc-per-node N ... bench.py --gpus N ...        # one rank per GPU, weak scaling (64 images / rank)
    python bench.py --impl reference --steps 3 --warmup 1       # reference arm: CPU fp32 forward on the host cores
    python bench.py --steps 20 --dump-outputs DIR                # also write the last timed step's outputs to DIR

A "step" is one forward of the path over one synthetic batch: configs[1] of BASELINE.json
(bs=64 synthetic 256x256 inputs cropped to 256x192, ViT-H/16 + token decoder + SMPL, fp16 operands / fp32
accumulate), random-init weights of the release architecture (no checkpoints exist offline).

JSON line (rank 0):  value = whole-job images/s with the batch already resident in HBM (CUDA-graph replay of
the engine forward; on N > 1 GPUs the per-step NCCL all-gather of the outputs is inside the timed region),
e2e = the same through the public API TokenHMREngine.forward(batch) with pinned HOST input (H2D inside) and a
D2H read-back of the results a caller consumes, roofline = live per-kernel-family accounting from the engine's
timed replay, cpu_baseline = the oracle (CPU restatement of the reference) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "images/sec (256x192) at bs=64 per GPU, full TokenHMR forward"
FLOP_PER_IMAGE = 252.10e9   # BASELINE.md §2
PER_GPU_BATCH = 64


def _profile_json(stem: str):
    """Newest committed profiles/r<N>_<stem>.json (None when absent)."""
    cands = sorted((ROOT / "profiles").glob(f"r*_{stem}.json"))
    return cands[-1] if cands else None


def _profile_json_load(stem: str):
    p = _profile_json(stem)
    try:
        return json.loads(p.read_text()) if p else None
    except Exception:
        return None


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel (dram__bytes_read.sum + dram__bytes_write.sum of one
    `ncu --set full` capture, scripts/make_profiles.sh -> profiles/r<N>_traffic.json); None when no capture is committed."""
    p = _profile_json("traffic")
    try:
        d = json.loads(p.read_text())
        return {"bytes_per_launch": d["dram_bytes_per_launch"], "algorithmic_bytes_per_launch": d["algorithmic_bytes_per_launch"],
                "kernel": d["kernel"], "source": str(p.relative_to(ROOT))}
    except Exception:
        return None


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.time()] + [c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()

    def stats(self, t0: float, t1: float) -> dict:
        """Median SM clock and the throttle reasons seen between wall-clock t0 and t1 (+ one sampling period)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        rows = [r[1:] for r in list(self.rows) if t0 <= r[0] <= t1 + 0.15]
        sm = sorted(float(r[1]) for r in rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = max([float(r[2]) for r in rows if len(r) >= 8 and r[2].replace(".", "").isdigit()] or [0.0])
        reasons = set()
        for r in rows:
            if len(r) < 8:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # (power.draw is a ~1 s moving average: meaningless over a 0.4 s window; scripts/dev_sustained.py reads it over 2 s runs)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------
def pick_cpu_threads(sd, smpl, cfg) -> int:
    """128 torch threads on 1.5 k-row GEMMs is slower than 32 (oversubscription): time one ViT-block-sized
    matmul at a few thread counts and keep the fastest, so the CPU baseline is the best the host can do."""
    import torch
    ncpu = os.cpu_count() or 1
    x = torch.randn(4 * 192, 1280)
    w = sd["backbone.blocks.0.mlp.fc1.weight"]
    best, best_t = ncpu, None
    for n in sorted({min(ncpu, c) for c in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(n)
        torch.nn.functional.linear(x, w)
        t = time.perf_counter()
        for _ in range(5):
            torch.nn.functional.linear(x, w)
        dt = time.perf_counter() - t
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    return best


def cpu_forward_rate(budget_s: float = 15.0):
    """The oracle (fp32 CPU restatement of the reference forward) timed on the host cores.  Host speed differs by more
    than an order of magnitude between boxes, so the sample is sized from a 4-image probe to ~`budget_s` seconds of CPU
    work (4..64 of the 64 images)."""
    import torch
    from oracle import tokenhmr_oracle as O
    from tokenhmr_b200 import synth
    from tokenhmr_b200.config import release_config
    cfg = release_config()
    sd, smpl = synth.make_state_dict(cfg), synth.make_smpl(cfg)
    threads = pick_cpu_threads(sd, smpl, cfg)
    torch.set_num_threads(threads)
    with torch.no_grad():
        probe = synth.make_images(4, cfg)
        t = time.perf_counter()
        O.forward(sd, smpl, probe, cfg)
        t4 = time.perf_counter() - t
        n = max(4, min(64, int(budget_s / t4 * 4) // 4 * 4))
        img = synth.make_images(n, cfg)
        t = time.perf_counter()
        O.forward(sd, smpl, img, cfg)
        dt = time.perf_counter() - t
    return n / dt, n, dt, threads


WORKLOAD = "bs=64 synthetic 256x256 -> 256x192, full TokenHMR forward (ViT-H/16 + token decoder + SMPL)"


def workload_config(world: int) -> dict:
    """`config` of the JSON line: identical for both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "per_gpu_batch": PER_GPU_BATCH, "global_batch": world * PER_GPU_BATCH,
            "parallelism": f"dp{world} + 1 all-gather of outputs", "weights": "random-init release architecture (seed 1234)",
            "l2": "1.4 GB of fp16 weights + 0.6 GB of activations stream through the 126 MB L2 every step (inputs larger "
                  "than L2, no flush needed)"}


def run_reference(args):
    """--impl reference: the reference's own CPU path.  /root/reference does not exist on the GPU box and the
    reference package cannot be installed offline (pytorch_lightning / smplx / yacs missing, DESIGN.md), so this
    times the oracle port, which is bit-identical to the reference modules (tests/test_oracle_pinned.py).  Each step
    is a bounded sample of the bs=64 batch (stated in cpu_baseline.sample), sized from a 4-image probe so that the whole
    --steps / --warmup run stays within a few minutes; the rate is per image."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import tokenhmr_oracle as O
    from tokenhmr_b200 import synth
    from tokenhmr_b200.config import release_config
    cfg = release_config()
    sd, smpl = synth.make_state_dict(cfg), synth.make_smpl(cfg)
    threads = pick_cpu_threads(sd, smpl, cfg)
    torch.set_num_threads(threads)
    with torch.no_grad():
        probe = synth.make_images(4, cfg)
        t = time.perf_counter()
        O.forward(sd, smpl, probe, cfg)
        t4 = time.perf_counter() - t
    budget_s = 240.0 / max(1, args.steps + args.warmup)          # whole run ~4 minutes
    sample = max(4, min(PER_GPU_BATCH, int(budget_s / t4 * 4) // 4 * 4))
    img = synth.make_images(sample, cfg)
    with torch.no_grad():
        for _ in range(args.warmup):
            O.forward(sd, smpl, img, cfg)
        t = time.perf_counter()
        for _ in range(args.steps):
            O.forward(sd, smpl, img, cfg)
        dt = time.perf_counter() - t
    value = sample * args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3 * PER_GPU_BATCH / sample,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} of the 64 images per step x {args.steps} steps (ms_per_step is scaled to 64 "
                                   f"images), fp32 eager torch, best of 8/16/32/64/all host threads ({os.cpu_count()} available)"},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


DUMP_MAX_BYTES = 64 << 20
DUMP_MAX_ELEMS_PER_ARRAY = 4 << 20


def clone_outputs(out: dict) -> dict:
    """Device copy of a forward's output dict (the aliased buffers are overwritten by later forwards)."""
    return {k: clone_outputs(v) if isinstance(v, dict) else v.clone() for k, v in out.items()}


def dump_outputs(out: dict, directory: str) -> list:
    """Writes every array of a forward's output dict as <directory>/<name>.npy in float32 (a nested dict's arrays as
    <outer>.<inner>.npy), within DUMP_MAX_BYTES in all.  An array larger than its share of the budget (at this workload
    only cls_logits_softmax: 64 x 160 x 2048) is written as a fixed sample of its flattened elements: the sorted indices
    drawn by numpy's default_rng(0), the same in every run, so that two builds compare element for element."""
    import numpy as np
    flat = {}

    def walk(prefix, d):
        for k, v in d.items():
            if isinstance(v, dict):
                walk(f"{prefix}{k}.", v)
            else:
                flat[prefix + k] = v.detach().float().cpu().numpy()

    walk("", out)
    os.makedirs(directory, exist_ok=True)
    left = (DUMP_MAX_BYTES - 4096 * len(flat)) // 4          # elements; 4 KB per file covers the .npy header
    written = []
    for i, (name, a) in enumerate(sorted(flat.items(), key=lambda kv: (kv[1].size, kv[0]))):
        share = min(DUMP_MAX_ELEMS_PER_ARRAY, left // (len(flat) - i))
        if a.size > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
            name += ".sample"
        np.save(os.path.join(directory, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))
        left -= a.size
        written.append(name)
    return written


# ---------------------------------------------------------------------------------------------------------
def cuda_time(fn, n=5, warm=2):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def standalone_configs(dev, peaks) -> dict:
    """BASELINE.json configs 1, 4 and 5 (1-based as SURVEY.md section 8d numbers them) under the same clock as the headline:
    CPU bs=1 forward (oracle port), VQ nearest-code arg-min 1 M x 2048 x 256, SMPL lbs() 4096 poses."""
    import torch
    from oracle import tokenhmr_oracle as O
    from tokenhmr_b200 import ops, synth
    from tokenhmr_b200.config import release_config
    cfg = release_config()
    out = {}
    # config 4: VQ arg-min (quantize_cnn.py:80-86); inputs larger than L2 (1 GB of queries)
    cb = torch.randn(2048, 256, device=dev, generator=torch.Generator(dev).manual_seed(1))
    x = torch.randn(1_000_000, 256, device=dev, generator=torch.Generator(dev).manual_seed(2))
    # two arithmetically equivalent schedules (csrc/vq.cuh): "exact" = one 3-product split-fp16 pass over every query;
    # "screened" = a 1-product pass that settles every row whose top-2 margin clears a rigorous error bound, then the exact
    # pass on the rest.  Both are timed; the library default is the first key of `modes`.
    prev = os.environ.get("THMR_VQ_SCREEN")
    modes, idx_by_mode = {}, {}
    for name, flag in (("screened", "1"), ("exact", "0")):
        os.environ["THMR_VQ_SCREEN"] = flag
        idx_by_mode[name] = ops.vq_quantize(x, cb)
        modes[name] = {"ms": cuda_time(lambda: ops.vq_quantize(x, cb))}
    if prev is None:
        os.environ.pop("THMR_VQ_SCREEN")
    else:
        os.environ["THMR_VQ_SCREEN"] = prev
    ms = cuda_time(lambda: ops.vq_quantize(x, cb))          # the library default
    pick = torch.randint(0, 2048, (100_000,), device=dev)
    near = cb[pick] + 0.05 * torch.randn(100_000, 256, device=dev)
    traffic = _profile_json("vq_traffic")
    out["vq_argmin_1M_x_2048_x_256"] = {
        "ms": ms, "queries_per_s": 1e6 / (ms * 1e-3), "algorithmic_tflops": 2 * 1e6 * 2048 * 256 / (ms * 1e-3) / 1e12,
        "modes": modes, "screened_equals_exact": bool(torch.equal(idx_by_mode["screened"], idx_by_mode["exact"])),
        "tensor_tflops_exact_mode_incl_3x_split": 3 * 2 * 1e6 * 2048 * 256 / (modes["exact"]["ms"] * 1e-3) / 1e12,
        "algorithmic_bytes": 1.034e9, "algorithmic_gbs": 1.034 / (ms * 1e-3),
        "dram_bytes_ncu": (json.loads(traffic.read_text()) if traffic else None),
        "exact_on_near_code_queries": bool(torch.equal(ops.vq_quantize(near, cb), pick)), "l2": "1 GB of queries > L2"}
    del x, near, idx_by_mode
    # config 5: LBS 4096 poses (smplx lbs as restated in oracle/smpl_oracle.py), pose2rot=True
    m = ops.SMPLModel(synth.make_smpl(cfg), dev)
    aa = 0.3 * torch.randn(4096, 24, 3, device=dev)
    be = torch.randn(4096, 10, device=dev)
    prev = os.environ.get("THMR_SKIN_THREADS")
    shapes = {}
    for t in ("256", "128"):
        os.environ["THMR_SKIN_THREADS"] = t
        shapes[f"skin_block_{t}"] = {"ms": cuda_time(lambda: m.lbs(be, aa))}
    if prev is None:
        os.environ.pop("THMR_SKIN_THREADS")
    else:
        os.environ["THMR_SKIN_THREADS"] = prev
    ms = cuda_time(lambda: m.lbs(be, aa))                   # the library default
    out["smpl_lbs_4096_poses"] = {"ms": ms, "launch_shapes": shapes, "poses_per_s": 4096 / (ms * 1e-3), "algorithmic_gbs": 4096 * 84.1e3 / (ms * 1e-3) / 1e9,
                                  "hbm_gbs_peak": peaks["hbm_gbs"], "frac_of_hbm": 4096 * 84.1e3 / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                  "l2": "344 MB of outputs > L2"}
    # config 1: the reference's CPU path at bs=1 (oracle port, all host threads the probe found best)
    sd, smpl = synth.make_state_dict(cfg), synth.make_smpl(cfg)
    threads = pick_cpu_threads(sd, smpl, cfg)
    torch.set_num_threads(threads)
    img1 = synth.make_images(1, cfg)
    with torch.no_grad():
        O.forward(sd, smpl, img1, cfg)
        ts = []
        for _ in range(3):
            t = time.perf_counter()
            O.forward(sd, smpl, img1, cfg)
            ts.append(time.perf_counter() - t)
    out["cpu_reference_bs1"] = {"ms": sorted(ts)[1] * 1e3, "images_per_s": 1.0 / sorted(ts)[1], "cores": threads,
                                "kind": "port", "runs": 3}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the standalone configs and the strict-mode rate")
    ap.add_argument("--streams", type=int, default=0, choices=[0, 1, 2, 3, 4],
                    help="1: consecutive steps replay on one stream; n > 1: round-robin on n streams (n steps in flight, single "
                         "GPU only); 0 (default): measure 1 and 4 at N=1 and report the faster as `value`")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last step of the path `value` was measured on "
                         "as DIR/<name>.npy (float32, at most 64 MB in all; see dump_outputs).  The one- and n-stream "
                         "engines sum in different orders and their outputs differ slightly; --streams fixes which one "
                         "is measured")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 engine's timed path")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from tokenhmr_b200 import synth
    from tokenhmr_b200.config import release_config
    from tokenhmr_b200.dist import ShardedTokenHMR
    from tokenhmr_b200.engine import TokenHMREngine, TokenHMRPipeline

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # a wedged collective must never eat the box's time limit: dump every thread's Python stack and exit
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("THMR_BENCH_WATCHDOG", "900")), exit=True)
    # NCCL_DEBUG is left alone: its log is the evidence for rank count and transport (the JSON line is printed last)
    if world > 1:
        # The process group only carries control traffic (the 128-byte NCCL unique id, shard sizes, barriers, the max over
        # ranks of the timings): gloo.  The data path is the library's own NCCL communicator (thmr_comm_create).
        backend = os.environ.get("THMR_BENCH_PG", "gloo")
        if backend == "nccl":
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
        else:
            dist.init_process_group("gloo")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    cfg = release_config()
    B = PER_GPU_BATCH
    sd, smpl = synth.make_state_dict(cfg), synth.make_smpl(cfg)
    model = TokenHMREngine(cfg, sd, smpl, device=dev, use_cuda_graph=True)
    sharded = ShardedTokenHMR(model) if world > 1 else None        # creates the library's own NCCL communicator
    spec = sharded.spec(B) if sharded else None
    img_host = synth.make_images(B, cfg, seed=rank).pin_memory()
    img_dev = img_host.to(dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev if dist.get_backend() == "nccl" else "cpu")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- (1) device-resident throughput: ONE CUDA-graph replay per step = forward (+ in-place all-gather when world > 1)
    def step_resident():
        return model.forward({"img": img_dev}, alias_outputs=True, shard=spec)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()            # started early: nvidia-smi needs ~0.5 s before its first sample
    for _ in range(args.warmup):
        step_resident()
    barrier()
    t_win0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out_last = step_resident()
    e1.record()
    barrier()
    t_win1 = time.time()
    last_outputs = {"serial": clone_outputs(out_last)} if args.dump_outputs and rank == 0 else None
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    ms_step = ms_total / args.steps
    value = world * B * 1e3 / ms_step
    serial = {"value": value, "ms_per_step": ms_step, "streams": 1, "window": (t_win0, t_win1)}

    # ---- (1b) the same K steps round-robin on n streams (single GPU): step i replays slot i%n's CUDA graph on stream i%n,
    # so whenever the kernel one step is running leaves SMs idle (the last wave of a persistent GEMM, the ~80 small launches
    # of the decoder / classifier / tokenizer-decoder / SMPL tail) the block scheduler fills them with another step's next
    # kernel.  Every step is still a complete bs=64 forward with its own buffers; the region is timed from an event all
    # streams wait for to an event that waits for all of them.  The engine is built with concurrent=True (no stream-K fc2:
    # its CTA pairs spin on each other and must own the GPU).  Measured (scripts/dev_streams.py): 1 / 2 / 3 / 4 streams =
    # 17.99 / 17.21 / 17.23 / 17.07 ms per step (17.72 for the default engine with stream-K on one stream).
    dual, model2 = None, None
    want_dual = world == 1 and args.streams != 1
    NS = args.streams if args.streams > 1 else 4
    if rank == 0:
        print(json.dumps({"early": "one-stream replay", "value": value, "ms_per_step": ms_step}), file=sys.stderr, flush=True)
    if want_dual:
        model2 = TokenHMREngine(cfg, sd, smpl, device=dev, use_cuda_graph=True, concurrent=True, max_cached_shapes=8)
        s2 = [torch.cuda.Stream(dev) for _ in range(NS)]
        last = [None] * NS

        def step_dual(i):
            with torch.cuda.stream(s2[i % NS]):
                last[i % NS] = model2.forward({"img": img_dev}, alias_outputs=True, slot=i % NS)

        for i in range(max(args.warmup, 2 * NS)):
            step_dual(i)
        torch.cuda.synchronize()
        ref_v = step_resident()["pred_vertices"]
        torch.cuda.synchronize()
        dev_max = max(float((last[s]["pred_vertices"] - ref_v).abs().max()) for s in range(NS))
        main = torch.cuda.current_stream()
        t_d0 = time.time()
        e0.record(main)
        for s in s2:
            s.wait_event(e0)
        for i in range(args.steps):
            step_dual(i)
        for s in s2:
            ev = torch.cuda.Event()
            ev.record(s)
            main.wait_event(ev)
        e1.record(main)
        torch.cuda.synchronize()
        t_d1 = time.time()
        if last_outputs is not None:
            last_outputs["dual"] = clone_outputs(last[(args.steps - 1) % NS])
        ms_dual = e0.elapsed_time(e1) / args.steps
        dual = {"value": B * 1e3 / ms_dual, "ms_per_step": ms_dual, "streams": NS, "window": (t_d0, t_d1),
                "max_abs_vertex_diff_vs_serial": dev_max,
                "what": f"step i replays slot i%{NS}'s graph on stream i%{NS} (TokenHMREngine(concurrent=True)); "
                        "ms_per_step = region / K (the latency of one step is about n times that)"}
        if rank == 0:
            print(json.dumps({"early": f"{NS}-stream replay", "value": dual["value"], "ms_per_step": ms_dual,
                              "max_abs_vertex_diff_vs_serial": dev_max}), file=sys.stderr, flush=True)
    head = dual if (dual is not None and (args.streams > 1 or dual["value"] > serial["value"])) else serial
    value, ms_step_head = head["value"], head["ms_per_step"]
    if last_outputs is not None:
        names = dump_outputs(last_outputs["dual" if head is dual else "serial"], args.dump_outputs)
        print(json.dumps({"dumped": names, "dir": args.dump_outputs, "steps_in_flight": head["streams"]}), file=sys.stderr,
              flush=True)
        del last_outputs
    clocks = None
    if rank == 0:
        time.sleep(0.12)
        sampler.stop()
        clocks = sampler.stats(*head["window"])
        for d in (serial, dual):
            if d is not None:
                d["clocks"] = sampler.stats(*d.pop("window"))

    # ---- (2) end to end through the public API: pinned host input -> H2D -> forward -> D2H of the results.
    # TokenHMRPipeline (the streaming driver a dataloader loop uses, engine.py) double-buffers the device-side
    # input / output slots: the H2D of batch i+1 overlaps the forward of batch i.  Every step still copies its own
    # 50 MB input from pinned host memory and reads its own results back; the region is timed from an event in front
    # of the first H2D (copy stream) to one behind the last D2H (compute stream).  On N > 1 GPUs every rank reads back
    # its OWN 64 images (the ranks of one host hand their shards to the same consumer; the gathered buffers stay on
    # the device for device-side consumers such as the GPU Evaluator).
    consumed = ["pred_vertices", "pred_keypoints_3d", "pred_cam", "pred_cam_t"]   # demo.py:80-118, pose_utils.py:217-239
    rows = slice(rank * spec.rows, rank * spec.rows + B) if spec else None
    pipe = TokenHMRPipeline(model, depth=2, read_back=consumed, shard=spec, read_rows=rows)

    def run_e2e(n):
        """n batches through the pipeline, pipe.depth of them in flight; every batch's results are waited for on the host."""
        tickets, done, out = [], 0, None
        for _ in range(n):
            tickets.append(pipe.submit({"img": img_host}))
            if len(tickets) - done >= pipe.depth:
                out = pipe.result(tickets[done])
                done += 1
        while done < len(tickets):
            out = pipe.result(tickets[done])
            done += 1
        return out

    run_e2e(4)                       # builds both slots (plans, graphs, pinned result buffers)
    barrier()
    e0.record(pipe.copy_stream)
    host_out = run_e2e(args.steps)
    e1.record(pipe.join())
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    e2e_value = world * B * 1e3 / ms_e2e
    e2e_modes = {"streams_1": {"value": e2e_value, "ms_per_step": ms_e2e}}
    e2e_streams = 1
    if want_dual:
        pipe1, pipe = pipe, TokenHMRPipeline(model2, depth=NS, read_back=consumed, streams=NS)
        run_e2e(2 * NS)
        torch.cuda.synchronize()
        e0.record(pipe.copy_stream)
        host_out2 = run_e2e(args.steps)
        e1.record(pipe.join())
        torch.cuda.synchronize()
        ms2 = e0.elapsed_time(e1) / args.steps
        e2e_modes["streams_n"] = {"value": B * 1e3 / ms2, "ms_per_step": ms2, "streams": NS, "depth": NS,
                                  "max_abs_vertex_diff_vs_streams_1": float((host_out2["pred_vertices"] - host_out["pred_vertices"]).abs().max())}
        if args.streams > 1 or B * 1e3 / ms2 > e2e_value:
            e2e_value, ms_e2e, e2e_streams = B * 1e3 / ms2, ms2, NS
        del pipe1
    h2d = img_host.numel() * 4
    d2h = sum(v.numel() * 4 for v in host_out.values())

    # ---- (3) live per-kernel-family accounting (rank 0): timed eager replay of the same forward
    roofline, families, families_ev, attention = None, None, None, None
    peaks = measured_peaks()
    if rank == 0:
        def aggregate(rows_list):
            agg = {}
            for rows in rows_list:
                for name, ms, fl, by in rows:
                    a = agg.setdefault(name, [0.0, 0.0, 0.0, 0])
                    a[0] += ms; a[1] += fl; a[2] += by; a[3] += 1
            n = len(rows_list)
            tot = sum(a[0] for a in agg.values())
            fam = {k: {"ms_per_step": a[0] / n, "share": a[0] / tot, "launch_groups_per_step": a[3] // n,
                       "tflops": (a[1] / (a[0] * 1e-3) / 1e12) if a[1] and a[0] else None,
                       "gbs": (a[2] / (a[0] * 1e-3) / 1e9) if a[2] and a[0] else None} for k, a in agg.items()}
            return agg, fam, tot / n

        # (a) in-graph: every kernel stamps the GPU's nanosecond timer at its start inside the CUDA-graph replay (20
        #     back-to-back replays, stamps of the last one; 5 such samples).  Nothing sits between the launches, the
        #     entries sum to the replay time: this is the step the headline number measures.
        agg, families, sum_ms = aggregate([model.profile_in_graph(img_dev, replays=20) for _ in range(5)])
        # (b) cross-check, round-1 method: eager replay with a CUDA event between launch groups (each event drains the
        #     GPU front end: short kernels are inflated by ~5 us, the entries sum to more than the step)
        agg_ev, families_ev, sum_ev = aggregate([model.profile(img_dev) for _ in range(3)])

        def gemm_rate(a):
            g = [v for k, v in a.items() if k.endswith("_gemm")]
            ms, fl = sum(v[0] for v in g), sum(v[1] for v in g)
            return fl / (ms * 1e-3) / 1e12, ms
        achieved, g_ms = gemm_rate(agg)
        achieved_ev, _ = gemm_rate(agg_ev)
        roofline = {"kernel": "gemm_f16_tn_2cta_kernel / gemm_f16_tn_kernel (tcgen05, all ViT/decoder GEMM launches)",
                    "bound": "tensor", "achieved": achieved, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                    "frac": achieved / peaks["tf_sustained"],
                    "peak_source": peaks["source"] + " bf16 sustained (cuBLAS 8192^3 back to back; kernel timed inside a long step)",
                    "method": "in-graph start stamps (globaltimer) of every launch inside the CUDA-graph replay, 5 samples x "
                              "the last of 20 back-to-back replays (thmr_engine_forward_stamped)",
                    "share_of_step": g_ms / sum(a[0] for a in agg.values()),
                    "in_graph_sum_ms": sum_ms, "graph_ms_per_step": ms_step, "accounting_of": "the one-stream replay",
                    "achieved_event_separated": achieved_ev, "frac_event_separated": achieved_ev / peaks["tf_sustained"],
                    "event_separated_sum_ms": sum_ev, "traffic": ncu_traffic(),
                    "cublas_same_shapes": _profile_json_load("sustained_gemm"),
                    "whole_step_tflops_per_gpu": B * FLOP_PER_IMAGE / (ms_step * 1e-3) / 1e12}
        # the second half of BASELINE.json's metric: the fused ViT attention kernel
        a = agg["vit.attention"]
        us_layer = a[0] / a[3] * 1e3
        attention = {"kernel": "vit_attention3_kernel (S/P/O in TMEM, TS-mode PV)", "us_per_layer_in_step": us_layer,
                     "us_per_layer_event_separated": agg_ev["vit.attention"][0] / agg_ev["vit.attention"][3] * 1e3,
                     "tflops": a[1] / (a[0] * 1e-3) / 1e12, "hbm_gbs_algorithmic": a[2] / (a[0] * 1e-3) / 1e9,
                     "frac_of_hbm_peak": a[2] / (a[0] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                     "frac_of_tensor_burst": a[1] / (a[0] * 1e-3) / 1e12 / peaks["tf_burst"],
                     "ncu": _profile_json_load("attention")}

    # ---- (4) strict mode (fp32-grade split-fp16 contractions, DESIGN.md section 2) on the same batch, and the standalone configs
    strict, standalone = None, None
    if rank == 0 and world == 1 and not args.no_extras:
        del pipe
        model2 = None
        sm = TokenHMREngine(cfg, sd, smpl, device=dev, use_cuda_graph=True, strict=True)
        ms = cuda_time(lambda: sm.forward({"img": img_dev}, alias_outputs=True), n=5, warm=3)
        strict = {"value": B * 1e3 / ms, "unit": "images/s", "ms_per_step": ms, "launches_per_step": sm.num_launches(),
                  "what": "TokenHMREngine(strict=True): every contraction as a 3-product split-fp16 GEMM, fp32 activations, "
                          "fp32 CUDA-core attention; vertices within 1e-4 of the fp32 reference, identical pose tokens"}
        del sm
        torch.cuda.empty_cache()
        standalone = standalone_configs(dev, peaks)

    # ---- (5) CPU baseline (rank 0, N=1 only): oracle on a bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, n, dt, threads = cpu_forward_rate()
        cpu = {"value": v, "unit": "images/s", "cores": threads, "kind": "port",
               "sample": f"{n} of the 64 images, one fp32 eager-torch forward of the oracle ({dt:.1f} s, sized from a "
                         f"4-image probe), thread count picked from 8/16/32/64/{os.cpu_count()}"}

    launches = model.num_launches() + (1 if world > 1 else 0)
    line = None
    if rank == 0:
        line = json.dumps({
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step_head, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16 operands / f32 accumulate", "data": "synthetic",
            "config": workload_config(world),           # identical for both arms (the driver compares them)
            "steps_in_flight": head["streams"],         # streams the K timed steps were replayed on (see streams_1 / streams_n)
            "scaling_note": (None if world == 1 else
                             "every rank keeps ONE step in flight (the sharded forward carries its NCCL all-gather inside the CUDA "
                             "graph; the multi-stream mode is single-GPU only): the like-for-like single-GPU number is `streams_1` "
                             "of the N=1 line, not its `value` when that was measured with several steps in flight"),
            "streams_1": serial, "streams_n": dual,
            "e2e": {"value": e2e_value, "unit": "images/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "read_back": consumed, "streams": e2e_streams, "modes": e2e_modes,
                    "api": (f"TokenHMRPipeline.submit/result (depth {e2e_streams}, streams {e2e_streams}: {e2e_streams} batches in "
                            "flight, H2D / forward / D2H of different batches overlap)" if e2e_streams > 1 else
                            "TokenHMRPipeline.submit/result (depth 2: H2D of the next batch overlaps the forward)")
                           + ("; each rank reads back its own shard" if world > 1 else "")},
            "gpu_launches": args.steps * launches, "launches_per_step": launches,
            "exchange": (None if world == 1 else "thmr_allgather_outputs: 8 grouped in-place ncclAllGather (one NCCL kernel) "
                         "inside the forward's CUDA graph, library-owned communicator"),
            "clocks": clocks, "roofline": roofline, "attention": attention, "kernel_families": families,
            "kernel_families_event_separated": families_ev,
            "strict": strict, "standalone": standalone, "cpu_baseline": cpu,
        })
    # Teardown must not be able to lose the measurement: if it does not finish in 30 s, print the line and leave.
    def bail():
        if rank == 0:
            print(line, flush=True)
        os._exit(0)
    guard = threading.Timer(30.0, bail)
    guard.daemon = True
    guard.start()
    if world > 1:
        pipe = None
        sharded.close()              # releases the graphs that captured the communicator, then destroys it
        dist.barrier()
        dist.destroy_process_group()
    guard.cancel()
    faulthandler.cancel_dump_traceback_later()
    if rank == 0:
        if world > 1:
            time.sleep(1.0)          # let the other ranks' NCCL teardown messages drain: the JSON line stays last
        sys.stdout.flush()
        print(line, flush=True)
    if world > 1:
        sys.stderr.flush()
        os._exit(0)                  # skip libnccl's atexit chatter (NCCL_DEBUG=INFO): nothing may follow the JSON line


if __name__ == "__main__":
    main()
