#!/usr/bin/env python
"""bench.py - relevancy maps/s (BASELINE.json metric), one process per GPU.

    python bench.py --gpus 1 --steps 20 --warmup 3                  # our arm: CLIP ViT-B/32 (the headline, BASELINE config 2)
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1  # the reference's CPU PyTorch path (oracle port)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                      # N > 1: per-sample sharding + ONE all-gather per step
    python bench.py --workload detr_r50|lxmert|clip_l14_336         # one of the other BASELINE configs as the main line
    python bench.py --steps 5 --dump-outputs DIR                    # + the maps of the last timed step as DIR/<name>.npy

Headline workload: a "step" = one interpret() pass over one batch of 64 synthetic (image, text) pairs PER GPU (weak
scaling), all 12+12 blocks (start_layer = start_layer_text = 0: forward staging every A_l, dgrad-only backward staging
every dA_l, rule 5, rule 6), fp32, random-init weights.  `value` is timed on the device (CUDA events, inputs resident in
HBM, max over ranks); `e2e` is the same metric with host buffers in and host maps out (H2D / D2H inside the timed region).
The default run also measures BASELINE configs 3, 4, 5 (DETR-R50, LXMERT, CLIP ViT-L/14@336) with a few steps each and
reports them under `other_workloads` (per-GPU shares: 16 / 16 / 256 units, i.e. config 4 = 2 GPUs, config 5 = 8 GPUs).
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH_PER_GPU = 64
START_LAYER = 0          # all layers: the full rule (the reference API default -1 is reported as `default_mode`)
METRIC = "relevancy maps/sec for CLIP ViT-B/32 224^2"
UNIT = "maps/s"
WORKLOAD = "clip_vit_b32_224_interpret_all_layers_b64_per_gpu"
PROMPT_NOTE = "U{1..75} tokens + SOT/EOT, the same length multiset on every rank (dead rows after the EOT are skipped, results identical)"


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def csrc_hash() -> str:
    """Hash of the kernel sources: ties an ncu capture under profiles/ to the build it was taken on."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "transformer-mm-explainability_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            with open(os.path.join(d, f), "rb") as fh:
                h.update(fh.read())
    return h.hexdigest()[:16]


# the files a kernel family is compiled from: an ncu capture stays valid while THESE are unchanged
KERNEL_SOURCES = {
    "gemm_f16x3": ("gemm_f16x3.cu", "gemm_epilogue.cuh", "tcgen05_ptx.cuh", "gemm.cuh", "mmx_common.cuh"),
    "gemm_tf32x3": ("gemm_tcgen05.cu", "gemm_epilogue.cuh", "tcgen05_ptx.cuh", "gemm.cuh", "mmx_common.cuh"),
    "avg_heads": ("rules.cu", "mmx_common.cuh"),
}


def _code_only(text: str) -> str:
    """Source text without `//` comments, trailing blanks and empty lines (no string literal in csrc/ contains `//`)."""
    out = []
    for line in text.splitlines():
        line = line.split("//", 1)[0].rstrip()
        if line:
            out.append(line)
    return "\n".join(out)


def kernel_sources_hash(kernel_key: str, read=None) -> str:
    """Hash of the CODE (comments stripped) of the files a kernel family is compiled from.  `read(name) -> str` overrides
    the file reader (tests; hashing the files of another commit)."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "transformer-mm-explainability_b200", "csrc")
    for f in KERNEL_SOURCES.get(kernel_key, ()):
        if read is None:
            with open(os.path.join(d, f)) as fh:
                text = fh.read()
        else:
            text = read(f)
        h.update(_code_only(text).encode())
    return h.hexdigest()[:16]


def captured_traffic(kernel_key: str):
    """DRAM traffic per launch from the committed `ncu --set full` capture (profiles/traffic_r2.json, written by
    profiles/capture_traffic.py); None when there is no capture for this kernel."""
    p = os.path.join(ROOT, "profiles", "traffic_r2.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    rec = d.get(kernel_key)
    if not rec:
        return None, None
    rec = dict(rec)
    rec["capture_build"] = d.get("build")
    # valid for the running build when the kernel's own sources are the ones the capture was taken on
    rec["build_matches"] = (rec.get("sources_hash") == kernel_sources_hash(kernel_key)) if rec.get("sources_hash") \
        else d.get("build") == csrc_hash()
    return rec.get("dram_bytes"), rec


def workload_config(world: int, B: int, cfg) -> dict:
    """The `config` object of the JSON line - the SAME dict for our arm and for `--impl reference`."""
    return {"workload": WORKLOAD, "batch_per_gpu": B, "global_batch": B * world, "start_layer": START_LAYER,
            "start_layer_text": START_LAYER, "image": cfg.image_resolution, "context": cfg.context_length,
            "weights": "random-init (seed 0)", "prompt_lengths": PROMPT_NOTE,
            "parallelism": f"sample-sharded x{world}, 1 all-gather of maps",
            "l2": "no flush: per-step working set (1.2 GB weights + >2 GB staged activations) >> 126 MB L2"}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """`--dump-outputs`: every array as `out_dir/<name>.npy` in float32.  All arrays lead with the sample dimension; above
    DUMP_LIMIT_BYTES in all, the same seeded sample of samples (sorted indices) is kept from each."""
    import numpy as np
    arrays = {k: np.ascontiguousarray(v.detach().cpu().numpy() if hasattr(v, "detach") else v, dtype=np.float32)
              for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        n = min(a.shape[0] for a in arrays.values())
        keep = np.sort(np.random.default_rng(0).choice(n, max(1, n * DUMP_LIMIT_BYTES // total), replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_ev = index, [], threading.Event()

    def run(self):
        while not self._stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop_ev.wait(0.1)

    def stop(self):
        self._stop_ev.set()
        self.join(timeout=3)
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for n, v in zip(names, s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = int(float(self.samples[0][1])) if self.samples else None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(self.samples)}


# ======================================================================================================================
# reference arm: the reference's own CPU PyTorch path (oracle port; /root/reference does not exist on the GPU box)
# ======================================================================================================================
def pick_threads() -> int:
    """torch CPU kernels stop scaling (and on 100+ core hosts get much slower) with too many threads; give the
    reference its best thread count from a quick probe so the baseline is not handicapped."""
    import torch
    from oracle import clip_oracle as co
    cores = os.cpu_count() or 1
    cfg = co.VIT_B32
    sd = co.init_state_dict(cfg, seed=0)
    images, tokens = co.synthetic_inputs(cfg, 4, seed=1)
    best, best_t = cores, None
    for n in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16)}, reverse=True):
        torch.set_num_threads(n)
        co.clip_interpret(sd, cfg, images[:1], tokens[:1], -1, -1)          # warm the thread pool
        t0 = time.perf_counter()
        co.clip_interpret(sd, cfg, images, tokens, -1, -1)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    return best


def cpu_baseline_run(batch: int, reps: int, warm: int, threads: int, start_layer: int = START_LAYER, outputs=None):
    """The reference's own CPU PyTorch path, restated: per-block autograd.grad exactly like the notebook, the SAME
    synthetic batch rank 0 of our arm processes (seed 1234, shared length multiset).  Returns (maps_per_s, median s);
    the maps of the last step go into ``outputs`` when given."""
    import torch
    import mmx_b200
    from oracle import clip_oracle as co
    torch.set_num_threads(threads)
    cfg = co.VIT_B32
    sd = co.init_state_dict(cfg, seed=0)
    images, tokens = mmx_b200.clip_synthetic_inputs(cfg, BATCH_PER_GPU, seed=1234, length_seed=4321)
    images, tokens = images[:batch], tokens[:batch]
    ts = []
    for i in range(warm + reps):
        t0 = time.perf_counter()
        maps = co.clip_interpret(sd, cfg, images, tokens, start_layer, start_layer, per_layer_grad=True)
        if i >= warm:
            ts.append(time.perf_counter() - t0)
    if outputs is not None:
        outputs.update(R_text=maps[0], R_image=maps[1])
    ts.sort()
    med = ts[len(ts) // 2]
    return batch / med, med


def run_reference(args):
    rank = _env_int("RANK", 0)
    if rank != 0:
        return
    import mmx_b200
    threads = pick_threads()
    batch = BATCH_PER_GPU          # one step = the whole per-GPU batch of the workload, both arms the same config
    t_all0 = time.perf_counter()
    outputs = {}
    val, sec = cpu_baseline_run(batch, args.steps, max(0, args.warmup), threads, outputs=outputs)
    val_def, sec_def = cpu_baseline_run(batch, 2, 1, threads, start_layer=-1)
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(max(1, args.gpus), batch, mmx_b200.VIT_B32),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "host_cores": os.cpu_count(),
                         "sample": f"each step = the {batch} pairs rank 0 of the GPU arm processes (all layers), median of "
                                   f"{max(1, args.steps)} steps; ONE CPU process whatever --gpus says; oracle port of "
                                   "CLIP_explainability.ipynb:151-208 incl. its per-block autograd.grad; thread count = "
                                   "fastest of {all,64,32,16} in a quick probe"},
        "default_mode": {"start_layer": -1, "value": val_def, "unit": UNIT, "ms_per_step": sec_def * 1e3,
                         "note": "reference API default (last block of each tower only), 1 warm-up + median of 2 steps"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t_all0,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(out), flush=True)


# ======================================================================================================================
# our arm
# ======================================================================================================================
class Dist:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = _env_int("WORLD_SIZE", 1)
        self.rank = _env_int("RANK", 0)
        self.local = _env_int("LOCAL_RANK", 0)
        torch.cuda.set_device(self.local)
        self.dev = torch.device(f"cuda:{self.local}")
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather_floats(self, x: float):
        if self.world == 1:
            return [x]
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        out = self.torch.empty(self.world, device=self.dev, dtype=self.torch.float64)
        self.dist.all_gather_into_tensor(out, t)
        return [float(v) for v in out.tolist()]

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def timed_loop(D: Dist, step, finish, steps: int, warm: int, lib):
    """W untimed + EXACTLY `steps` timed steps between barriers; CUDA events on the launching stream.
    Returns (ms per step of THIS rank, launches)."""
    torch = D.torch
    for _ in range(warm):
        step()
    finish()
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = lib.mmx_launch_count()
    e0.record()
    for _ in range(steps):
        step()
    finish()
    e1.record()
    D.barrier()
    return e0.elapsed_time(e1) / steps, lib.mmx_launch_count() - l0


def bench_clip(D: Dist, cfg, B: int, steps: int, warm: int, max_batch: int, with_default: bool, with_check: bool, e2e_steps: int,
               outputs=None):
    """CLIP interpret() for B pairs per GPU: device-timed value, e2e through host buffers, per-rank times, the collective
    alone, and (N > 1) the bitwise sharded == single-GPU check.  The maps of the last timed step (all ranks' after the
    all-gather) go into ``outputs`` when given."""
    import mmx_b200
    from mmx_b200.distributed import gather_maps_packed, split_packed
    torch, dist = D.torch, D.dist
    world, rank, dev = D.world, D.rank, D.dev
    lib = mmx_b200.lib()
    sd = mmx_b200.clip_init_state_dict(cfg, seed=0)           # identical weights on every rank (replicated)
    eng = mmx_b200.ClipEngine(cfg, sd, max_batch=max_batch, device=dev)
    del sd
    # pixels / token ids differ per rank; the prompt LENGTHS are the same multiset on every rank, so that every rank has
    # the same amount of (ragged) text work and the max over ranks measures the machine, not the draw
    images, tokens = mmx_b200.clip_synthetic_inputs(cfg, B, seed=1234 + rank, length_seed=4321)
    images_pin, tokens_pin = images.pin_memory(), tokens.to(torch.int32).pin_memory()
    d_images, d_tokens = images.to(dev), tokens.to(dev)
    n_total = B * world
    ctx, sv = cfg.context_length, cfg.vision_tokens
    pending = []
    last = {}

    # The one collective of the path: ONE all-gather of the packed maps per step.  In stream order by default; with
    # MMX_BENCH_GATHER=async it overlaps the next step's forward - measured SLOWER at N = 2 (8.72 vs 7.95 ms per step): while
    # the NCCL kernel waits for its peer it holds SMs, and the persistent GEMMs (one CTA per SM, static tile assignment)
    # then run with a CTA missing.
    gather_async = os.environ.get("MMX_BENCH_GATHER", "sync") == "async"

    def step_fn(sl):
        def step():
            rt, ri = eng.interpret(d_images, d_tokens, sl, sl, validate=False)
            last["maps"] = rt, ri
            if world > 1:
                if gather_async:
                    pending.append(gather_maps_packed(rt, ri, n_total, async_op=True))
                    last["full"] = pending[-1][1]
                    while len(pending) > 2:
                        pending.pop(0)[0].wait()
                else:
                    last["full"] = gather_maps_packed(rt, ri, n_total, async_op=False)[1]
            return rt, ri
        return step

    def finish():
        while pending:
            pending.pop(0)[0].wait()

    sampler = ClockSampler(D.local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_rank, launches = timed_loop(D, step_fn(START_LAYER), finish, steps, warm, lib)
    clocks = sampler.stop() if sampler else None
    if outputs is not None:
        rt, ri = split_packed(last["full"], ctx, sv - 1) if world > 1 else last["maps"]
        outputs.update(R_text=rt.cpu(), R_image=ri.cpu())
    per_rank = D.gather_floats(ms_rank)
    ms_step = max(per_rank)
    res = {"ms_per_step": ms_step, "value": n_total / (ms_step * 1e-3), "launches": int(launches), "clocks": clocks,
           "per_rank_ms": per_rank, "engine_bytes": None}
    if with_default:
        ms_def, _ = timed_loop(D, step_fn(-1), finish, max(3, steps // 2), warm, lib)
        ms_def = D.max(ms_def)
        res["default_mode"] = {"start_layer": -1, "value": n_total / (ms_def * 1e-3), "unit": UNIT, "ms_per_step": ms_def,
                               "note": "reference API default (last block of each tower only)"}

    # ---- the collective alone (N > 1): ONE all_gather_into_tensor of the packed maps
    if world > 1:
        rt, ri = eng.interpret(d_images, d_tokens, START_LAYER, START_LAYER, validate=False)
        for _ in range(3):
            gather_maps_packed(rt, ri, n_total, async_op=False)
        D.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            gather_maps_packed(rt, ri, n_total, async_op=False)
        e1.record()
        D.barrier()
        res["collective"] = {"kind": "ncclAllGather (torch.distributed all_gather_into_tensor), R_text and R_image packed in one buffer",
                             "calls_per_step": 1, "bytes_per_rank": int((ctx * ctx + sv - 1) * 4 * B),
                             "ms_alone": D.max(e0.elapsed_time(e1) / 10),
                             "overlapped_with": "the next step's forward" if gather_async else None,
                             "order": "async, overlapped" if gather_async else "in stream order at the end of every step"}

    # ---- e2e: host buffers in, host maps out, copies inside the timed region
    if world == 1:
        out_pin = (torch.empty(B, ctx, ctx).pin_memory(), torch.empty(B, sv - 1).pin_memory())

        def e2e_step():
            eng.interpret_host(images_pin, tokens_pin, START_LAYER, START_LAYER, out=out_pin)
            return float(out_pin[1][0, 0])                     # read the result on the host
        d2h = out_pin[0].numel() * 4 + out_pin[1].numel() * 4
    else:
        out_pin = torch.empty(n_total, ctx * ctx + sv - 1).pin_memory()

        def e2e_step():
            di, dt = images_pin.to(dev, non_blocking=True), tokens_pin.to(dev, non_blocking=True)
            rt, ri = eng.interpret(di, dt, START_LAYER, START_LAYER, validate=False)
            _, full = gather_maps_packed(rt, ri, n_total, async_op=False)
            out_pin.copy_(full, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return float(out_pin[0, 0])
        d2h = out_pin.numel() * 4
    for _ in range(warm):
        e2e_step()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    D.barrier()
    e2e_s = D.max((time.perf_counter() - t0) / e2e_steps)
    res["e2e"] = {"value": n_total / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(images_pin.numel() * 4 + tokens_pin.numel() * 4),
                  "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_s * 1e3,
                  "path": "mmx_clip_interpret_host (pinned host buffers -> maps on the host)" if world == 1 else
                          "pinned H2D -> ClipEngine.interpret -> one all-gather -> D2H of all maps"}

    # ---- N > 1: the sharded result must equal the single-GPU result BITWISE (every rank recomputes the global batch)
    if world > 1 and with_check:
        rt, ri = eng.interpret(d_images, d_tokens, START_LAYER, START_LAYER, validate=False)
        _, full = gather_maps_packed(rt, ri, n_total, async_op=False)
        g_img = torch.empty((n_total,) + tuple(d_images.shape[1:]), device=dev)
        g_tok = torch.empty((n_total, ctx), device=dev, dtype=d_tokens.dtype)
        dist.all_gather_into_tensor(g_img, d_images)
        dist.all_gather_into_tensor(g_tok, d_tokens)
        ok = True
        for r in range(world):
            st, si = eng.interpret(g_img[r * B:(r + 1) * B], g_tok[r * B:(r + 1) * B], START_LAYER, START_LAYER, validate=False)
            ft, fi = split_packed(full[r * B:(r + 1) * B], ctx, sv - 1)
            same = torch.equal(st, ft) and torch.equal(si, fi)
            if not same:
                print(f"[rank {rank}] shard {r}: recomputed != gathered: text max|d| {(st - ft).abs().max().item():.3e} "
                      f"({int((st != ft).sum())} elements), image max|d| {(si - fi).abs().max().item():.3e} "
                      f"({int((si != fi).sum())} elements)", file=sys.stderr)
            ok = ok and same
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        res["sharded_equals_single"] = bool(flag.item())
        del g_img, g_tok
    return res, eng, (d_images, d_tokens)


def clip_roofline(D: Dist, eng, inputs, B: int, cfg, steps_serial: int = 3):
    """Roofline of the dominant kernel (the transformer GEMMs).  The two towers normally share the GPU on two streams, so
    per-launch event times overlap and their sum can exceed the step; here the engine is switched to ONE stream
    (mmx_clip_set_serial), where every launch has the GPU to itself: sum(GEMM time) <= step time by construction."""
    import mmx_b200
    torch = D.torch
    lib = mmx_b200.lib()
    d_images, d_tokens = inputs
    hbm_peak, tf_burst, tf_sust, peak_src = _peaks()
    backend = lib.mmx_get_gemm_backend()
    eng.set_serial(True)
    for _ in range(2):
        eng.interpret(d_images, d_tokens, START_LAYER, START_LAYER, validate=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps_serial):
        eng.interpret(d_images, d_tokens, START_LAYER, START_LAYER, validate=False)
    e1.record()
    torch.cuda.synchronize()
    serial_ms = e0.elapsed_time(e1) / steps_serial
    lib.mmx_profile_gemm(1)
    for _ in range(steps_serial):
        eng.interpret(d_images, d_tokens, START_LAYER, START_LAYER, validate=False)
    lib.mmx_profile_gemm(0)
    tms, tfl, nl = C.c_double(), C.c_double(), C.c_int()
    lib.mmx_profile_gemm_report(C.byref(tms), C.byref(tfl), C.byref(nl))
    eng.set_serial(False)
    gemm_ms = tms.value / steps_serial
    tflops = tfl.value / (tms.value * 1e-3) / 1e12 if tms.value > 0 else 0.0
    names = {0: "fp32 FFMA", 1: "tcgen05 3xTF32, 1 CTA/tile", 2: "tcgen05 fp16x3 (packed fp16 hi/lo weight planes, 3 kind::f16 passes)"}
    traffic, traffic_rec = captured_traffic("gemm_f16x3" if backend >= 2 else "gemm_tf32x3")
    ceiling = tf_sust / (3.0 if backend >= 2 else 6.0)
    return {"kernel": f"transformer GEMMs ({names.get(backend, '?')}, tile width 128/144/160 per launch)",
            "bound": "tensor", "achieved": tflops, "peak": tf_sust, "unit": "TFLOP/s", "frac": tflops / tf_sust,
            "traffic": traffic, "traffic_capture": traffic_rec,
            "peak_source": peak_src + " bf16 dense, sustained",
            "launches_per_step": nl.value // steps_serial, "gemm_ms_per_step": gemm_ms,
            "serial_step_ms": serial_ms, "gemm_share_of_serial_step": gemm_ms / serial_ms if serial_ms > 0 else None,
            "flops_per_step": tfl.value / steps_serial,
            "scheme_ceiling": {"tflops": ceiling, "frac_of_ceiling": tflops / ceiling,
                               "note": "fp32-faithful results (1e-4 parity after ~100 chained GEMMs) need 3 tensor passes: "
                                       "3 x kind::f16 -> 1/3 of the bf16 peak (3 x kind::tf32 -> 1/6)"},
            "note": "algorithmic 2MNK per launch / CUDA-event launch time, measured with both towers on ONE stream "
                    "(no overlap between launches), so the GEMM time is a share of that serial step"}


def rule5_roofline(D: Dist, cfg, B: int):
    """Rule 5 (HBM-bound Hadamard / clamp / head-mean) at C2 all-layer size, timed alone with an L2 flush between reps."""
    import mmx_b200
    from mmx_b200._lib import ptr, current_stream
    torch = D.torch
    lib = mmx_b200.lib()
    dev = D.dev
    hbm_peak, _, _, peak_src = _peaks()
    Hh, S, Lr = cfg.transformer_heads, cfg.context_length, cfg.transformer_layers
    ld = (S + 3) // 4 * 4
    A = torch.rand(Lr * B, Hh, S, ld, device=dev)
    G = torch.randn(Lr * B, Hh, S, ld, device=dev)
    Ab = torch.empty(Lr * B, S, ld, device=dev)
    for _ in range(3):
        lib.mmx_avg_heads(ptr(A), ptr(G), ptr(Ab), Lr * B, Hh, S, ld, ld, ld, current_stream())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ts = []
    for _ in range(10):
        flush.zero_()                                          # L2 flush (256 MiB > 126 MB L2)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        lib.mmx_avg_heads(ptr(A), ptr(G), ptr(Ab), Lr * B, Hh, S, ld, ld, ld, current_stream())
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    r5_bytes = (2 * A.numel() + Ab.numel()) * 4
    r5_gbs = r5_bytes / (ts[len(ts) // 2] * 1e-3) / 1e9
    traffic, rec = captured_traffic("avg_heads")
    return {"kernel": "avg_heads (rule 5)", "bound": "hbm", "achieved": r5_gbs, "peak": hbm_peak, "unit": "GB/s",
            "frac": r5_gbs / hbm_peak, "traffic": traffic, "traffic_capture": rec, "bytes_per_launch": r5_bytes,
            "us_per_launch": ts[len(ts) // 2] * 1e3, "peak_source": peak_src}


def torch_eager_leg(D: Dist, cfg, B: int):
    """Informational: the reference's REAL deployment - eager fp32 PyTorch with one autograd.grad per block
    (CLIP_explainability.ipynb:175,198) - on the same GPU, via the oracle port moved to the device.  Never the target; it
    is the number a user of the reference on a B200 would compare against."""
    import torch
    import mmx_b200
    from oracle import clip_oracle as co
    dev = D.dev
    sd = {k: v.to(dev) for k, v in co.init_state_dict(co.VIT_B32, seed=0).items()}
    images, tokens = mmx_b200.clip_synthetic_inputs(cfg, B, seed=1234, length_seed=4321)
    images, tokens = images.to(dev), tokens.to(dev)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for _ in range(2):
            co.clip_interpret(sd, co.VIT_B32, images, tokens, START_LAYER, START_LAYER, per_layer_grad=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            co.clip_interpret(sd, co.VIT_B32, images, tokens, START_LAYER, START_LAYER, per_layer_grad=True)
        torch.cuda.synchronize()
        sec = (time.perf_counter() - t0) / reps
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return {"value": B / sec, "unit": UNIT, "ms_per_step": sec * 1e3, "kind": "port",
            "what": "oracle port of the notebook on cuda:0: eager fp32 PyTorch (cuBLAS fp32, TF32 off), one autograd.grad per "
                    "block, batch 64, all layers; 2 warm-ups + mean of 3 steps; informational only"}


# ---------------------------------------------------------------------------------------------------------------------
# the other BASELINE configs: DETR-R50 (config 3), LXMERT (config 4): host-side tapes replayed as CUDA graphs
# ---------------------------------------------------------------------------------------------------------------------
def _time_graph(D: Dist, call, steps: int, warm: int):
    torch = D.torch
    for _ in range(warm):
        call()
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        call()
    e1.record()
    D.barrier()
    return D.max(e0.elapsed_time(e1) / steps)


def _gemm_profile(lib, call, reps: int = 2):
    lib.mmx_profile_gemm(1)
    for _ in range(reps):
        call()
    lib.mmx_profile_gemm(0)
    tms, tfl, nl = C.c_double(), C.c_double(), C.c_int()
    lib.mmx_profile_gemm_report(C.byref(tms), C.byref(tfl), C.byref(nl))
    return tms.value / reps, tfl.value / reps, nl.value // reps


def bench_detr(D: Dist, B: int, steps: int, warm: int, outputs=None):
    """BASELINE config 3: DETR-R50 transformer (d 256, 8 heads, 6+6 layers, 100 queries) on 25x25 backbone features
    (625 tokens), B (image, query) pairs per GPU: Generator.generate_ours(use_lrp=False) (DETR/modules/
    ExplanationGenerator.py:142-195) captured once and replayed as a CUDA graph."""
    import mmx_b200
    torch = D.torch
    dev, lib = D.dev, mmx_b200.lib()
    cfg = mmx_b200.DETR_R50
    eng = mmx_b200.DetrEngine(mmx_b200.detr_init_state_dict(cfg, seed=9), nhead=cfg.nhead, device=dev)
    src, pos, tq = mmx_b200.detr_synthetic_inputs(cfg, B, 25, 25, seed=4 + D.rank)
    gen = mmx_b200.Generator(eng)
    args = (src.to(dev), pos.to(dev), tq.to(dev))
    l0 = lib.mmx_launch_count()
    eager_out = gen.generate_ours((args[0], args[1]), args[2], use_lrp=False).clone()
    launches = int(lib.mmx_launch_count() - l0)
    t_eager = _time_graph(D, lambda: gen.generate_ours((args[0], args[1]), args[2], use_lrp=False), max(2, steps // 2), 1)
    g = gen.capture((args[0], args[1]), args[2], use_lrp=False)
    ms = _time_graph(D, lambda: g(*args), steps, warm)
    if outputs is not None:
        (rel,) = g.outputs()
        outputs["relevance"] = rel.cpu()
    g.check()
    same = bool(torch.equal(g(*args), eager_out))
    # e2e: pinned host features in, the target query's relevance rows out
    pins = [a.cpu().pin_memory() for a in args]
    out_pin = torch.empty(B, 625).pin_memory()

    def e2e():
        out = g(*pins)
        out_pin.copy_(out.reshape(B, -1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(out_pin[0, 0])
    for _ in range(2):
        e2e()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e()
    D.barrier()
    e2e_s = D.max((time.perf_counter() - t0) / steps)
    gemm_ms, gemm_fl, gemm_n = _gemm_profile(lib, lambda: gen.generate_ours((args[0], args[1]), args[2], use_lrp=False))
    _, _, tf_sust, _ = _peaks()
    n_total = B * D.world
    return {"config": {"workload": "detr_r50_generate_ours_625tok_100q", "batch_per_gpu": B, "global_batch": n_total,
                       "tokens": 625, "queries": 100, "use_lrp": False, "features": "synthetic N(0,1) [B,256,25,25] + sine pos"},
            "unit": UNIT, "value": n_total / (ms * 1e-3), "ms_per_step": ms, "steps": steps, "warmup": warm,
            "launch": "CUDA graph replay (capture once)", "kernels_per_step": launches,
            "eager_tape": {"value": n_total / (t_eager * 1e-3), "ms_per_step": t_eager},
            "graph_equals_eager_bitwise": same,
            "e2e": {"value": n_total / e2e_s, "unit": UNIT, "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(sum(p.numel() * p.element_size() for p in pins)), "d2h_bytes_per_step": int(out_pin.numel() * 4)},
            "roofline": {"kernel": "transformer + rule GEMMs (all backends)", "bound": "tensor", "achieved": gemm_fl / (gemm_ms * 1e-3) / 1e12,
                         "peak": tf_sust, "unit": "TFLOP/s", "frac": gemm_fl / (gemm_ms * 1e-3) / 1e12 / tf_sust, "traffic": None,
                         "gemm_ms_per_step": gemm_ms, "launches_per_step": gemm_n, "flops_per_step": gemm_fl,
                         "note": "eager tape, per-launch CUDA events on one stream"}}


def bench_lxmert(D: Dist, B: int, steps: int, warm: int, outputs=None):
    """BASELINE config 4: LXMERT base (768 hidden, 12 heads, 9/5/5 layers), 20 tokens x 36 boxes, B questions per GPU:
    GeneratorOurs.generate_ours(use_lrp=False) (lxmert/lxmert/src/ExplanationGenerator.py:131-211) as a CUDA graph."""
    import mmx_b200
    torch = D.torch
    dev, lib = D.dev, mmx_b200.lib()
    cfg = mmx_b200.LXMERT_BASE
    eng = mmx_b200.LxmertEngine(mmx_b200.lxmert_init_state_dict(cfg, seed=1), num_heads=cfg.heads, device=dev)
    ids, feats, boxes = mmx_b200.lxmert_synthetic_inputs(cfg, B, 20, 36, seed=8 + D.rank)
    gen = mmx_b200.GeneratorOurs(eng)
    args = (ids.to(dev), feats.to(dev), boxes.to(dev))
    l0 = lib.mmx_launch_count()
    e_tt, e_ti = (t.clone() for t in gen.generate_ours(args, use_lrp=False))
    launches = int(lib.mmx_launch_count() - l0)
    t_eager = _time_graph(D, lambda: gen.generate_ours(args, use_lrp=False), max(2, steps // 2), 1)
    g = gen.capture(args, use_lrp=False)
    ms = _time_graph(D, lambda: g(*args), steps, warm)
    if outputs is not None:
        r_tt, r_ti = g.outputs()
        outputs.update(R_t_t=r_tt.cpu(), R_t_i=r_ti.cpu())
    g.check()
    o_tt, o_ti = g(*args)
    same = bool(torch.equal(o_tt, e_tt) and torch.equal(o_ti, e_ti))
    pins = [a.cpu().pin_memory() for a in args]
    out_pin = (torch.empty_like(o_tt, device="cpu").pin_memory(), torch.empty_like(o_ti, device="cpu").pin_memory())

    def e2e():
        a, b = g(*pins)
        out_pin[0].copy_(a, non_blocking=True)
        out_pin[1].copy_(b, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(out_pin[1].reshape(-1)[0])
    for _ in range(2):
        e2e()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e()
    D.barrier()
    e2e_s = D.max((time.perf_counter() - t0) / steps)
    gemm_ms, gemm_fl, gemm_n = _gemm_profile(lib, lambda: gen.generate_ours(args, use_lrp=False))
    _, _, tf_sust, _ = _peaks()
    n_total = B * D.world
    return {"config": {"workload": "lxmert_base_generate_ours_20tok_36box", "batch_per_gpu": B, "global_batch": n_total,
                       "use_lrp": False, "inputs": "synthetic ids / N(0,1) features [B,36,2048] / U(0,1) boxes"},
            "unit": UNIT, "value": n_total / (ms * 1e-3), "ms_per_step": ms, "steps": steps, "warmup": warm,
            "launch": "CUDA graph replay (capture once)", "kernels_per_step": launches,
            "eager_tape": {"value": n_total / (t_eager * 1e-3), "ms_per_step": t_eager},
            "graph_equals_eager_bitwise": same,
            "e2e": {"value": n_total / e2e_s, "unit": UNIT, "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(sum(p.numel() * p.element_size() for p in pins)),
                    "d2h_bytes_per_step": int(sum(p.numel() * 4 for p in out_pin))},
            "roofline": {"kernel": "transformer GEMMs (all backends)", "bound": "tensor", "achieved": gemm_fl / (gemm_ms * 1e-3) / 1e12,
                         "peak": tf_sust, "unit": "TFLOP/s", "frac": gemm_fl / (gemm_ms * 1e-3) / 1e12 / tf_sust, "traffic": None,
                         "gemm_ms_per_step": gemm_ms, "launches_per_step": gemm_n, "flops_per_step": gemm_fl,
                         "note": "eager tape, per-launch CUDA events on one stream"}}


def bench_l14(D: Dist, B: int, steps: int, warm: int, outputs=None):
    """BASELINE config 5: CLIP ViT-L/14@336, B pairs per GPU (2048 over 8 GPUs = 256 per GPU), micro-batches of 64."""
    import mmx_b200
    cfg = mmx_b200.VIT_L14_336
    res, eng, inputs = bench_clip(D, cfg, B, steps, warm, max_batch=64, with_default=False, with_check=False, e2e_steps=max(1, steps // 2),
                                  outputs=outputs)
    lib = mmx_b200.lib()
    eng.set_serial(True)
    gemm_ms, gemm_fl, gemm_n = _gemm_profile(lib, lambda: eng.interpret(inputs[0], inputs[1], START_LAYER, START_LAYER, validate=False), reps=1)
    eng.set_serial(False)
    _, _, tf_sust, _ = _peaks()
    out = {"config": {"workload": "clip_vit_l14_336_interpret_all_layers", "batch_per_gpu": B, "global_batch": B * D.world,
                      "micro_batch": 64, "start_layer": START_LAYER, "image": 336, "context": 77},
           "unit": UNIT, "value": res["value"], "ms_per_step": res["ms_per_step"], "steps": steps, "warmup": warm,
           "per_rank_ms": res["per_rank_ms"], "e2e": res["e2e"], "gpu_launches": res["launches"],
           "roofline": {"kernel": "transformer GEMMs (tcgen05 fp16x3)", "bound": "tensor", "achieved": gemm_fl / (gemm_ms * 1e-3) / 1e12,
                        "peak": tf_sust, "unit": "TFLOP/s", "frac": gemm_fl / (gemm_ms * 1e-3) / 1e12 / tf_sust, "traffic": None,
                        "gemm_ms_per_step": gemm_ms, "launches_per_step": gemm_n, "flops_per_step": gemm_fl,
                        "note": "both towers on one stream (mmx_clip_set_serial), per-launch CUDA events"}}
    if "collective" in res:
        out["collective"] = res["collective"]
    del eng
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="clip_b32", choices=["clip_b32", "detr_r50", "lxmert", "clip_l14_336"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the maps of the last timed step as DIR/<name>.npy (float32; seeded inputs, so runs compare)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import mmx_b200
    D = Dist()
    world, rank = D.world, D.rank
    warm = max(3, args.warmup)
    lib = mmx_b200.lib()
    outputs = {} if args.dump_outputs and rank == 0 else None

    if args.workload != "clip_b32":                       # one of the other configs as the main (and only) line
        fn, Bdef = {"detr_r50": (bench_detr, 16), "lxmert": (bench_lxmert, 16), "clip_l14_336": (bench_l14, 256)}[args.workload]
        r = fn(D, args.batch or Bdef, args.steps, warm, outputs=outputs)
        if rank == 0:
            r.update({"metric": "relevancy maps/sec (" + r["config"]["workload"] + ")", "n_gpus": world, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic"})
            if outputs is not None:
                dump_outputs(args.dump_outputs, outputs)
            print(json.dumps(r), flush=True)
        return D.close()

    B = args.batch or BATCH_PER_GPU
    cfg = mmx_b200.VIT_B32
    res, eng, inputs = bench_clip(D, cfg, B, args.steps, warm, max_batch=B, with_default=True, with_check=True, e2e_steps=args.steps,
                                  outputs=outputs)
    roofline = clip_roofline(D, eng, inputs, B, cfg)
    roofline_rule5 = rule5_roofline(D, cfg, B)
    eager = None
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            eager = torch_eager_leg(D, cfg, B)
        except Exception as exc:              # informational leg only
            eager = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    del eng, inputs
    torch.cuda.empty_cache()

    other = {}
    if not args.no_extra:
        for name, fn, Bo, st, wm in (("detr_r50", bench_detr, 16, 5, 3), ("lxmert", bench_lxmert, 16, 10, 3),
                                     ("clip_l14_336", bench_l14, 256, 2, 1)):
            try:
                other[name] = fn(D, Bo, st, wm)
            except Exception as exc:          # a secondary workload must not take the headline line down with it
                other[name] = {"error": f"{type(exc).__name__}: {exc}"[:500]}
            torch.cuda.empty_cache()

    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            threads = pick_threads()
            v, sec = cpu_baseline_run(16, 3, 1, threads)
            cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "host_cores": os.cpu_count(),
                   "sample": "the first 16 of the 64 pairs of the same batch (all layers), 1 warm-up + median of 3 reps; oracle port "
                             "of the reference's CPU PyTorch path incl. its per-block autograd.grad; thread count = fastest of "
                             "{all,64,32,16} in a quick probe"}
        out = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(world, B, cfg),
            "clocks": res["clocks"], "gpu_launches": res["launches"], "e2e": res["e2e"],
            "per_rank_ms": res["per_rank_ms"], "build": csrc_hash(),
            "roofline": roofline, "roofline_rule5": roofline_rule5, "cpu_baseline": cpu, "torch_eager_b200": eager,
            "default_mode": res.get("default_mode"), "other_workloads": other,
        }
        for k in ("collective", "sharded_equals_single"):
            if k in res:
                out[k] = res[k]
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(out), flush=True)
    D.close()


if __name__ == "__main__":
    main()
