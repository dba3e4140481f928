#!/usr/bin/env python
"""bench.py — denoising steps/sec of the VidToMe hot path on B200 (BASELINE.json metric, configs[1]).

Workload (config.workload = "sd15_512_f16_chunk_ratio0.9"): one denoising step of an SD1.5-shaped
skeleton UNet (vidtome_b200/skeleton.py: the 16 transformer blocks of SD1.5 with their (T, C, heads), 10 of
them merged at max_downsample=2) on a 16-frame chunk of 512x512 video (latents [16, 4, 64, 64], CFG batch 2,
fp16), local merge ratio 0.9, followed by the CFG combine and the DDIM update (vidtome_b200/driver.py restating
generate.py:205-311).  `--workload hot` (default) runs the self-attention section of every block (SURVEY §8 rows
a1-a15); `--workload full` adds each block's cross-attention and GEGLU feed-forward (row f3).  Weights are random
(no network for checkpoints), data synthetic.

One JSON line (rank 0):
  value         steps/s, latents resident in HBM, CUDA-graph replay of the step (whole job: N ranks x their chunk)
  e2e           same step through the public API with HOST latents: pinned host -> device copy of x_t, step,
                device -> host read of x_{t-1}, all inside the timed region
  roofline      KA (tcgen05 similarity + arg-max), the dominant kernel: algorithmic FLOPs of its launches / their
                CUDA-event durations (a short eager pass: events cannot bracket kernels inside a graph), against the
                measured cuBLAS peak;  rooflines: the same for KD (attention), K0, KC, KE (HBM-bound row kernels)
  comparators   measured in the same process on the same GPU (N=1, rank 0):
                  gpu_reference      the reference's own GPU formulation of the step (baseline/torch_reference_path.py:
                                     materialised score matrix + max + argsort + gathers/scatters, torch SDPA)
                  attention_ms       KD vs the module's own attention forward (cuBLAS projections + torch SDPA)
                  merge_ms_per_call  compute_merge + merge + unmerge + residual, attention excluded (BASELINE metric 2)
  cpu_baseline  the same restatement in torch fp32 on the host cores, bounded sample (numpy oracle as a second field)

`--impl reference` times that CPU restatement alone (the Python reference itself cannot travel to the GPU box).

`--dump-outputs DIR` writes, after the run, the latents x_{t-1} that the last timed step returned, as
DIR/latents.npy (float32, [16, 4, 64, 64]; DIR/latents_rank<k>.npy per rank when N > 1).  Weights and inputs are
seeded, so two builds run with the same arguments can be compared output for output.

Multi-GPU (`--gpus N` under torchrun): local merging makes frame chunks independent (generate.py:216-219), so
each rank denoises its own 16-frame chunk with replicated weights; nothing crosses GPUs in the data path
("scaling": "weak").  Timing = max over ranks of the CUDA-event time between two barriers.
For N > 1 the line also carries `c4_global`: BASELINE config 4 (SD2.1 768^2, one 8-frame chunk per GPU, global-token
exchange as NCCL all-gather and fused into the merge gather over peer memory); a watchdog prints the line without it if the
block does not return (`--no-c4-global` skips it).
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
sys.path.insert(0, ROOT)

FRAMES, LATENT = 16, 64
RATIO = 0.9
METRIC = "denoising steps/sec (SD1.5, 16-frame chunk)"


def workload_name(kind: str) -> str:
    return "sd15_512_f16_chunk_ratio0.9" + ("" if kind == "hot" else "_full_blocks")


def config_dict(world: int, kind: str) -> dict:
    blocks = ("sd15 census, 10 merged of 16, self-attention section" if kind == "hot" else
              "sd15 census, 10 merged of 16, self-attention + cross-attention + GEGLU feed-forward")
    return {"workload": workload_name(kind), "frames_per_chunk": FRAMES, "chunks": world, "latent": [4, LATENT, LATENT],
            "cfg_batch": 2, "local_merge_ratio": RATIO, "max_downsample": 2, "blocks": blocks,
            "parallelism": f"chunk-per-gpu x{world}",
            "l2": "per-step activation traffic (>1 GB) exceeds the 126 MB L2; no explicit flush between steps"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sust": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "src": "MEASURED_PEAKS.json"}
    return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sust": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock and throttle reasons sampled during the timed region: NVML in-process every 10 ms (pynvml; a 0.2 s timed
    region still gets ~20 samples), `nvidia-smi -lms 50` as the fallback when NVML cannot be loaded."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    # nvmlClocksThrottleReason* bit masks (nvml.h)
    BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index: int, uuid: str = ""):
        self.rows, self.proc, self.mode = [], None, None       # rows: (sm_mhz, max_mhz, set(reasons))
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
                except Exception:
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self._stop.is_set():
                    try:
                        sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        mask = int(reasons_fn(h))
                        self.rows.append((sm, mx, {n for n, b in self.BITS if mask & b}))
                    except Exception:
                        pass
                    self._stop.wait(0.01)
            self.thr = threading.Thread(target=loop, daemon=True)
            self.thr.start()
            self.mode = "nvml"
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
            self.mode = "nvidia-smi"
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                sm, mx = float(r[0]), float(r[1])
            except Exception:
                continue
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            self.rows.append((sm, mx, {n for n, c in zip(names, (4, 5, 6, 7)) if len(r) > c and r[c].lower().startswith("active")}))

    def count(self):
        return len(self.rows)

    def stop(self):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml / nvidia-smi unavailable"], "samples": 0}
        if self.mode == "nvidia-smi":
            time.sleep(0.25)
            self.proc.terminate()
        self._stop.set()
        rows = list(self.rows)
        sm = sorted(r[0] for r in rows)
        mx = rows[-1][1] if rows else None
        reasons = set().union(*[r[2] for r in rows]) if rows else set()
        # median over samples under load (idle samples at the edges report the idle clock)
        load = [v for v in sm if mx and v > 0.4 * mx] or sm
        return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": self.mode}


# ------------------------------------------------------------------------------------------------ CPU legs
def cpu_torch_block_calls(threads: int):
    """Self-attention section (patch.py:139-169) of one ds1 and one ds2 block of the workload on the host cores, in
    fp32 torch ops (the reference's formulation, baseline/torch_reference_path.py).  Returns callables -> seconds."""
    import torch
    from baseline import torch_reference_path as R
    from vidtome_b200.skeleton import BasicTransformerBlock, ModelMixin
    torch.set_num_threads(threads)

    def make(T, C, heads, ds):
        class One(ModelMixin):
            def __init__(self):
                super().__init__()
                self.block = BasicTransformerBlock(C, heads)

            def forward(self, latent, hidden):
                return self.block(hidden)
        torch.manual_seed(123)
        net = One().float().eval()
        R.apply_reference_path(net, RATIO, 2)
        base = torch.randn(2, 1, T, C)
        hid = (base + 0.1 * torch.randn(2, FRAMES, T, C)).reshape(2 * FRAMES, T, C)
        lat = torch.zeros(2 * FRAMES, 4, LATENT, LATENT)

        def run():
            t0 = time.perf_counter()
            with torch.no_grad():
                net(lat, hid)
            return time.perf_counter() - t0
        return run
    return make(4096, 320, 8, 1), make(1024, 640, 8, 2)


def cpu_numpy_block_calls():
    """The numpy oracle of the same two block calls (kept as a second CPU figure)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vidtome_oracle as O
    rng = np.random.default_rng(123)

    def make(T, C, heads):
        B, F = 2, FRAMES
        base = rng.standard_normal((B, 1, T, C))
        hid = (base + 0.1 * rng.standard_normal((B, F, T, C))).reshape(B * F, T, C).astype(np.float16)
        w = lambda *s: (rng.standard_normal(s) / np.sqrt(s[-1])).astype(np.float16)
        args = (np.ones(C, np.float16), np.zeros(C, np.float16), w(C, C), w(C, C), w(C, C), w(C, C), np.zeros(C, np.float16), heads)

        def run():
            t0 = time.perf_counter()
            O.tome_block_self_attention(hid, (LATENT, LATENT), *args, batch_size=B, local_merge_ratio=RATIO,
                                        draw_randf=lambda s: 1)
            return time.perf_counter() - t0
        return run
    return make(4096, 320, 8), make(1024, 640, 8)


def run_reference(args):
    """Reference arm: the torch fp32 restatement of the reference path on the host cores, all threads.  A step of
    the workload is 5 ds1 + 5 ds2 merged block calls (the 6 un-merged ds4/ds8 blocks are <1 % of the work); each
    timed "step" here is a bounded sample — one ds2 block call, plus one ds1 block call in the first three steps —
    and the step time is assembled as 5*mean(ds1) + 5*mean(ds2)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    ds1, ds2 = cpu_torch_block_calls(cores)
    for _ in range(max(1, min(args.warmup, 2))):
        ds2()
    t1, t2 = [], []
    for i in range(max(1, args.steps)):
        if i < 3:
            t1.append(ds1())
        t2.append(ds2())
    m1, m2 = sum(t1) / len(t1), sum(t2) / len(t2)
    step_s = 5.0 * m1 + 5.0 * m2
    val = 1.0 / step_s
    sample = ("torch fp32 restatement on %d threads: ds1 block call timed %d times (mean %.2f s), ds2 block call timed %d times "
              "(mean %.3f s); step = 5*ds1 + 5*ds2" % (cores, len(t1), m1, len(t2), m2))
    _print_json({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (host)", "data": "synthetic",
        "config": config_dict(max(1, args.gpus), args.workload),
        "cpu_baseline": {"value": val, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


# ------------------------------------------------------------------------------------------------ GPU helpers
_flush_buf = None


def _flush_l2(torch):
    global _flush_buf
    if _flush_buf is None:
        _flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    _flush_buf.fill_(1)


def _median_ms(torch, fn, iters=7, warm=2):
    """Median CUDA-event time of fn(), L2 flushed (256 MiB write) before every timed call."""
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(iters):
        _flush_l2(torch)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ts.sort()
    return ts[len(ts) // 2]


def ka_traffic():
    """dram bytes of the largest KA launch from the committed ncu --set full capture (profiles/r02_ka_traffic.json,
    written by tools/ncu_extract.py from the .ncu-rep); None when no capture of this build is committed."""
    p = os.path.join(ROOT, "profiles", "r02_ka_traffic.json")
    if not os.path.exists(p):
        return None
    try:
        return json.load(open(p))
    except Exception:
        return None


def comparators(torch, net, dev, steps, kind, cond=None):
    """Same-GPU, same-process comparators (N=1).  `net` arrives unpatched."""
    import vidtome_b200
    from types import SimpleNamespace
    from baseline import torch_reference_path as R
    from vidtome_b200 import ops, patch
    from vidtome_b200.driver import ChunkedDenoiser
    out = {"restatement_bit_exact_on_exact_inputs": R.check_exact(dev)}

    # ---- (i) the reference's GPU formulation of the whole step
    R.apply_reference_path(net, RATIO, 2)
    den = ChunkedDenoiser(net, n_timesteps=50, chunk_size=FRAMES, cond=cond)
    g = torch.Generator(device=dev).manual_seed(123)
    x = torch.randn((FRAMES, 4, LATENT, LATENT), generator=g, device=dev, dtype=torch.float16)
    for i in range(2):
        x = den.step(x, i)
    n = max(3, min(steps, 5))
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(n):
        x = den.step(x, i % 50)
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / n
    R.remove_reference_path(net)
    out["gpu_reference"] = {"value": round(1e3 / ms, 3), "unit": "steps/s", "ms_per_step": round(ms, 3), "steps": n,
                            "what": "reference formulation in torch ops on the same GPU (materialised a@b^T, max, argsort, "
                                    "gather/scatter, torch SDPA attention), same skeleton and weights, eager"}

    # ---- (ii) attention and (iii) merge ms/call at the two merged block shapes of the workload
    att, mrg = {}, {}
    for label, T, C, heads in (("C2_ds1", 4096, 320, 8), ("C2_ds2", 1024, 640, 8)):
        B = 2
        gg = torch.Generator(device=dev).manual_seed(7)
        base = torch.randn((B, 1, T, C), generator=gg, device=dev)
        xf = (base + 0.1 * torch.randn((B, FRAMES, T, C), generator=gg, device=dev)).reshape(B * FRAMES, T, C).half()
        module = SimpleNamespace(generator=torch.Generator(device=dev).manual_seed(7), global_tokens=None)
        info = {"size": (LATENT, LATENT), "args": dict(max_downsample=2, batch_size=B, align_batch=False, merge_global=False,
                                                        global_merge_ratio=0.8, local_merge_ratio=RATIO, global_rand=0.5,
                                                        target_stride=4)}
        plan = patch.build_merge_plan(module, xf, info)
        randfs = [int(r) for r in plan.randf]
        xj = xf.reshape(B, FRAMES * T, C)

        def ours_merge():
            p = patch.build_merge_plan(module, xf, info)
            return p.unmerge_add(p.merged_tokens, xf)
        ms_o = _median_ms(torch, ours_merge)
        ms_t = _median_ms(torch, lambda: R.torch_merge_call(xj, FRAMES, T, RATIO, randfs, xj), iters=5)
        mrg[label] = {"ours_ms": round(ms_o, 4), "torch_reference_path_ms": round(ms_t, 4), "speedup": round(ms_t / ms_o, 2),
                      "merged_len": int(plan.merged_tokens.shape[1])}
        L = int(plan.merged_tokens.shape[1])
        blk = [b for b in net.blocks if b.attn1.to_q.weight.shape[0] == C][0]
        merged = plan.merged_tokens
        from vidtome_b200 import attention as A
        ms_o = _median_ms(torch, lambda: A.self_attention(blk.attn1, merged))
        with torch.no_grad():
            ms_t = _median_ms(torch, lambda: blk.attn1(merged))
        att[label] = {"ours_ms": round(ms_o, 4), "torch_module_ms": round(ms_t, 4), "speedup": round(ms_t / ms_o, 2),
                      "B": B, "L": L, "C": C, "heads": heads}
    out["attention_ms"] = dict(att, what="KD (QKV projection + flash attention + out projection) vs the attention module's own "
                                        "forward (cuBLAS linears + torch scaled_dot_product_attention) on the merged tokens; L2 flushed")
    out["merge_ms_per_call"] = dict(mrg, what="compute_merge + merge + unmerge + residual for one block, attention excluded; L2 flushed")
    return out


def c4_global_block(torch, dist, dev, rank, world, steps, timed):
    """BASELINE config 4 (secondary block, `--c4-global`, N > 1): SD2.1-shaped skeleton at 768^2 (latent 96x96), one
    8-frame chunk per GPU, local 0.9 + GLOBAL 0.8 merging with the global-token set exchanged once per merged block
    (SURVEY §8e option A: rank k matches against the merged tokens of rank k-1), in both exchange modes."""
    import vidtome_b200
    from vidtome_b200 import ops, patch
    from vidtome_b200.driver import ChunkedDenoiser
    from vidtome_b200.skeleton import make_skeleton
    torch.manual_seed(123)
    net = make_skeleton("sd21", hot_path_only=True, device=dev)
    vidtome_b200.apply_patch(net, local_merge_ratio=RATIO, batch_size=2, merge_global=True, global_merge_ratio=0.8)
    g = torch.Generator(device=dev).manual_seed(900 + rank)
    x0 = torch.randn((8, 4, 96, 96), generator=g, device=dev, dtype=torch.float16)
    res = {"workload": "sd21_768_f8_chunk_per_gpu_local0.9_global0.8", "chunks": world, "frames_per_chunk": 8,
           "latent": [4, 96, 96], "exchange": {}}
    n = max(2, min(steps, 5))
    for mode in ("allgather", "p2p_all", "p2p"):
        patch.GLOBAL_EXCHANGE = mode
        try:
            den = ChunkedDenoiser(net, n_timesteps=50, chunk_size=8, merge_global=True)
            st = {"x": x0.clone()}

            def step(i):
                st["x"] = den.step(st["x"], i % 50)
            for i in range(2):
                step(i)
            ops.STATS.reset(timed=("KF",))
            ms = timed(step, n)
            ev = ops.STATS.events.get("KF", [])
            kf_ms = sum(s.elapsed_time(e) for s, e, _, _ in ev)
            kf_bytes = sum(b for _, _, _, b in ev)
            ops.STATS.reset()
            t = torch.tensor([kf_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res["exchange"][mode] = {"ms_per_step": round(ms / n, 3), "steps_per_s_all_ranks": round(world * n / (ms / 1e3), 3),
                                     "merge_gather_plus_exchange_ms_per_step": round(float(t.item()) / n, 4),
                                     "exchanges_per_step": len(ev) // n,
                                     "nvlink_bytes_per_rank_per_step": int(kf_bytes / n),
                                     "nvlink_GBs_per_rank_within_exchange": round(kf_bytes / max(kf_ms, 1e-9) / 1e6, 1)}
        except Exception as exc:                      # reported, never fatal for the headline line
            res["exchange"][mode] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    patch.GLOBAL_EXCHANGE = "recurrence"
    vidtome_b200.remove_patch(net)
    return res


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import vidtome_b200
    from vidtome_b200 import ops
    from vidtome_b200.driver import ChunkedDenoiser
    from vidtome_b200.skeleton import make_skeleton

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(123)
    kind = args.workload
    net = make_skeleton("sd15", hot_path_only=(kind == "hot"), device=dev)
    vidtome_b200.apply_patch(net, local_merge_ratio=RATIO, batch_size=2, merge_global=False)
    cond = None
    if kind != "hot":
        gc = torch.Generator(device=dev).manual_seed(5)
        cond = torch.randn((2, 77, 768), generator=gc, device=dev, dtype=torch.float16)
    den_eager = ChunkedDenoiser(net, n_timesteps=50, chunk_size=FRAMES, cond=cond)
    den_graph = ChunkedDenoiser(net, n_timesteps=50, chunk_size=FRAMES, cond=cond, cuda_graph=True)
    g = torch.Generator(device=dev).manual_seed(123 + rank)
    x0 = torch.randn((FRAMES, 4, LATENT, LATENT), generator=g, device=dev, dtype=torch.float16)
    x_host = x0.cpu().pin_memory()
    out_host = torch.empty_like(x_host).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            fn(i)
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    state = {"x": x0.clone()}

    def dev_step(i):                                           # latents resident in HBM, graph replay
        state["x"] = den_graph.step(state["x"], i % 50)

    def eager_step(i):
        state["x"] = den_eager.step(state["x"], i % 50)

    def e2e_step(i):
        x = x_host.to(dev, non_blocking=True)                  # H2D of this step's input (pinned)
        y = (den_eager if args.e2e_eager else den_graph).step(x, i % 50)
        out_host.copy_(y, non_blocking=True)                   # D2H of the step's result
        torch.cuda.current_stream().synchronize()              # the caller reads the result

    warm = max(3, args.warmup)
    for i in range(warm + 2):                                  # 2 eager steps, capture, then >= 3 replays
        dev_step(i)
    sampler = ClockSampler(local, str(getattr(torch.cuda.get_device_properties(local), "uuid", "") or "")) if rank == 0 else None
    ms = timed(dev_step, args.steps)
    last_x = state["x"]                                        # what the last timed step returned
    if sampler and world == 1 and sampler.mode is not None:
        # a timed region shorter than the sampler's period: keep the SAME workload running (untimed) until it has
        # a few samples under load, and say so
        t_end, extra = time.time() + 3.0, 0
        while sampler.count() < 5 and time.time() < t_end:
            dev_step(extra)
            torch.cuda.synchronize()
            extra += 1
    clocks = sampler.stop() if sampler else None
    if clocks is not None and sampler and world == 1:
        clocks["untimed_continuation_steps"] = extra if sampler.mode is not None else 0
    for i in range(3):
        e2e_step(i)
    ms_e2e = timed(e2e_step, args.steps)

    # per-kernel pass: eager stepping with every hot kernel bracketed by CUDA events on the launching stream
    n_k = max(2, min(args.steps, 5))
    eager_step(0)
    ops.STATS.reset(timed=("KA", "KD", "K0", "KC", "KE", "KB1", "FF1", "FF2", "XA"))
    ms_eager = timed(eager_step, n_k)
    launches_per_step = ops.STATS.launches / n_k
    events = dict(ops.STATS.events)
    ops.STATS.reset()

    line = {}

    def emit():
        """Print the one JSON line (rank 0).  Called exactly once: normally at the end; by the watchdog if the optional
        config-4 block does not come back (a stuck collective cannot be cancelled, but it must not cost the headline)."""
        if rank == 0 and line and not line.get("_printed"):
            line["_printed"] = True
            _print_json({k: v for k, v in line.items() if k != "_printed"})

    if rank == 0:
        pk = peaks()

        def summarise(name):
            ev = events.get(name, [])
            t = sum(s.elapsed_time(e) for s, e, _, _ in ev)
            return t, sum(f for _, _, f, _ in ev), sum(b for _, _, _, b in ev), len(ev)
        ka_ms, ka_flops, ka_bytes, ka_n = summarise("KA")
        tf = ka_flops / ka_ms / 1e9 if ka_ms > 0 else 0.0
        tr = ka_traffic()
        roof = {"bound": "tensor", "kernel": "gemm_kernel<256, ArgmaxEpi> (KA sim+argmax)", "achieved": round(tf, 1),
                "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": round(tf / pk["tf_sust"], 3),
                "frac_of_burst_peak": round(tf / pk["tf_burst"], 3),
                "peak_source": pk["src"] + " (sustained cuBLAS bf16: kernel timed inside a long step; burst figure beside it)",
                "launches": ka_n, "share_of_step": round(ka_ms / ms_eager, 3), "timed_in": f"{n_k} eager steps",
                "algorithmic_GB_per_step": round(ka_bytes / n_k / 1e9, 3),
                "traffic": None if tr is None else tr.get("dram_bytes"),
                "traffic_detail": tr}
        others = {}
        for name, bound, label in (("KD", "tensor", "vtm_attention: QKV gemm + flash_attn_kernel + out gemm"),
                                   ("K0", "hbm", "normalize_split_kernel (+ fused LayerNorm)"),
                                   ("KC", "hbm", "gather_rows_kernel (merge gather, + fused LayerNorm)"),
                                   ("KE", "hbm", "gather_rows_kernel<ADD> (unmerge + residual)"),
                                   ("KB1", "hbm", "radix_sort_fused_kernel (latency-bound: 3 grid barriers)"),
                                   ("FF1", "tensor", "gemm_kernel<256, GegluEpi> (GEGLU projection, gate fused)"),
                                   ("FF2", "tensor", "gemm_kernel<StoreEpi> (feed-forward output projection + bias + residual)"),
                                   ("XA", "hbm", "vtm_cross_attention: q / kv projections + flash over 77 keys + out projection (+residual)")):
            t, fl, by, n = summarise(name)
            if n == 0 or t <= 0:
                continue
            if bound == "tensor":
                a = fl / t / 1e9
                others[name] = {"bound": "tensor", "kernel": label, "achieved": round(a, 1), "peak": pk["tf_burst"],
                                "unit": "TFLOP/s", "frac": round(a / pk["tf_burst"], 3), "launches": n,
                                "ms_per_step": round(t / n_k, 4), "share_of_step": round(t / ms_eager, 3),
                                "note": ("head_dim 40/80: the softmax exponentials (MUFU) bound this kernel before the tensor pipe does"
                                         if name == "KD" else "tcgen05 GEMM with a fused epilogue")}
            else:
                a = by / t / 1e6
                others[name] = {"bound": "hbm", "kernel": label, "achieved": round(a, 1), "peak": pk["hbm"], "unit": "GB/s",
                                "frac": round(a / pk["hbm"], 3), "launches": n, "ms_per_step": round(t / n_k, 4),
                                "share_of_step": round(t / ms_eager, 3)}
        value = world * args.steps / (ms / 1e3)
        out = {
            "metric": METRIC, "value": round(value, 3), "unit": "steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": round(ms / args.steps, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": config_dict(world, kind),
            "value_mode": "cuda_graph replay (ChunkedDenoiser(cuda_graph=True)), latents resident",
            "clocks": clocks,
            "e2e": {"value": round(world * args.steps / (ms_e2e / 1e3), 3), "unit": "steps/s",
                    "h2d_bytes_per_step": x_host.numel() * 2, "d2h_bytes_per_step": out_host.numel() * 2,
                    "ms_per_step": round(ms_e2e / args.steps, 3),
                    "mode": "eager" if args.e2e_eager else "cuda_graph replay (ChunkedDenoiser(cuda_graph=True))"},
            "gpu_launches": int(round(launches_per_step * args.steps)),
            "gpu_launches_note": "kernels of this library per step (counted over the eager pass) x steps; the timed region replays them from a CUDA graph",
            "eager_ms_per_step": round(ms_eager / n_k, 3),
            "roofline": roof,
            "rooflines": others,
        }
        if world == 1 and not args.no_gpu_ref:
            vidtome_b200.remove_patch(net)
            out["comparators"] = comparators(torch, net, dev, args.steps, kind, cond)
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            ds1, ds2 = cpu_torch_block_calls(cores)
            t1, t2 = ds1(), min(ds2(), ds2())
            step_s = 5 * t1 + 5 * t2
            cb = {"value": round(1.0 / step_s, 5), "unit": "steps/s", "cores": cores, "kind": "port",
                  "sample": "torch fp32 restatement of the reference path (baseline/torch_reference_path.py), self-attention section "
                            "of 1 ds1 block (%.2f s) and 1 ds2 block (%.3f s); step = 5*ds1 + 5*ds2" % (t1, t2)}
            if not args.no_numpy:
                n1, n2 = cpu_numpy_block_calls()
                u1, u2 = n1(), n2()
                cb["numpy_oracle"] = {"value": round(1.0 / (5 * u1 + 5 * u2), 5), "unit": "steps/s",
                                      "sample": "numpy oracle, same two block calls (%.2f s, %.3f s)" % (u1, u2)}
            out["cpu_baseline"] = cb
        line.update(out)
    # BASELINE config 4 (global-token exchange) as a secondary block of the N > 1 line; guarded by a watchdog
    if world > 1 and not args.no_c4_global:
        def bail():
            if rank == 0:
                line["c4_global"] = {"error": "timed out after %d s; headline numbers above are unaffected" % args.c4_timeout}
            emit()
            os._exit(0)
        wd = threading.Timer(args.c4_timeout, bail)
        wd.daemon = True
        wd.start()
        try:
            c4 = c4_global_block(torch, dist, dev, rank, world, args.steps, timed)
        except Exception as exc:
            c4 = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        wd.cancel()
        if rank == 0:
            line["c4_global"] = c4
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "latents" if world == 1 else f"latents_rank{rank}"
        np.save(os.path.join(args.dump_outputs, name + ".npy"), last_x.float().cpu().numpy())
    emit()
    if world > 1:
        dist.destroy_process_group()


_JSON_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write to fd 1 behind Python's back (NCCL prints its version line
    there at WARN level), so fd 1 is pointed at stderr for the whole run and the JSON line goes to a private duplicate of
    the original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _print_json(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="hot", choices=["hot", "full"],
                    help="hot = self-attention section of every block (SURVEY §8 a1-a15); full = + cross-attention and feed-forward (f3)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-numpy", action="store_true", help="skip the numpy-oracle second CPU figure")
    ap.add_argument("--no-gpu-ref", action="store_true", help="skip the same-GPU comparators")
    ap.add_argument("--e2e-eager", action="store_true", help="end-to-end leg without CUDA-graph replay")
    ap.add_argument("--c4-global", action="store_true", help="(default for N > 1; kept for compatibility)")
    ap.add_argument("--no-c4-global", action="store_true",
                    help="N > 1: skip the secondary BASELINE config-4 block (global-token exchange: all-gather and fused p2p)")
    ap.add_argument("--c4-timeout", type=int, default=240, help="watchdog for the config-4 block, seconds")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the latents returned by the last timed step to DIR/latents.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times block calls, not steps)")
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
