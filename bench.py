#!/usr/bin/env python
"""Benchmark of the B200-native PARSeq engine: images/sec, PARSeq-S 32x128, AR + 1 refine iteration
(BASELINE.json metric; configs[1]: bs=512 per GPU, bf16 tensor-core operands, synthetic crops / seeded
random weights), end to end through the host-buffer C-ABI call, p50 latency at bs=1 (engine call and the
reference's own `model(x)` protocol), roofline entries for every kernel kind >= 10 % of the step, a parity
check of the timed batch against the fp32 oracle, the other BASELINE configs, and the reference's CPU path
timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One JSON line on stdout (rank 0).  "step" = one forward of `batch` images per GPU (weak scaling:
images are independent, no data-path collective; model.py:105-169 has no cross-image dependency).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY.md section 8(d): algorithmic FLOPs per image (2 FLOP per MAC)
ALG_GFLOP_PER_IMAGE = 6.038          # PARSeq-S, AR + 1 refine (C2 / C3)
ALG_GFLOP_C4 = 6.253                 # PARSeq-S, AR + 3 refine
ALG_GFLOP_C1 = 1.558                 # PARSeq-Ti, NAR, no refine
ALG_GFLOP_C5_ENC, ALG_GFLOP_C5_FULL = 42.93, 44.34    # ViT-B-width 48x160: encoder only / AR + 1 refine


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=512, help="images per GPU per step")
    ap.add_argument("--chunk", type=int, default=0, help="images per pipeline stage (0 = engine default)")
    ap.add_argument("--max-batch", type=int, default=0, help="images per super-chunk / CUDA graph (0 = default)")
    ap.add_argument("--dec-chunk", type=int, default=0, help="images per decoder chain (0 = engine default 128)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-pdl", action="store_true")
    ap.add_argument("--fuse-ln", type=int, default=-1, help="bit 0: attn.proj, bit 1: mlp.fc2 fused with the following LayerNorm (engine default 3)")
    ap.add_argument("--attn-impl", type=int, default=-1, help="encoder attention: 1 tcgen05 (default), 0 mma.sync")
    ap.add_argument("--ar-kernel", type=int, default=-1, help="AR loop: 2 cluster kernel (default), 1 grid-barrier kernel, 0 separate kernels")
    ap.add_argument("--cta-group", type=int, default=0, help="GEMM tile: 0 auto, 1 single CTA, 2 CTA pair")
    ap.add_argument("--ln-cta-group", type=int, default=0, help="fused GEMM+LN tile: 0 auto, 1 single CTA, 2 CTA pair")
    ap.add_argument("--pair-pdl", type=int, default=-1, help="experiments: PDL attribute on CTA-pair launches")
    ap.add_argument("--ln-split", type=int, default=-1, help="fused GEMM+LN: 2 = column-split CTA-pair kernel (gemm_ln2.cuh), 1 = full-row kernel")
    ap.add_argument("--fuse-mlp", type=int, default=-1, help="1: fc1 + GELU + fc2 + residual + LayerNorm in one kernel (mlp_ln.cuh)")
    ap.add_argument("--block-n", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configs (C1, C4, C5)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-two-in-flight", action="store_true", help="skip the two-handles / two-threads end-to-end extra")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0: logits, ids, steps) to DIR/<name>.npy as float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the engine's outputs: it needs --impl ours")
    return args


DUMP_MAX_BYTES = 64_000_000


def dump_outputs(out_dir, logits, ids, steps):
    """The arrays the caller of the timed path receives, as float32 .npy files (ids <= 96 and the step count are exact).
    When the batch is too large for DUMP_MAX_BYTES, a fixed seeded sample of rows is written with its row indices."""
    import numpy as np
    import torch
    B = logits.shape[0]
    row_bytes = (logits[0].numel() + ids[0].numel()) * 4
    arrays = {"logits": logits, "ids": ids}
    if B * row_bytes > DUMP_MAX_BYTES:
        n = (DUMP_MAX_BYTES - 4096) // (row_bytes + 4)          # + its row index; 4 KB for the .npy headers
        rows = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:n].sort().values
        arrays = {k: v.cpu()[rows] for k, v in arrays.items()}
        arrays["rows"] = rows
    arrays["steps"] = steps
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().to(torch.float32).numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: an NVML polling thread (every 5 ms; the timed region of the
    default run is ~130 ms - too short for a freshly started `nvidia-smi -lms`), `nvidia-smi` as the fallback."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.thread = None
        self.stop_flag = False
        self.sm, self.mx, self.reasons, self.power = [], [], set(), []
        self.path = f"/tmp/parseq_clocks_{os.getpid()}.csv"

    def _poll(self):
        import pynvml as N
        h = self.handle
        masks = [(N.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"), (N.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                 (N.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"), (N.nvmlClocksEventReasonSwPowerCap, "sw_power_cap")]
        get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.sm.append(float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)))
                r = int(get_reasons(h))
                for m, n in masks:
                    if r & m:
                        self.reasons.add(n)
                self.power.append(N.nvmlDeviceGetPowerUsage(h) / 1000.0)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import pynvml as N
            import threading
            N.nvmlInit()
            self.handle = N.nvmlDeviceGetHandleByIndex(self.index)
            self.mx = [float(N.nvmlDeviceGetMaxClockInfo(self.handle, N.NVML_CLOCK_SM))]
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            if self.sm:
                out = {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": max(self.mx), "reasons": sorted(self.reasons),
                       "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None, "source": "nvml"}
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 7:
                    continue
                try:
                    sm.append(float(parts[0])); mx.append(float(parts[1]))
                except ValueError:
                    continue
                for n, v in zip(self.NAMES, parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            os.remove(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                   "samples": len(sm), "source": "nvidia-smi"}
        return out


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_forward_fn(cfg, sd, decode_ar=True, refine_iters=1):
    """The reference's CPU implementation of the path: the UNMODIFIED `strhub.models.parseq.model.PARSeq`
    (byte-compiled into oracle/_ref by oracle/build_ref.py, or the source tree when present) -> kind "reference";
    else the oracle port (pinned to it by tests/golden) -> kind "port"."""
    import torch
    from oracle import reference_loader as RL
    if RL.available():
        ref, tok = RL.build_reference_model(cfg, sd)
        ref.decode_ar, ref.refine_iters = decode_ar, refine_iters

        def fwd(x):
            with torch.inference_mode():
                return ref(tok, x)
        return fwd, "reference", f"strhub.models.parseq.model.PARSeq ({RL.kind()} @ {os.path.relpath(RL.REF_ROOT, ROOT) if RL.kind() == 'pyc' else RL.REF_ROOT}, timm shim)"
    from oracle.parseq_oracle import ParseqOracle
    o = ParseqOracle(cfg, sd, "fp32")
    return (lambda x: o.forward(x, None, decode_ar, refine_iters).logits), "port", "fp32 torch CPU oracle of model.py:105-169"


def pick_cpu_threads(fwd, cfg):
    """torch's intra-op pool is not automatically fastest at os.cpu_count() threads on a many-core host (the
    decoder's small matmuls oversubscribe); give the CPU arm its best thread count from a short probe."""
    import torch
    from parseq_b200.weights import synth_images
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    probe = synth_images(cfg, 16, 7)
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        fwd(probe[:4])
        t0 = time.perf_counter(); fwd(probe); dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_images_per_sec(cfg, sd, batch, repeats):
    import torch
    from parseq_b200.weights import synth_images
    fwd, kind, what = cpu_forward_fn(cfg, sd)
    pick_cpu_threads(fwd, cfg)
    x = synth_images(cfg, batch, 4242)
    fwd(x[: max(1, batch // 8)])     # warm-up
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fwd(x)
        ts.append(time.perf_counter() - t0)
    return batch / statistics.median(ts), torch.get_num_threads(), kind, what


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores, same metric / config,
    a bounded sample per step."""
    import torch
    from parseq_b200.config import make_config
    from parseq_b200.weights import init_state_dict, synth_images
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = make_config("parseq")
    sd = init_state_dict(cfg, 0)
    fwd, kind, what = cpu_forward_fn(cfg, sd)
    pick_cpu_threads(fwd, cfg)
    probe = synth_images(cfg, 8, 1)
    fwd(probe)
    t0 = time.perf_counter(); fwd(probe); dt = time.perf_counter() - t0
    ips0 = 8 / dt
    budget_s = 150.0
    sample = int(max(1, min(args.batch, ips0 * budget_s / max(1, args.steps + args.warmup))))
    x = synth_images(cfg, sample, 2)
    for _ in range(args.warmup):
        fwd(x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fwd(x)
    dt = time.perf_counter() - t0
    val = sample * args.steps / dt
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": "images/sec PARSeq-S 32x128 AR+1refine", "value": val, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "PARSeq-S 32x128 94-char max_len=25 bs=512/GPU AR + 1 refine (BASELINE configs[1])",
                   "note": f"CPU arm steps over a bounded sample of {sample} images", "batch_per_step": sample},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": kind,
                         "sample": f"{sample} images/step x {args.steps} steps, {what}"},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm helpers
def device_time_ms(fn, iters, warm=3):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def build_model(experiment, dev, decode_ar, refine_iters, opts=None, seed=0):
    from parseq_b200.config import make_config
    from parseq_b200.factory import create_model
    from parseq_b200.weights import init_state_dict
    cfg = make_config(experiment)
    sd = init_state_dict(cfg, seed)
    m = create_model(experiment, decode_ar=decode_ar, refine_iters=refine_iters)
    m.model.load_state_dict(sd)
    for k, v in (opts or {}).items():
        m.model.set_engine_option(k, v)
    return cfg, sd, m.eval().to(dev)


def infer(fn, x):
    import torch
    with torch.inference_mode():
        return fn(x)


def other_configs(dev, world, peak_tf, dist):
    """BASELINE.json configs[0], [3], [4]: device-timed, module API (`model(x)`), same engine."""
    import torch
    from parseq_b200.weights import synth_images
    out = {}
    if True:
        if world == 1:
            # C1: PARSeq-Ti bs=1 NAR (decode_ar=False, refine_iters=0): latency
            cfg, _, m = build_model("parseq-tiny", dev, False, 0)
            x = synth_images(cfg, 1, 3).to(dev)
            ms = device_time_ms(lambda: infer(m, x), 300, 20)
            out["C1"] = {"workload": "PARSeq-Ti 32x128 bs=1 NAR, no refine (configs[0])", "ms": ms, "images_per_s": 1000.0 / ms,
                         "frac_of_tensor_peak": (1000.0 / ms) * ALG_GFLOP_C1 * 1e9 / (peak_tf * 1e12)}
            del m
            # C4: PARSeq-S bs=1024 AR + 3 refine (two super-chunks of 512)
            cfg, _, m = build_model("parseq", dev, True, 3)
            x = synth_images(cfg, 1024, 4).to(dev)
            ms = device_time_ms(lambda: infer(m, x), 5, 2)
            ips = 1024 * 1000.0 / ms
            out["C4"] = {"workload": "PARSeq-S 32x128 bs=1024 AR + 3 refine, 1 GPU (configs[3])", "ms": ms, "images_per_s": ips,
                         "frac_of_tensor_peak": ips * ALG_GFLOP_C4 * 1e9 / (peak_tf * 1e12)}
            del m
        # C5: ViT-B-width encoder 48x160 (T = 240, D = 768), 256 images per GPU (bs=2048 over 8 GPUs)
        cfg, _, m = build_model("parseq-base-48x160", dev, True, 1, {"max_batch": 256})
        x = synth_images(cfg, 256, 5).to(dev)
        ms_full = device_time_ms(lambda: infer(m, x), 4, 2)
        ms_enc = device_time_ms(lambda: infer(m.model.encode, x), 4, 2)
        if dist is not None:
            t = torch.tensor([ms_full, ms_enc], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_full, ms_enc = float(t[0]), float(t[1])
        ips_full, ips_enc = world * 256 * 1000.0 / ms_full, world * 256 * 1000.0 / ms_enc
        out["C5"] = {"workload": f"PARSeq ViT-B-width encoder (D=768) 48x160, 256 images/GPU x {world} GPU (configs[4])",
                     "full_ar1": {"ms": ms_full, "images_per_s": ips_full,
                                  "frac_of_tensor_peak": ips_full / world * ALG_GFLOP_C5_FULL * 1e9 / (peak_tf * 1e12)},
                     "encode_only": {"ms": ms_enc, "images_per_s": ips_enc,
                                     "frac_of_tensor_peak": ips_enc / world * ALG_GFLOP_C5_ENC * 1e9 / (peak_tf * 1e12)}}
        del m
    torch.cuda.empty_cache()
    return out


def parity_block(model, cfg, sd, batch_cpu, logits_dev, ids_dev, nrows=16, tau=2e-2, fuse_restore=3):
    """Rows of the LAST TIMED batch against the fp32 CPU oracle (outside the timed region):
    free-running (what the timed step computed) and teacher-forced along the oracle's own id trajectory."""
    import torch
    from oracle.parseq_oracle import ParseqOracle
    B = batch_cpu.shape[0]
    rows = torch.linspace(0, B - 1, nrows).long()
    x = batch_cpu[rows]
    o = ParseqOracle(cfg, sd, "fp32").forward(x, None, True, 1)
    lg = logits_dev.cpu()[rows]
    ids = ids_dev.cpu()[rows].long()
    clear_rows = o.min_margin > tau
    same_rows = (ids == o.ids).all(dim=1)
    free = {"rows": int(nrows), "decisions_identical_frac": float((ids == o.ids).float().mean()),
            "rows_all_margins_clear": int(clear_rows.sum()),
            "of_those_ids_identical": int((same_rows & clear_rows).sum()),
            "rows_ids_identical": int(same_rows.sum())}
    if bool(same_rows.any()):           # logits are comparable where the trajectories coincide
        d = (lg[same_rows] - o.logits[same_rows]).abs()
        free["max_abs_dlogit_on_identical_rows"] = float(d.max())
        free["mean_abs_dlogit_on_identical_rows"] = float(d.mean())
    # teacher forcing: the engine follows the oracle's ids, so every row compares (same kernels as the timed batch:
    # fused residual-GEMM + LayerNorm forced for the small batch)
    forced = o.ar_ids.int()
    forced_refine = torch.stack([c.int() for c in o.refine_ctx])
    model.model.set_engine_option("fuse_ln", 7)
    with torch.inference_mode():
        lt = model.model.forward(model.tokenizer, x.to(logits_dev.device), None, forced_ids=forced,
                                 forced_refine=forced_refine).cpu()
    model.model.set_engine_option("fuse_ln", fuse_restore)
    d = (lt - o.logits).abs()
    top2 = o.logits.topk(2, dim=-1).values
    clear = (top2[..., 0] - top2[..., 1]) > tau
    tf = {"max_abs_dlogit": float(d.max()), "mean_abs_dlogit": float(d.mean()),
          "clear_decisions": int(clear.sum()), "decisions": int(clear.numel()),
          "clear_decisions_identical": bool((lt.argmax(-1) == o.logits.argmax(-1))[clear].all())}
    ok = tf["clear_decisions_identical"] and tf["max_abs_dlogit"] <= 2e-2 and free["of_those_ids_identical"] == free["rows_all_margins_clear"]
    return {"oracle": "fp32 CPU oracle (oracle/parseq_oracle.py, pinned to the reference's modules by tests/golden)",
            "tau": tau, "tolerance": {"max_abs_dlogit": 2e-2}, "free_running": free, "teacher_forced": tf, "ok": bool(ok)}


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    from parseq_b200.weights import synth_images

    opts = {}
    if args.max_batch:
        opts["max_batch"] = args.max_batch
    if args.chunk:
        opts["chunk"] = args.chunk
    if args.dec_chunk:
        opts["dec_chunk"] = args.dec_chunk
    if args.no_graph:
        opts["use_graph"] = 0
    if args.no_pdl:
        opts["pdl"] = 0
    if args.attn_impl >= 0:
        opts["attn_impl"] = args.attn_impl
    if args.ar_kernel >= 0:
        opts["ar_kernel"] = args.ar_kernel
    if args.fuse_ln >= 0:
        opts["fuse_ln"] = args.fuse_ln
    if args.cta_group:
        opts["cta_group"] = args.cta_group
    if args.ln_cta_group:
        opts["ln_cta_group"] = args.ln_cta_group
    if args.pair_pdl >= 0:
        opts["pair_pdl"] = args.pair_pdl
    if args.ln_split >= 0:
        opts["ln_split"] = args.ln_split
    if args.fuse_mlp >= 0:
        opts["fuse_mlp"] = args.fuse_mlp
    if args.block_n:
        opts["block_n"] = args.block_n
    cfg, sd, model = build_model("parseq", dev, True, 1, opts)
    eng = model.model.engine()
    B = args.batch
    st = torch.cuda.current_stream(dev)

    # Inputs larger than L2: NROT distinct resident batches (NROT * 25.2 MB > 126 MB), rotated per step.
    NROT = 8
    batches_cpu = [synth_images(cfg, B, 100 + rank * NROT + i) for i in range(NROT)]
    batches = [b.to(dev) for b in batches_cpu]
    logits = torch.empty((B, 26, cfg.num_classes), dtype=torch.float32, device=dev)
    ids = torch.empty((B, 26), dtype=torch.int32, device=dev)
    steps_t = torch.empty((1,), dtype=torch.int32, device=dev)

    def step(i):
        eng.forward(batches[i % NROT].data_ptr(), B, logits.data_ptr(), ids.data_ptr(), steps_t.data_ptr(),
                    st.cuda_stream, None, True, 1)

    for i in range(max(3, args.warmup)):
        step(i)
    torch.cuda.synchronize(dev)
    if distributed:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record(st)
    for i in range(args.steps):
        step(i)
    e1.record(st)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    launches = eng.launches - l0
    last_batch = (args.steps - 1) % NROT
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, logits, ids, steps_t)
    if distributed:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else {}
    value = world * B * args.steps / (ms / 1000.0)

    # ---- the one collective of the path, outside the throughput region: all-gather of the decoded ids over NCCL ----
    gather = None
    if distributed:
        from parseq_b200.parallel import gather_ids, global_steps
        total = world * B
        for _ in range(3):
            g = gather_ids(ids, total)
        torch.cuda.synchronize(dev)
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        NG = 20
        a.record(st)
        for _ in range(NG):
            g = gather_ids(ids, total)
        b.record(st)
        torch.cuda.synchronize(dev)
        t = torch.tensor([a.elapsed_time(b) / NG], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t0 = time.perf_counter()
        S = global_steps(int(steps_t.item()) if int(steps_t.item()) > 0 else 26, dev)
        s_us = (time.perf_counter() - t0) * 1e6
        ok = bool(g.shape == (total, 26) and torch.equal(g[rank * B:(rank + 1) * B], ids))
        gather = {"op": "NCCL all_gather of int32 ids [B/G, 26] (parseq_b200.parallel.gather_ids)", "us": float(t.item()) * 1000.0,
                  "bytes_out_per_rank": total * 26 * 4, "bytes_in_per_rank": B * 26 * 4, "own_block_verified": ok,
                  "max_reduce_steps_us_host": s_us, "S": S, "in_timed_region": False}

    # ---- end-to-end through the host-buffer entry point (pinned host memory, H2D + D2H inside) ----
    himg = [synth_images(cfg, B, 500 + rank * 2 + i).pin_memory() for i in range(2)]
    hlog = torch.empty((B, 26, cfg.num_classes), dtype=torch.float32).pin_memory()
    hids = torch.empty((B, 26), dtype=torch.int32).pin_memory()
    hsteps = torch.empty((1,), dtype=torch.int32).pin_memory()
    for i in range(2):
        eng.forward_host(himg[i % 2].data_ptr(), B, hlog.data_ptr(), hids.data_ptr(), hsteps.data_ptr(),
                         st.cuda_stream, None, True, 1)
    if distributed:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        eng.forward_host(himg[i % 2].data_ptr(), B, hlog.data_ptr(), hids.data_ptr(), hsteps.data_ptr(),
                         st.cuda_stream, None, True, 1)
    e2e_s = time.perf_counter() - t0
    if distributed:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_val = world * B * args.steps / e2e_s
    # extra (SURVEY 8f-2): same end-to-end call with raw uint8 HWC crops (transform folded into the patch gather)
    hu8 = [torch.randint(0, 256, (B, cfg.img_size[0], cfg.img_size[1], 3), dtype=torch.uint8).pin_memory() for _ in range(2)]
    for i in range(2):
        eng.forward_u8(hu8[i % 2].data_ptr(), B, hlog.data_ptr(), hids.data_ptr(), hsteps.data_ptr(), st.cuda_stream, None,
                       True, 1, host=True)
    t0 = time.perf_counter()
    for i in range(args.steps):
        eng.forward_u8(hu8[i % 2].data_ptr(), B, hlog.data_ptr(), hids.data_ptr(), hsteps.data_ptr(), st.cuda_stream, None,
                       True, 1, host=True)
    e2e_u8_s = time.perf_counter() - t0
    if distributed:
        t = torch.tensor([e2e_u8_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_u8_s = float(t.item())
    e2e_u8_val = world * B * args.steps / e2e_u8_s
    h2d = B * 3 * cfg.img_size[0] * cfg.img_size[1] * 4
    d2h = B * 26 * cfg.num_classes * 4 + B * 26 * 4 + 4

    # extra: the same host-buffer call with TWO batches in flight - two engine handles (same weights), two streams, two
    # host threads (the C ABI's contract: one handle per calling thread).  One handle's uploads / downloads run under the
    # other's kernels.  Reported next to `e2e` (one synchronous call after the other), never instead of it.
    e2e2 = None
    if not args.no_two_in_flight:
        import threading
        _, _, model_b = build_model("parseq", dev, True, 1, opts)
        engs = [eng, model_b.model.engine()]
        streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
        outs = [(torch.empty((B, 26, cfg.num_classes), dtype=torch.float32).pin_memory(),
                 torch.empty((B, 26), dtype=torch.int32).pin_memory(), torch.empty((1,), dtype=torch.int32).pin_memory())
                for _ in range(2)]
        per = (args.steps + 1) // 2

        def worker(k, n):
            torch.cuda.set_device(dev)
            for _ in range(n):
                engs[k].forward_host(himg[k].data_ptr(), B, outs[k][0].data_ptr(), outs[k][1].data_ptr(), outs[k][2].data_ptr(),
                                     streams[k].cuda_stream, None, True, 1)

        for k in range(2):
            worker(k, 2)                         # warm-up (graphs of the second handle), single-threaded
        torch.cuda.synchronize(dev)
        if distributed:
            dist.barrier()
        th = [threading.Thread(target=worker, args=(k, per)) for k in range(2)]
        t0 = time.perf_counter()
        for t_ in th:
            t_.start()
        for t_ in th:
            t_.join()
        e2e2_s = time.perf_counter() - t0
        if distributed:
            t = torch.tensor([e2e2_s], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e2_s = float(t.item())
        e2e2 = {"value": world * B * 2 * per / e2e2_s, "unit": "images/s", "steps": 2 * per, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": 1000 * e2e2_s / (2 * per),
                "what": "parseq_forward_host from two host threads on two engine handles / streams (two batches in flight)"}
        # the same with inputs resident in HBM (device pointers): what two batches in flight are worth without the copies
        douts = [(torch.empty((B, 26, cfg.num_classes), dtype=torch.float32, device=dev),
                  torch.empty((B, 26), dtype=torch.int32, device=dev), torch.empty((1,), dtype=torch.int32, device=dev))
                 for _ in range(2)]

        def dworker(k, n):
            torch.cuda.set_device(dev)
            for i in range(n):
                engs[k].forward(batches[(2 * i + k) % NROT].data_ptr(), B, douts[k][0].data_ptr(), douts[k][1].data_ptr(),
                                douts[k][2].data_ptr(), streams[k].cuda_stream, None, True, 1)

        for k in range(2):
            dworker(k, 2)
        torch.cuda.synchronize(dev)
        th = [threading.Thread(target=dworker, args=(k, per)) for k in range(2)]
        t0 = time.perf_counter()
        for t_ in th:
            t_.start()
        for t_ in th:
            t_.join()
        torch.cuda.synchronize(dev)
        dev2_s = time.perf_counter() - t0
        e2e2["device_resident"] = {"value": world * B * 2 * per / dev2_s, "ms_per_step": 1000 * dev2_s / (2 * per),
                                   "timing": "host wall clock around both threads + device synchronize (rank-local)"}
        del model_b

    peaks, peak_src = load_peaks()
    # kernels are timed inside a long step -> the sustained cuBLAS figure is the tensor denominator
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    peak_hbm = float(peaks.get("hbm_gbs", 6650.0))

    configs = None
    if not args.no_configs:
        configs = other_configs(dev, world, peak_tf, dist if distributed else None)

    if distributed:
        dist.barrier()
    if rank != 0:
        if distributed:
            dist.destroy_process_group()
        return

    # ---- roofline pass: per-category device time from CUDA-event pairs around every launch (serialised on one stream) ----
    eng.set_option("timing", 1)
    step(last_batch)
    torch.cuda.synchronize(dev)
    tim = eng.get_timing()
    eng.set_option("timing", 0)
    total_timed = sum(v["ms"] for v in tim.values())
    ncu = {}
    for name in ("r2_ncu_traffic.json", "r1_gemm_ncu_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):          # dram__bytes_read+write per launch from the committed ncu --set full captures
            with open(tpath) as f:
                ncu = json.load(f)
            ncu["_file"] = "profiles/" + name
            break
    by_cat = {k: round(v["ms"], 4) for k, v in tim.items()}
    whole = (value / world) * ALG_GFLOP_PER_IMAGE * 1e9 / (peak_tf * 1e12)
    D_, T_, Mrows = cfg.embed_dim, cfg.enc_tokens, B * cfg.enc_tokens
    L_, C_, V_, Md_ = 26, cfg.num_classes, cfg.num_tokens, cfg.embed_dim * cfg.dec_mlp_ratio

    def entry(cat, bound, kernel, alg_per_launch_total, unit, traffic_key, note=None):
        """alg_per_launch_total: algorithmic bytes (hbm) or flops (tensor) summed over the category's launches."""
        t = tim.get(cat)
        if not t or t["launches"] == 0 or t["ms"] <= 0:
            return None
        ach = alg_per_launch_total / (t["ms"] * 1e-3) / (1e9 if bound == "hbm" else 1e12)
        peak = peak_hbm if bound == "hbm" else peak_tf
        e = {"bound": bound, "kernel": kernel, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
             "peak_source": f"{peak_src} " + ("hbm_gbs" if bound == "hbm" else "bf16_tflops_sustained"),
             "traffic": ncu.get(traffic_key), "traffic_source": ncu.get("_file"),
             ("bytes_per_launch" if bound == "hbm" else "flops_per_launch"): alg_per_launch_total / t["launches"],
             "launches_per_step": t["launches"], "avg_launch_ms": t["ms"] / t["launches"],
             "share_of_step": t["ms"] / total_timed if total_timed else None,
             "tflops": t["flops"] / (t["ms"] * 1e-3) / 1e12 if t["flops"] else None}
        if note:
            e["note"] = note
        return e

    def fused_bytes(K):      # x += A W^T + b ; xn = LN(x): A (bf16) + W (bf16) + x read and written (fp32) + xn (bf16)
        return Mrows * K * 2 + D_ * K * 2 + 2 * Mrows * D_ * 4 + Mrows * D_ * 2

    n_fused = tim.get("enc_gemm_ln", {}).get("launches", 0)
    # AR kernel, per launch: every step re-reads the cross K/V cache of the batch (it does not fit on chip: B T 2D bf16 =
    # 100.7 MB at bs=512), gathers the (position, token) K/V rows of the context, reads the decoder weights once per
    # cluster pass and writes one logits row per image
    ar_bytes = sum(B * T_ * 2 * D_ * 2 + B * (s + 1) * 2 * D_ * 2 + (3 * D_ * D_ + 2 * D_ * Md_ + C_ * D_) * 2 + B * C_ * 4
                   for s in range(L_))
    entries = [
        entry("enc_gemm", "tensor", "gemm_bf16_tcgen05_kernel (QKV, fc1+GELU, patch embedding)", tim["enc_gemm"]["flops"], "TFLOP/s",
              "avg_dram_bytes_per_launch"),
        entry("enc_gemm_ln", "hbm", "gemm_ln_fused_kernel (attn.proj) / gemm_ln_split_kernel (mlp.fc2): residual GEMM + the following LayerNorm",
              (fused_bytes(D_) + fused_bytes(D_ * cfg.enc_mlp_ratio)) * (n_fused / 2.0), "GB/s", "fused_avg_dram_bytes_per_launch"),
        entry("dec_ar", "hbm", "dec_ar2_kernel (whole AR loop: 26 steps; independent clusters of 6 / 8 CTAs, TMA producer warp)"
              if args.ar_kernel in (-1, 2) else "dec_ar_kernel (whole AR loop, grid barriers)",
              ar_bytes * tim.get("dec_ar", {}).get("launches", 0), "GB/s", "dec_ar_dram_bytes_per_launch",
              note="bytes = 26 x (cross K/V cache of the batch + context K/V rows + decoder weights + logits row); the loop is "
                   "a chain of 26 x 11 dependent phases per cluster (latency-bound: profiles/r2_ar_phase_stamps_bs512.txt), "
                   "tensor view: see tflops"),
        entry("enc_attn", "hbm", "enc_attention_tc_kernel (QK^T, softmax, PV per (image, head))",
              (Mrows * 3 * D_ * 2 + Mrows * D_ * 2) * tim["enc_attn"]["launches"], "GB/s", "attn_dram_bytes_per_launch"),
        entry("dec_gemm", "tensor", "gemm_bf16_tcgen05_kernel (cross K/V projection, refine-pass projections, head)",
              tim["dec_gemm"]["flops"], "TFLOP/s", None),
    ]   # dec_attn / layernorm / other are a few percent of the step: see by_category_ms
    entries = [e for e in entries if e is not None]
    entries.sort(key=lambda e: -(e["share_of_step"] or 0.0))
    kernels = [e for e in entries if (e["share_of_step"] or 0.0) >= 0.10]
    roofline = dict(entries[0])          # headline: the kernel kind with the largest share of the step, over ALL categories
    roofline["by_category_ms"] = by_cat
    roofline["whole_step_frac_of_tensor_peak"] = whole
    roofline["kernels"] = kernels        # every kernel kind >= 10 % of the step
    roofline["timing_note"] = ("shares come from a serialised pass with a CUDA-event pair around every launch (no overlap "
                               "between decoder chains); ms_per_step is the overlapped graph replay")

    # ---- parity of the timed batch (outside the timed region) ----
    parity = None
    if not args.no_parity:
        # `logits` / `ids` still hold the roofline pass over the last timed batch (same inputs, same kernels)
        parity = parity_block(model, cfg, sd, batches_cpu[last_batch], logits, ids,
                              fuse_restore=args.fuse_ln if args.fuse_ln >= 0 else 3)

    # ---- p50 latency at bs=1: engine call with raw pointers, and the reference's protocol (bench.py:43-49: model(x)) ----
    lat = lat_mod = None
    if not args.no_latency and world == 1:
        x1 = synth_images(cfg, 1, 9).to(dev)
        l1 = torch.empty((1, 26, cfg.num_classes), dtype=torch.float32, device=dev)
        i1 = torch.empty((1, 26), dtype=torch.int32, device=dev)
        for _ in range(20):
            eng.forward(x1.data_ptr(), 1, l1.data_ptr(), i1.data_ptr(), steps_t.data_ptr(), st.cuda_stream, None, True, 1)
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(1000):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            eng.forward(x1.data_ptr(), 1, l1.data_ptr(), i1.data_ptr(), steps_t.data_ptr(), st.cuda_stream, None, True, 1)
            b.record(st)
            b.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        lat = {"p50_ms": ts[len(ts) // 2], "p99_ms": ts[int(len(ts) * 0.99) - 1], "iters": len(ts),
               "what": "parseq_forward (device pointers), CUDA events"}
        # module API, host clock around model(x) + synchronize, as torch.utils.benchmark.Timer does for the reference
        with torch.inference_mode():
            for _ in range(20):
                model(x1)
            torch.cuda.synchronize(dev)
            tm = []
            for _ in range(1000):
                t0 = time.perf_counter()
                model(x1)
                torch.cuda.synchronize(dev)
                tm.append((time.perf_counter() - t0) * 1e3)
        tm.sort()
        lat_mod = {"p50_ms": tm[len(tm) // 2], "p99_ms": tm[int(len(tm) * 0.99) - 1], "mean_ms": sum(tm) / len(tm),
                   "iters": len(tm), "what": "model(x) through strhub-compatible PARSeq.forward, host clock + synchronize "
                                             "(reference bench.py:43-49 protocol)"}

    # ---- CPU baseline on this box's host cores (bounded sample) ----
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        sample = 96
        ips, cores, kind, what = cpu_images_per_sec(cfg, sd, sample, 2)
        cpu = {"value": ips, "unit": "images/s", "cores": cores, "kind": kind,
               "sample": f"median of 2 forwards of {sample} images (of the 512-image workload), {what}"}

    line = {
        "metric": "images/sec PARSeq-S 32x128 AR+1refine", "value": value, "unit": "images/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": "PARSeq-S 32x128 94-char max_len=25 bs=512/GPU AR + 1 refine (BASELINE configs[1])",
                   "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world} (batch-sharded, no collective)",
                   "l2": f"inputs rotate over {NROT} resident batches ({NROT * B * 49152 / 1e6:.0f} MB > 126 MB L2)",
                   "chunk": args.chunk or (args.max_batch or 512), "max_batch": args.max_batch or 512, "dec_chunk": args.dec_chunk or 128, "cuda_graph": not args.no_graph},
        "clocks": clocks,
        "e2e": {"value": e2e_val, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1000 * e2e_s / args.steps},
        "e2e_u8": {"value": e2e_u8_val, "unit": "images/s", "h2d_bytes_per_step": h2d // 4, "d2h_bytes_per_step": d2h,
                   "note": "parseq_forward_host_u8: raw uint8 HWC crops, ToTensor+Normalize folded into the patch gather"},
        "e2e_two_in_flight": e2e2,
        "gpu_launches": launches,
        "roofline": roofline,
        "parity": parity,
        "cpu_baseline": cpu,
        "latency_bs1": lat,
        "latency_bs1_module": lat_mod,
        "configs": configs,
        "ids_gather": gather,
    }
    print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
