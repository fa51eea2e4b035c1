#!/usr/bin/env python
"""Benchmark of the Spann3R per-frame forward path (BASELINE.json metric: frames/sec, 10-frame 512x384
sequence through encoder -> memory-attn -> decoder -> DPT).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host CPU cores

One "step" = one whole 10-frame 512x384 sequence (BASELINE config[1]) through `Spann3R.forward` (eval mode,
batch 1 per GPU, spatial memory reset per sequence).  N > 1: one process per GPU (torchrun), every rank runs its
own independent sequences (weak scaling, no data-path collective -- SURVEY.md §8e); time = max over ranks.
Rank 0 prints ONE JSON line.  Keys beyond the base contract: `roofline` (dominant kernel = the split-bf16
tcgen05 GEMM/conv engine, CUDA-event timed per launch in a separate profiling pass), `cpu_baseline` (the oracle
port of the reference on the host cores, bounded sample), `e2e` (same metric with pinned-host inputs copied H2D
and predictions copied D2H inside the timed region), `gpu_launches`, `clocks`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAMES, HEIGHT, WIDTH = 10, 384, 512
FLOP_PER_SEQ = 13.95e12            # algorithmic, SURVEY.md §8a (10 frames, B=1, 512x384)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_sustained=float(d.get("bf16_tflops_sustained", 1454.1)), hbm=float(d.get("hbm_gbs", 6578.3)),
                    src="measured (MEASURED_PEAKS.json, bf16 sustained)")
    return dict(bf16_sustained=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed regions (B200_PROFILING.md recipe).  The process is started
    BEFORE the warm-up (nvidia-smi needs ~0.3 s to deliver its first row; a 5-step run is over by then) and only the rows that
    arrive inside [mark_begin, mark_end] -- the device-timed loop -- are reported; it is stopped before the e2e loop."""

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.t0 = self.t1 = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        t0, t1 = self.t0 or 0.0, (self.t1 or time.time()) + 0.12     # a row describes the 100 ms before it arrives
        rows = [r for t, r in self.rows if t0 <= t <= t1]
        window = "timed regions"
        if not rows and self.rows:      # shorter than one sampling period: the last rows before the end (warm-up load)
            rows, window = [r for _, r in self.rows[-3:]], "last rows before the end of the timed regions"
        sm = sorted(int(float(r[0])) for r in rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 3 + j and r[3 + j].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "window": window}


def _dist():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def _host_threads():
    """Host threads a baseline leg may use: every core this process is allowed on (torchrun exports OMP_NUM_THREADS=1;
    the reference arm is entitled to the whole host).  Physical cores when SMT doubles the count."""
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    return max(1, avail // 2 if avail >= 4 else avail)


def _reference_model(sd):
    """(model, kind): the UNMODIFIED reference `spann3r.model.Spann3R` from the staged copy under baseline/_ref
    (tools/stage_reference.py) on the synthetic checkpoint -> kind "reference"; None when it is not staged."""
    try:
        from baseline import ref_loader
        from spann3r_b200 import synth
        if ref_loader.root() is None:
            return None, "reference not staged under baseline/_ref"
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):     # the reference prints while constructing
            m = ref_loader.build_model(sd, synth.DUST3R_ARGS)
        return m, "reference"
    except Exception as ex:   # a baseline leg must never cost the bench line
        return None, "reference unavailable: " + repr(ex)[:160]


def _cpu_reference_leg(sd, model_ref, budget_s, max_steps):
    """The reference's CPU path on the host cores, on the FULL headline config (one 10-frame 512x384 sequence per step):
    `Spann3R.forward` of the staged reference when available (kind "reference"), else the oracle port (kind "port").
    Runs whole sequences until `budget_s` is spent or `max_steps` are done (at least one)."""
    from spann3r_b200 import synth
    cores = _host_threads()
    os.environ["OMP_NUM_THREADS"] = str(cores)
    torch.set_num_threads(cores)
    frames = synth.make_frames(FRAMES, HEIGHT, WIDTH)
    if model_ref is not None:
        kind = "reference"

        def fwd(fr):
            with torch.no_grad():
                return model_ref(fr)
    else:
        from oracle import spann3r_oracle as orc
        kind = "port"

        def fwd(fr):
            return orc.forward(sd, fr)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()), torch.no_grad():
        fwd(synth.make_frames(2, 224, 224))              # page the weights in (2 s), not a step of the workload
        steps, t0 = 0, time.time()
        while True:
            fwd(frames)
            steps += 1
            if steps >= max_steps or time.time() - t0 > budget_s:
                break
    dt = (time.time() - t0) / steps
    what = "UNMODIFIED reference Spann3R.forward (baseline/_ref)" if kind == "reference" else "oracle port"
    return {"value": FRAMES / dt, "unit": "frames/s", "cores": cores, "kind": kind, "seconds_per_step": dt, "steps": steps,
            "sample": f"{steps} x the full {FRAMES}-frame {WIDTH}x{HEIGHT} sequence (the headline config), {what}, torch CPU fp32, "
                      f"{cores} threads (OMP_NUM_THREADS={cores})"}


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores, same config / metric
    as the CUDA arm.  Rank 0 alone runs it; the other ranks exit without work."""
    rank, world, _ = _dist()
    if rank != 0:
        return
    from spann3r_b200 import synth
    torch.set_num_threads(_host_threads())      # torchrun exports OMP_NUM_THREADS=1; constructing the reference is CPU work too
    sd = synth.make_state_dict(sharpen=True)
    m, why = _reference_model(sd)
    cpu = _cpu_reference_leg(sd, m, budget_s=100.0, max_steps=max(1, args.steps))
    if m is None:
        cpu["note"] = why
    print(json.dumps({
        "impl": "reference", "metric": "frames/sec (512x384, 10-frame seq) enc->mem-attn->dec->DPT", "value": cpu["value"],
        "unit": "frames/s", "n_gpus": args.gpus, "steps": cpu["steps"], "warmup": 1, "ms_per_step": cpu["seconds_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{FRAMES}-frame {WIDTH}x{HEIGHT} sequence per step, batch 1 per GPU, ViT-L enc / ViT-B dec + DPT, "
                               f"random-init sharpened checkpoint (SURVEY.md §8d config 2)",      # the CUDA arm's workload, verbatim
                   "parallelism": "host CPU cores, rank 0 only (the reference's CPU path)"},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def _eager_gpu_legs(mref, why, sd, frames_dev, model, dev, F_):
    """The reference as PyTorch eager on THIS GPU, same frames, batch 1 (SURVEY.md §8d(i)): the staged unmodified
    `Spann3R.forward` with (a) its shipped TF32 default and the PyTorch RoPE fallback it uses when curope is not built,
    (b) strict fp32, (c) TF32 + the reference's OWN curope extension built for sm_100 (tools/stage_reference.py --curope,
    one-token patch) -- the reference's best shot.  Falls back to the oracle port when the reference is not staged.
    Also returns the parity of the CUDA path against the reference's strict-fp32 GPU run on these frames."""
    fr = [{"img": f["img"][:1].contiguous()} for f in frames_dev]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    import contextlib
    import io
    if mref is not None:
        mref = mref.to(dev)
        # the reference caches token positions per (h, w) WITHOUT the device (croco/models/blocks.py:195-207): a model that ran
        # on the CPU first (the cpu_baseline leg) would index with CPU positions on the GPU -- drop the caches, code untouched
        for mod in mref.modules():
            pg = getattr(mod, "position_getter", None)      # a plain object hanging off PatchEmbed, not an nn.Module
            if pg is not None and hasattr(pg, "cache_positions"):
                pg.cache_positions = {}
        what = "UNMODIFIED reference Spann3R.forward (baseline/_ref), PyTorch eager (cuBLAS/cuDNN), batch 1, same frames"

        def fwd(f):
            with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
                return mref(f)
    else:
        from oracle import spann3r_oracle as orc
        sdg = {k: v.to(dev) for k, v in sd.items()}
        what = "oracle port of Spann3R.forward (" + why + "), PyTorch eager, batch 1, same frames"

        def fwd(f):
            return orc.forward(sdg, f)

    def timed(reps=2):
        fwd(fr)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            out = fwd(fr)
        e1.record()
        torch.cuda.synchronize(dev)
        return reps * F_ / (e0.elapsed_time(e1) / 1e3), out

    eager, parity = {}, None
    for name, tf32 in (("tf32_default", True), ("strict_fp32", False)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32
        v, out = timed()
        eager[name] = {"value": v, "unit": "frames/s", "what": what + (", RoPE = the PyTorch fallback" if mref is not None else "")}
        if not tf32:
            # in-run parity: the CUDA path vs the reference's own strict-fp32 forward on this GPU, same frames / weights
            preds, _ = model([{"img": f["img"][:1].contiguous()} for f in frames_dev])
            worst = 0.0
            for p, r in zip(preds, out[0]):
                for k in r:
                    worst = max(worst, float((p[k].double() - r[k].double()).norm() / r[k].double().norm()))
            parity = {"worst_rel_l2": worst, "against": "reference eager strict fp32 on this GPU" if mref is not None
                      else "oracle port strict fp32 on this GPU", "frames": F_, "bar": 1e-3}
    if mref is not None:
        try:
            from baseline import ref_loader
            if not ref_loader.curope_available():
                raise ImportError("baseline/_ref_curope/curope.so not built")
            if ref_loader.CUROPE_DIR not in sys.path:
                sys.path.insert(0, ref_loader.CUROPE_DIR)
            from models.curope.curope2d import cuRoPE2D   # noqa: the reference's own module (staged), now importable
            old = {}
            for name, mod in mref.named_modules():
                r = getattr(mod, "rope", None)
                if r is not None and not isinstance(r, cuRoPE2D):
                    old[name] = r
                    mod.rope = cuRoPE2D(freq=float(getattr(r, "base", 100.0)), F0=float(getattr(r, "F0", 1.0)))
            torch.backends.cuda.matmul.allow_tf32 = True
            torch.backends.cudnn.allow_tf32 = True
            v, out2 = timed()
            eager["tf32_default_curope"] = {"value": v, "unit": "frames/s", "rope_modules_switched": len(old),
                                            "what": "same, RoPE = the reference's own curope CUDA extension built for sm_100 "
                                                    "(kernels.cu:101 one-token patch): the reference's best shot"}
        except Exception as ex:
            eager["tf32_default_curope"] = {"unavailable": repr(ex)[:200]}
        finally:     # hand the model back as it was built (the CPU leg runs the stock fallback)
            mods = dict(mref.named_modules())
            for name, r in locals().get("old", {}).items():
                mods[name].rope = r
    return eager, parity


DUMP_BUDGET = 64_000_000           # bytes written by --dump-outputs at most


def _host_outputs(out):
    """name -> float32 host array of what `Spann3R.forward` returned: preds[i][k] and the res2 half of preds_all[i]
    (their res1 halves are the preds entries themselves)."""
    preds, preds_all = out
    arrays = {f"preds_{i}_{k}": v for i, p in enumerate(preds) for k, v in p.items()}
    arrays.update({f"preds_all_{i}_res2_{k}": v for i, (_, r2) in enumerate(preds_all) for k, v in r2.items()})
    return {n: v.detach().float().cpu().numpy() for n, v in arrays.items()}


def _write_outputs(arrays, out_dir):
    """DIR/<name>.npy; above DUMP_BUDGET every array keeps the same fraction of its elements, at indices drawn with a
    fixed seed (flattened, ascending), so the files of two runs line up element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_BUDGET - 256 * len(arrays)         # room for the .npy headers
    for name, a in arrays.items():
        if total > budget:
            m = max(1, a.size * budget // total)
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, m, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--frames", type=int, default=FRAMES)
    ap.add_argument("--with-eager-gpu", action="store_true", help="(default at N=1 now; kept for old command lines)")
    ap.add_argument("--no-eager-gpu", action="store_true",
                    help="skip the `reference_eager_gpu` leg: the reference ALGORITHM as PyTorch eager on this GPU (the oracle "
                         "port with the reference's TF32 default, and in strict fp32) -- the peer the north star asks to be "
                         "reported beside the CUDA path in the same run.  Untimed for the headline; ~5 s")
    ap.add_argument("--raw-checkpoint", action="store_true",
                    help="random-init weights as constructed (SURVEY.md §8d: ill-conditioned memory reads from the 7th frame on) "
                         "instead of the sharpened checkpoint the headline is quoted on; the work per frame is identical")
    ap.add_argument("--config3", action="store_true",
                    help="BASELINE config[2] as written: 8 x N independent 10-frame sequences (seeds 100 s + i) dealt round-robin to "
                         "the N ranks by shard.run_sharded and advanced 8 per GPU in lockstep (and, for comparison, one by one); "
                         "adds a `config3` object to the JSON line.  Off by default (the headline config is batch 1)")
    ap.add_argument("--no-raw", action="store_true", help="skip the extra `raw_checkpoint` leg (the headline config on the RAW "
                    "random-init checkpoint, SURVEY.md §8d: report both)")
    ap.add_argument("--batch", type=int, default=1,
                    help="sequences advanced in lockstep per GPU (BASELINE config[2] runs 8 per GPU); the headline is 1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy in float32: "
                         "preds_<frame>_<key> and preds_all_<frame>_res2_<key>.  The inputs are seeded, so two builds run with "
                         "the same arguments can be compared file by file.  Above 64 MB in all, every array is reduced to the "
                         "same fixed, seeded sample of its elements")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    rank, world, local = _dist()
    # torchrun exports OMP_NUM_THREADS=1: the one-time host work of every rank (synthetic checkpoint, weight packing, and on
    # rank 0 the baseline legs) gets this rank's share of the host cores instead of one thread
    if os.environ.get("OMP_NUM_THREADS"):
        torch.set_num_threads(max(1, _host_threads() // max(world, 1)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from spann3r_b200 import Spann3R, synth

    W_ = max(args.warmup, 3)
    K = args.steps
    F_ = args.frames
    sd = synth.make_state_dict(sharpen=not args.raw_checkpoint)
    model = Spann3R(dus3r_name=None)
    model.load_state_dict(sd, strict=True)
    model = model.to(dev).eval()

    # per-rank independent sequences (seeds differ per rank and per step)
    BATCH = max(1, args.batch)

    def host_frames(step):
        fr = synth.make_frames(F_, HEIGHT, WIDTH, batch=BATCH, seed0=1 + 1000 * rank + 100 * step)
        return [{"img": f["img"].pin_memory()} for f in fr]

    n_distinct = 2
    host = [host_frames(s) for s in range(n_distinct)]
    resident = [[{"img": f["img"].to(dev)} for f in seq] for seq in host]
    out_host = None

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(dev)

    from spann3r_b200 import shard

    def max_over_ranks(ms):   # spann3r_b200/shard.py (covered by the world_size-2 gloo test)
        return shard.max_over_ranks(ms, device=dev)

    # ---- warm-up (also builds every tensor map / plan) ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(W_):
        model(resident[i % n_distinct])
    eng = model._engine_for(BATCH, HEIGHT, WIDTH, n_frames=F_)
    torch.cuda.synchronize(dev)

    # ---- timed: inputs resident in HBM ----
    eng.take_launches(); eng.take_flops()
    barrier()
    sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        out_last = model(resident[i % n_distinct])
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    # copied out before anything else runs on the model: its outputs may live in buffers the next call reuses
    dumped = _host_outputs(out_last) if args.dump_outputs and rank == 0 else None
    del out_last
    launches = eng.take_launches()
    flops_issued = eng.take_flops()
    # the sampler stops HERE: nvidia-smi polling the driver every 100 ms costs the e2e loop below a third of its throughput
    # (135 vs 196 frames/s, profiles/r2q_bench.json vs r2m_bench.json) -- its queries serialise with the pinned-memory copies
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    value = world * BATCH * F_ * K / (ms / 1e3)

    # ---- timed: end to end through the public API, pinned host inputs -> device, predictions -> pinned host ----
    def e2e_step(seq_host):
        nonlocal out_host
        frames = [{"img": f["img"].to(dev, non_blocking=True)} for f in seq_host]
        preds, _ = model(frames)
        outs = [p[k] for p in preds for k in sorted(p)]
        if out_host is None:
            out_host = [torch.empty(o.shape, dtype=o.dtype, pin_memory=True) for o in outs]
        for o, h in zip(outs, out_host):
            h.copy_(o, non_blocking=True)
        return outs

    e2e_step(host[0])
    torch.cuda.synchronize(dev)
    barrier()
    e0.record()
    for i in range(K):
        outs = e2e_step(host[i % n_distinct])
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    h2d = BATCH * F_ * 3 * HEIGHT * WIDTH * 4
    d2h = sum(o.numel() * 4 for o in outs)
    e2e = world * BATCH * F_ * K / (ms_e2e / 1e3)

    # ---- roofline leg: per-launch CUDA-event timing of the tensor-core kernels (separate, untimed pass) ----
    eng.profile(True)
    model(resident[0])
    prof = eng.profile_read()
    eng.profile(False)
    pk = _peaks()
    gemm_tflops = prof["gemm_flops"] / (prof["gemm_ms"] * 1e-3) / 1e12 if prof["gemm_ms"] > 0 else 0.0
    # DRAM bytes per launch of the GEMM / conv engine from the committed ncu capture of this build (contract: "from one ncu
    # capture, per launch like achieved, or null"); ncu cannot run inside a timed bench, so this is read, not measured here
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        except Exception:
            traffic = None
    roofline = {
        "bound": "tensor", "kernel": "gemm_bf16x3_kernel (split-bf16 tcgen05 GEMM / implicit-GEMM conv)",
        "achieved": gemm_tflops, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": gemm_tflops / pk["bf16_sustained"],
        "traffic": traffic, "traffic_source": traffic_src, "peak_source": pk["src"],
        "note": "achieved = algorithmic 2MNK FLOPs / CUDA-event time summed over all GEMM/conv launches of one sequence; "
                "the split-bf16 scheme issues 3 MMAs per product, so issued-MMA rate = 3x achieved (cap 1/3 of peak).  The per-launch "
                "times come from a SEPARATE profiling pass with CUDA events around every launch (no PDL overlap, DPT side streams "
                "serialised), so gemm_ms_per_seq + attention_ms_per_seq exceeds ms_per_step: they are not in-situ times",
        "gemm_launches_per_seq": prof["gemm_launches"], "gemm_ms_per_seq": prof["gemm_ms"],
        "gemm_flops_per_launch": prof["gemm_flops"] / max(prof["gemm_launches"], 1),
        "attention_ms_per_seq": prof["attn_ms"], "attention_tflops": (prof["attn_flops"] / (prof["attn_ms"] * 1e-3) / 1e12
                                                                       if prof["attn_ms"] > 0 else 0.0),
        "whole_path_frac": (FLOP_PER_SEQ * BATCH * F_ / FRAMES * K * world / (ms / 1e3)) / 1e12 / pk["bf16_sustained"] / world,
    }

    # ---- baseline legs (rank 0, N=1 only; never on the product path).  ONE construction of the staged, unmodified
    # reference model serves the CPU leg and the eager-GPU legs. ----
    cpu, eager, parity_ref = None, None, None
    want_cpu = rank == 0 and world == 1 and not args.no_cpu_baseline
    want_eager = rank == 0 and world == 1 and not args.no_eager_gpu
    if want_cpu or want_eager:
        sd_base = sd
        mref, why = _reference_model(sd_base)
        # GPU legs FIRST: a CPU forward leaves the host's OpenMP pool spinning, which depresses whatever is timed on the GPU
        # right after it (measured: the CUDA arm's own e2e drops from 195 to 138 frames/s under a 64-thread pool,
        # profiles/r2k_e2e_threads.txt) -- the reference's eager-GPU numbers must not pay for its own CPU leg
        if want_eager:
            try:
                eager, parity_ref = _eager_gpu_legs(mref, why, sd_base, resident[0], model, dev, F_)
            except Exception as ex:   # a baseline leg must never cost the bench line
                eager = {"unavailable": repr(ex)[:200]}
            finally:
                torch.backends.cuda.matmul.allow_tf32 = False
                torch.backends.cudnn.allow_tf32 = False
        if want_cpu:
            # the reference's CPU path on the host cores: ONE full 10-frame 512x384 sequence (the headline config)
            try:
                if mref is not None:
                    mref = mref.cpu()
                    for mod in mref.modules():                 # positions cached on the GPU by the legs above
                        pg = getattr(mod, "position_getter", None)
                        if pg is not None and hasattr(pg, "cache_positions"):
                            pg.cache_positions = {}
                        if hasattr(mod, "rope") and getattr(mod.rope, "cache", None) is not None:
                            mod.rope.cache = {}
                cpu = _cpu_reference_leg(sd_base, mref, budget_s=20.0, max_steps=1)
                if mref is None:
                    cpu["note"] = why
            except Exception as ex:
                cpu = {"unavailable": repr(ex)[:200]}
        del mref

    # ---- config 3 as written (SURVEY.md §8d): 8 sequences per GPU through shard.run_sharded, lockstep and one by one ----
    config3 = None
    if args.config3:
        per_gpu = 8
        n_seq = per_gpu * world
        mine = shard.shard_indices(n_seq, world, rank)
        seqs = [None] * n_seq                      # every rank holds the same LIST; only its own sequences carry data
        for s_ in mine:
            seqs[s_] = [{"img": f["img"].to(dev)} for f in synth.make_frames(F_, HEIGHT, WIDTH, seed0=100 * s_ + 1)]
        res3 = {}
        for name, pgb in (("lockstep_b8", per_gpu), ("sequential_b1", 1)):
            fwd = lambda fr: model(fr)             # noqa: E731
            shard.run_sharded(fwd, seqs, per_gpu_batch=pgb, rank=rank, world_size=world)   # warm-up (plans of this batch)
            barrier()
            e0.record()
            out3 = shard.run_sharded(fwd, seqs, per_gpu_batch=pgb, rank=rank, world_size=world)
            e1.record()
            barrier()
            ms3 = max_over_ranks(e0.elapsed_time(e1))
            finite = all(bool(torch.isfinite(v).all()) for preds in out3.values() for p in preds for v in p.values())
            res3[name] = {"frames_per_s": n_seq * F_ / (ms3 / 1e3), "per_gpu_frames_per_s": n_seq * F_ / (ms3 / 1e3) / world,
                          "max_rank_ms": ms3, "sequences": n_seq, "per_gpu_batch": pgb, "finite": finite}
            del out3
        config3 = res3
        del seqs

    # ---- the headline config on the RAW random-init checkpoint (SURVEY.md §8d: run and report both; the sharpened one is
    # the headline).  Same work per frame; the memory reads are ill-conditioned from the 7th frame on. ----
    raw = None
    if rank == 0 and world == 1 and not args.raw_checkpoint and not args.no_raw and BATCH == 1:
        model.norm_q.weight.data.div_(8.0)          # sharpened = raw with norm_q.weight * 8 (synth.make_state_dict)
        model.invalidate_packed()
        for _ in range(2):
            praw, _ = model(resident[0])
        torch.cuda.synchronize(dev)
        e0.record()
        for i in range(3):
            praw, _ = model(resident[i % n_distinct])
        e1.record()
        torch.cuda.synchronize(dev)
        raw = {"value": 3 * F_ / (e0.elapsed_time(e1) / 1e3), "unit": "frames/s", "steps": 3,
               "finite": all(bool(torch.isfinite(v).all()) for p in praw for v in p.values()),
               "what": "same config, raw random-init checkpoint (norm_q.weight not sharpened)"}
        model.norm_q.weight.data.mul_(8.0)
        model.invalidate_packed()

    if dumped is not None:
        _write_outputs(dumped, args.dump_outputs)
    if rank == 0:
        print(json.dumps({
            "reference_eager_gpu": eager, "parity_vs_reference_in_run": parity_ref, "raw_checkpoint": raw, "config3": config3,
            "metric": "frames/sec (512x384, 10-frame seq) enc->mem-attn->dec->DPT", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": K, "warmup": W_, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate; tf32 attention)", "data": "synthetic",
            "config": {"workload": f"{F_}-frame {WIDTH}x{HEIGHT} sequence per step, batch {BATCH} per GPU, ViT-L enc / ViT-B dec + DPT, "
                                   f"random-init {'raw' if args.raw_checkpoint else 'sharpened'} checkpoint (SURVEY.md §8d config 2)",
                       "parallelism": f"{world} independent replicas (one sequence stream per GPU, no collective)",
                       "l2": "per-step working set (2.6 GB packed weights + activations) >> 126 MB L2; inputs alternate between "
                             "2 distinct sequences"},
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / K},
            "gpu_launches": launches, "issued_algorithmic_tflop_per_step": flops_issued / K / 1e12,
            "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
        }))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
