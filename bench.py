#!/usr/bin/env python
"""
bench.py — 16384-sample frames/s of the Wave-U-Net forward (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--precision fp32|bf16|auto] [--dump-outputs DIR]
    python bench.py --impl reference ...        # the reference's CPU implementation of the path (host cores)
    python bench.py --mode train   [--batch 64] # SURVEY §8f N1 / configs[4]: fwd + bwd + Adam per step, grads all-reduced
    python bench.py --mode enhance              # configs[3]: 10 s clips through enhance_waveforms, 1024 frames/step sharded
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W   # one rank per GPU, batch sharded, no collective on the path

A "step" is one forward over one batch of B synthetic frames per GPU ([B,1,16384] fp32, eval mode). --steps is the number
of timed steps in every mode. --dump-outputs DIR writes what the last timed forward returned on rank 0 to DIR/output.npy
(float32); the weights and inputs are seeded, so two builds run with the same arguments can be compared output for output.
Workload at N=1 = BASELINE.json configs[2] shape (batch 256, 16384 samples, 12 levels); weak scaling:
every rank runs the same B.  One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

N_LAYERS, CH_INT, T = 12, 24, 16384
METRIC = "16384-sample frames/sec forward"


# ------------------------------------------------------------------------------------------------
# roofline model (SURVEY §8d): algorithmic flops / bytes per block for a batch of B frames
# ------------------------------------------------------------------------------------------------
def block_table(B: int, esize: int):
    """[(name, flops, bytes)] for the 2n+1 conv blocks (+ the head folded into the last decoder).
    bytes = fused-minimum traffic: read inputs once, write the output once, weights once per batch."""
    n, ci = N_LAYERS, CH_INT
    rows = []
    enc_out = [(i + 1) * ci for i in range(n)]
    for i in range(n):
        cin = 1 if i == 0 else i * ci
        cout = enc_out[i]
        L = T >> i
        flops = 2.0 * cin * cout * 15 * L * B
        in_b = (4 if i == 0 else esize) * cin * L            # raw fp32 input for enc0, else even half of skip_{i-1}
        byts = B * (in_b + esize * cout * L) + esize * cin * cout * 15
        rows.append((f"enc{i}", flops, byts))
    L = T >> n
    c = n * ci
    rows.append(("middle", 2.0 * c * c * 15 * L * B, B * 2 * esize * c * L + esize * c * c * 15))
    cprev = c
    for j in range(n):
        e = n - 1 - j
        cskip = enc_out[e]
        cout = enc_out[e]
        L = T >> e
        cin = cprev + cskip
        flops = 2.0 * cin * cout * 5 * L * B
        reads = esize * (cprev * (L // 2) + cskip * L)
        writes = esize * cout * L
        if j == n - 1:                                        # head fused: + raw input read, 1-channel fp32 write
            flops += 2.0 * (cout + 1) * L * B
            reads += 4 * L
            writes = 4 * L
        rows.append((f"dec{j}" + ("+out" if j == n - 1 else ""), flops, B * (reads + writes) + esize * cin * cout * 5))
        cprev = cout
    return rows


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tensor_tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json; bf16 sustained, kernels timed inside a long step)"}
    return {"hbm_gbs": 6650.0, "tensor_tflops": 1400.0, "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU baseline: the reference forward restated with torch ops (oracle/wunet_oracle.torch_port_forward)
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(iters: int, warmup: int):
    """BASELINE.json configs[0] (batch 1) and a batch of 8 frames, fp32, on the host cores: the thread count is chosen by a
    short sweep and set explicitly (under torch.distributed.run the environment carries OMP_NUM_THREADS=1), then `iters` timed
    forwards per batch size; best and median are reported, `value` = the better of the two batch sizes by its MEDIAN."""
    from oracle import wunet_oracle as wo
    st = {k: torch.from_numpy(np.asarray(v)) for k, v in wo.make_state(N_LAYERS, CH_INT, seed=0).items()}
    ncpu = os.cpu_count() or 1
    cands = sorted({t for t in (8, 16, 32, 64) if t <= ncpu} | {min(ncpu, 8)})
    out = {}
    with torch.no_grad():
        for fps in (1, 8):
            x = torch.from_numpy(wo.make_input(fps, T, seed=1234))
            sweep = {}
            for th in cands:
                torch.set_num_threads(th)
                for _ in range(2):
                    wo.torch_port_forward(st, x)
                ts = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    wo.torch_port_forward(st, x)
                    ts.append(time.perf_counter() - t0)
                sweep[th] = min(ts)
            best_th = min(sweep, key=sweep.get)
            torch.set_num_threads(best_th)
            for _ in range(max(3, warmup)):
                wo.torch_port_forward(st, x)
            ts = []
            for _ in range(iters):
                t0 = time.perf_counter()
                wo.torch_port_forward(st, x)
                ts.append(time.perf_counter() - t0)
            ts.sort()
            out[fps] = {"batch": fps, "threads": best_th, "iters": len(ts), "best_ms": round(1e3 * ts[0], 3),
                        "median_ms": round(1e3 * ts[len(ts) // 2], 3), "frames_per_s_best": round(fps / ts[0], 2),
                        "frames_per_s_median": round(fps / ts[len(ts) // 2], 2),
                        "thread_sweep_ms": {str(k): round(1e3 * v, 2) for k, v in sweep.items()}}
    top = max(out.values(), key=lambda r: r["frames_per_s_median"])
    return {"value": top["frames_per_s_median"], "unit": "frames/s", "cores": top["threads"], "kind": "port",
            "sample": f"{top['iters']} forwards of B={top['batch']} x 16384 samples (median), fp32, torch CPU ops (oneDNN) "
                      f"restating model/unet_basic.py:77-100, {top['threads']} threads (best of a sweep over {cands}) of {ncpu} cpus",
            "ms_per_step": top["median_ms"], "steps_done": top["iters"], "frames_per_step": top["batch"],
            "batch1": out[1], "batch8": out[8]}


# ------------------------------------------------------------------------------------------------
# incumbent on the same GPU: PyTorch eager (cuDNN / ATen) of the reference's forward, eval mode (SURVEY §8d, BASELINE.md §4)
# ------------------------------------------------------------------------------------------------
def incumbent_run(st, B, dev, iters=5, warm=3):
    from wave_u_net_for_speech_enhancement_b200 import Model
    m = Model(N_LAYERS, CH_INT, train_backend="torch")
    m.load_state_dict(st, strict=True)
    m = m.to(dev).eval()
    x = 0.3 * torch.randn(B, 1, T, device=dev)
    res = {"what": "torch eager (cuDNN convolutions, ATen batch_norm / leaky_relu / interpolate / cat), the op sequence of "
                   "model/unet_basic.py:77-100 via Model._forward_torch_reference_semantics, eval mode, same GPU",
           "batch": B, "cudnn": torch.backends.cudnn.version()}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    try:
        for mode in ("fp32", "tf32", "bf16_autocast"):
            torch.backends.cudnn.allow_tf32 = mode != "fp32"
            torch.backends.cuda.matmul.allow_tf32 = mode != "fp32"

            def run():
                with torch.no_grad():
                    if mode == "bf16_autocast":
                        with torch.autocast("cuda", dtype=torch.bfloat16):
                            return m._forward_torch_reference_semantics(x)
                    return m._forward_torch_reference_semantics(x)
            for _ in range(warm):
                run()
            torch.cuda.synchronize()
            ts = []
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(iters):
                e0.record()
                run()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ts.sort()
            res[mode] = {"best_ms": round(ts[0], 3), "median_ms": round(ts[len(ts) // 2], 3),
                         "frames_per_s": round(B / ts[len(ts) // 2] * 1e3, 1)}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
    del m, x
    torch.cuda.empty_cache()
    return res


DUMP_LIMIT = 64 * 10**6                                      # bytes written by --dump-outputs


def dump_output(out_dir: str, y: torch.Tensor) -> None:
    """y ([B,1,T], what model(x) returned) as out_dir/output.npy in float32. Above DUMP_LIMIT a fixed, seeded sample of the
    frames is written instead, and their indices (ascending) as out_dir/output_frames.npy in float64."""
    os.makedirs(out_dir, exist_ok=True)
    a = y.detach().float().cpu().numpy()
    keep = DUMP_LIMIT // (a[0].nbytes + 8)
    if keep < len(a):
        frames = np.sort(np.random.default_rng(0).choice(len(a), size=keep, replace=False))
        np.save(os.path.join(out_dir, "output_frames.npy"), frames.astype(np.float64))
        a = a[frames]
    np.save(os.path.join(out_dir, "output.npy"), a)


def time_steps(fn, steps, warm=3):
    """ms per call of fn() over `steps` back-to-back calls (CUDA events on the current stream)"""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def ncu_traffic(level: str, version: str):
    """DRAM bytes per launch of one block from the committed ncu capture, but ONLY if that capture was taken from the build
    that is running now (the summary CSV carries the library's source hash); otherwise (None, reason)."""
    import csv
    import glob
    import re
    m = re.search(r"src ([0-9a-f]+)", version)
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_conv_tc_*summary.csv")))
    if not m or not cands:
        return None, "no ncu summary under profiles/"
    path = cands[-1]
    text = open(path).read()
    if ("build " + m.group(1)) not in text:
        return None, f"{os.path.basename(path)} was captured from a different build"
    try:
        rows = [r for r in csv.reader(text.splitlines()) if r and not r[0].startswith("#")]
        hdr = rows[0]
        for r in rows[1:]:
            if r[0] == level:
                return (float(r[hdr.index("dram_rd_MB")]) + float(r[hdr.index("dram_wr_MB")])) * 1e6, os.path.basename(path)
    except Exception:  # noqa: BLE001
        pass
    return None, f"{level} not in {os.path.basename(path)}"


def run_train(ctx):
    """SURVEY §8f row N1 / BASELINE.json configs[4]: one step = forward (train-mode BatchNorm) + MSE + backward + Adam on a
    batch of B frames per GPU (trainer/trainer.py:34-38, train.py:31-35); under torchrun the gradients are averaged over the
    ranks inside backward() (one flat 40.5 MB bucket, NCCL, two overlapped parts)."""
    args, rank, world, dev, dist, emit, st = (ctx[k] for k in ("args", "rank", "world", "dev", "dist", "emit", "st"))
    from wave_u_net_for_speech_enhancement_b200 import Model, _lib
    from wave_u_net_for_speech_enhancement_b200.train_step import GradientBucket
    B = args.batch or 64
    steps = args.steps
    model = Model(N_LAYERS, CH_INT)
    model.load_state_dict(st, strict=True)
    model = model.to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, betas=(0.9, 0.999))
    loss_fn = torch.nn.MSELoss()
    gen = torch.Generator(device=dev).manual_seed(100 + rank)
    NBUF = 2
    clean = [0.1 * torch.randn(B, 1, T, device=dev, generator=gen) for _ in range(NBUF)]
    noisy = [c + 0.05 * torch.randn(B, 1, T, device=dev, generator=gen) for c in clean]
    clean_h = [c.cpu().pin_memory() for c in clean]
    noisy_h = [c.cpu().pin_memory() for c in noisy]

    def step(i):
        opt.zero_grad()
        loss = loss_fn(clean[i % NBUF], model(noisy[i % NBUF]))          # trainer/trainer.py:35-36
        loss.backward()
        opt.step()
        return loss

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(2, min(args.warmup, 3))):
        step(i)
    barrier()
    sampler = ClockSampler(ctx["local_rank"]) if rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        loss = step(i)
    e1.record()
    torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    barrier()
    clocks = sampler.stop() if sampler else None
    # end to end like the unchanged trainer loop: host batches (pinned), .to(device) every step, loss.item() every step
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        mixture = noisy_h[i % NBUF].to(dev, non_blocking=True)
        target = clean_h[i % NBUF].to(dev, non_blocking=True)
        opt.zero_grad()
        l2 = loss_fn(target, model(mixture))
        l2.backward()
        opt.step()
        float(l2.item())
    torch.cuda.synchronize()
    dt_e2e = time.perf_counter() - t0
    # phases of one step (events), and the all-reduce alone on the flat bucket
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    opt.zero_grad()
    ev[0].record()
    out = model(noisy[0])
    l3 = loss_fn(clean[0], out)
    ev[1].record()
    l3.backward()
    ev[2].record()
    opt.step()
    ev[3].record()
    torch.cuda.synchronize()
    phases = {"forward_ms": round(ev[0].elapsed_time(ev[1]), 3), "backward_ms": round(ev[1].elapsed_time(ev[2]), 3),
              "adam_ms": round(ev[2].elapsed_time(ev[3]), 3)}
    comm = None
    if dist is not None:
        bucket = GradientBucket([p.shape for p in model.parameters()], 2 * N_LAYERS + 1, dev)
        def ar():
            bucket.reduce_part(0)
            bucket.reduce_part(1)
            bucket.finish()
        comm = {"allreduce_ms_alone": round(time_steps(ar, 10), 4), "bucket_bytes": bucket.flat.numel() * 4,
                "backend": dist.get_backend(), "nranks": dist.get_world_size(),
                "overlap": "part 0 (head + decoder gradients) is reduced while part 1 (middle + encoders) is computed"}
    # incumbent on the same GPU (rank 0, single-GPU runs): the same step with PyTorch eager (cuDNN) kernels and autograd
    incumbent = None
    if world == 1 and not args.no_incumbent:
        del model, opt
        torch.cuda.empty_cache()
        mt = Model(N_LAYERS, CH_INT, train_backend="torch")
        mt.load_state_dict(st, strict=True)
        mt = mt.to(dev).train()
        ot = torch.optim.Adam(mt.parameters(), lr=1e-3, betas=(0.9, 0.999))
        torch.backends.cudnn.benchmark = True

        def tstep(i):
            ot.zero_grad()
            lt = loss_fn(clean[i % NBUF], mt(noisy[i % NBUF]))
            lt.backward()
            ot.step()
        incumbent = {"what": "the same step with PyTorch eager: cuDNN convolutions (TF32 allowed, torch default), ATen BatchNorm / "
                             "interpolate / cat, autograd, torch.optim.Adam", "batch": B}
        for tf32 in (True, False):
            torch.backends.cudnn.allow_tf32 = tf32
            ms_inc = time_steps(lambda: tstep(0), 5, warm=2)
            incumbent["tf32" if tf32 else "fp32"] = {"ms_per_step": round(ms_inc, 3), "frames_per_s": round(B / ms_inc * 1e3, 1)}
        torch.backends.cudnn.allow_tf32 = True
    t = torch.tensor([ms_total, dt_e2e], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    ms_per_step = float(t[0]) / steps
    line = {"metric": "training samples/sec (16384-sample frames; fwd + bwd + Adam)", "value": B * world * steps / (float(t[0]) / 1e3),
            "unit": "frames/s", "n_gpus": world, "steps": steps, "warmup": max(2, min(args.warmup, 3)), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"unet_basic train step (train.py / trainer.py:34-38): batch {B}/GPU x 16384 samples, {N_LAYERS} levels, "
                                   f"{CH_INT} base filters, MSELoss, Adam(1e-3, 0.9, 0.999), train-mode BatchNorm (per-rank statistics)",
                       "global_batch": B * world, "parallelism": f"dp{world}: one process per GPU, gradients averaged by one flat-bucket "
                                                                   f"all-reduce inside backward()" if world > 1 else "dp1",
                       "l2": "activations + gradients of a step: > 5 GB >> 126 MB L2"},
            "clocks": clocks, "phases": phases, "comm": comm, "incumbent": incumbent, "final_loss": float(loss.detach()),
            "e2e": {"value": B * world * steps / float(t[1]), "unit": "frames/s", "h2d_bytes_per_step": 2 * B * T * 4,
                    "d2h_bytes_per_step": 4, "api": "the unchanged trainer loop's calls: .to(device) of pinned (mixture, clean), "
                                                    "model(mixture), loss(clean, enhanced), backward(), optimizer.step(), loss.item()"},
            "gpu_launches": None, "library": _lib.load().wunet_version().decode(),
            "note": "fp32 CUDA-core training kernels (csrc/wunet_train.cu); optimizer = torch.optim.Adam (the caller's, unchanged)"}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


def run_enhance(ctx):
    """BASELINE.json configs[3]: synthetic 10 s @ 16 kHz clips (160000 samples -> 10 frames after zero padding, exactly
    enhancement.py:57-62) through enhance_waveforms; one step = 1024 frames over all GPUs (128 frames/GPU at 8), clips dealt
    to the ranks, no collective."""
    args, rank, world, dev, dist, emit, st = (ctx[k] for k in ("args", "rank", "world", "dev", "dist", "emit", "st"))
    from wave_u_net_for_speech_enhancement_b200 import Model, _lib, enhance
    per_gpu = args.batch or 128
    steps = args.steps
    clips_per_step = max(1, (per_gpu * world) // 10)
    rng = np.random.default_rng(7)
    clips = [(0.3 * rng.standard_normal(160000)).astype(np.float32) for _ in range(min(clips_per_step, 16))]
    clips = [clips[i % len(clips)] for i in range(clips_per_step)]
    model = Model(N_LAYERS, CH_INT, precision="bf16" if args.precision in ("auto", "bf16") else "fp32")
    model.load_state_dict(st, strict=True)
    model = model.to(dev).eval()

    def step():
        return enhance.enhance_waveforms_sharded(model, clips, rank, world, batch_frames=per_gpu)

    for _ in range(2):
        res = step()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    # same call returning views of the pinned output buffer instead of fresh arrays (valid until the next call)
    t1 = time.perf_counter()
    for _ in range(steps):
        enhance.enhance_waveforms_sharded(model, clips, rank, world, batch_frames=per_gpu, copy=False)
    torch.cuda.synchronize()
    dt_views = time.perf_counter() - t1
    t = torch.tensor([dt, dt_views], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        frames = clips_per_step * 10
        emit({"metric": "10 s clips/sec through enhance_waveforms (enhancement.py:49-74 batched)", "value": clips_per_step * steps / float(t[0]),
              "unit": "clips/s", "frames_per_s": frames * steps / float(t[0]), "n_gpus": world, "steps": steps, "warmup": 2,
              "ms_per_step": 1e3 * float(t[0]) / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
              "dtype": model.precision, "data": "synthetic",
              "config": {"workload": f"{clips_per_step} clips x 160000 samples per step = {frames} frames, {per_gpu} frames/GPU batches, "
                                     f"host waveforms in, host waveforms out (padding, framing, pinned staging, H2D, kernels, D2H, trimming inside the timed region)",
                         "parallelism": f"dp{world}: clips dealt to the ranks by frame count, no collective"},
              "views_out": {"value": clips_per_step * steps / float(t[1]), "unit": "clips/s",
                            "note": "copy=False: results are views of the pooled pinned output buffer"},
              "host_threads": enhance.HOST_THREADS,
              "clips_on_rank0": len(res), "library": _lib.load().wunet_version().decode()})
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--mode", default="forward", choices=["forward", "train", "enhance"])
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (default 256 forward, 64 train, 128 enhance)")
    ap.add_argument("--no-incumbent", action="store_true")
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "bf16"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output of the last timed forward to DIR/output.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode != "forward" or args.impl != "b200"):
        ap.error("--dump-outputs applies to the forward of the b200 implementation (--mode forward --impl b200)")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # libraries (NCCL's version banner, ...) write to fd 1; keep the real stdout for the ONE JSON line only
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    def emit(obj):
        real_stdout.write(json.dumps(obj) + "\n")
        real_stdout.flush()

    # --------------------------------------------------------------------------------------------
    # reference arm: the reference's CPU implementation of the path, on the host cores (rank 0 only)
    # --------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference_run(iters=args.steps, warmup=args.warmup)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "frames/s", "n_gpus": args.gpus,
                "steps": r["steps_done"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"unet_basic forward, {N_LAYERS} levels, {CH_INT} base filters, 16384 samples, "
                                       f"bounded sample of {r['frames_per_step']} frame(s)/step on CPU (BASELINE.json configs[0] is "
                                       f"batch 1; batch 1 and 8 are both timed, the faster is the value)"},
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "batch1", "batch8")},
                "e2e": {"value": r["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return

    # --------------------------------------------------------------------------------------------
    # B200 arm
    # --------------------------------------------------------------------------------------------
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback on the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from oracle import wunet_oracle as wo                    # synthetic weights/inputs + cpu_baseline only
    from wave_u_net_for_speech_enhancement_b200 import Model, _lib

    st = {k: torch.from_numpy(np.asarray(v)) for k, v in wo.make_state(N_LAYERS, CH_INT, seed=0).items()}
    ctx = {"args": args, "rank": rank, "world": world, "local_rank": local_rank, "dev": dev, "dist": dist, "emit": emit,
           "st": st, "wo": wo}
    if args.mode == "train":
        return run_train(ctx)
    if args.mode == "enhance":
        return run_enhance(ctx)
    B = args.batch or 256
    precision = args.precision
    if precision == "auto":
        precision = "bf16"

    def make(prec):
        m = Model(N_LAYERS, CH_INT, precision=prec)
        m.load_state_dict(st, strict=True)
        return m.to(dev).eval()

    model = make(precision)
    # rotating device-resident inputs (the per-step working set, >3 GB of activations, is far larger than L2)
    NBUF = 4
    xs = [torch.from_numpy(wo.make_input(B, T, seed=1234 + 17 * rank + i)).to(dev) for i in range(NBUF)]
    try:
        with torch.no_grad():
            model(xs[0])
        torch.cuda.synchronize()
    except _lib.WunetError as e:
        if args.precision == "auto" and "not built yet" in str(e):
            precision = "fp32"
            model = make(precision)
        else:
            raise

    def step(i):
        with torch.no_grad():
            return model(xs[i % NBUF])

    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    launches_per_step = model.last_launch_count()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if sampler:
        sampler.start()
    e0.record()
    for i in range(args.steps):
        y = step(i)
    e1.record()
    torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    # the timed region is tens of milliseconds; nvidia-smi samples every 100 ms. Keep issuing the identical step (untimed)
    # for ~1.2 s so that the clock / throttle record is taken under the same load.
    t_load = time.perf_counter()
    extra = 0
    while time.perf_counter() - t_load < 1.2:
        for i in range(args.steps):
            step(i)
        torch.cuda.synchronize()
        extra += args.steps
    barrier()
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["note"] = f"sampled every 100 ms over the timed steps plus {extra} identical untimed steps"
    t = torch.tensor([ms_total], device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = B * world * args.steps / (ms_total / 1e3)

    # ---- per-level device times (CUDA events on the launch stream, same K steps) -> roofline ------------
    model.profile(True)
    per_block = None
    for i in range(args.steps):
        step(i)
        ms = np.array(model.profile_read())
        per_block = ms if per_block is None else per_block + ms
    model.profile(False)
    per_block = per_block / args.steps
    peaks = load_peaks()
    esize = 2 if precision == "bf16" else 4
    tab = block_table(B, esize)
    blk_ms = list(per_block[:len(tab)])
    if len(per_block) > len(tab):
        blk_ms[-1] += float(per_block[len(tab)])              # separate head launch belongs to dec11+out
    levels = []
    for (name, flops, byts), t_ms in zip(tab, blk_ms):
        t_mem = byts / (peaks["hbm_gbs"] * 1e9) * 1e3
        t_ten = flops / (peaks["tensor_tflops"] * 1e12) * 1e3
        bound = "hbm" if t_mem >= t_ten else "tensor"
        levels.append({"level": name, "ms": round(float(t_ms), 5), "roof_ms": round(max(t_mem, t_ten), 5), "bound": bound,
                       "gbs": round(byts / (t_ms * 1e-3) / 1e9, 1), "tflops": round(flops / (t_ms * 1e-3) / 1e12, 2),
                       "frac": round(max(t_mem, t_ten) / float(t_ms), 4)})
    dom = max(range(len(tab)), key=lambda i: blk_ms[i])
    dname, dflops, dbytes = tab[dom]
    d = levels[dom]
    if d["bound"] == "hbm":
        roof = {"bound": "hbm", "achieved": d["gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(d["gbs"] / peaks["hbm_gbs"], 4)}
    else:
        roof = {"bound": "tensor", "achieved": d["tflops"], "peak": peaks["tensor_tflops"], "unit": "TFLOP/s",
                "frac": round(d["tflops"] / peaks["tensor_tflops"], 4)}
    traffic, traffic_src = ncu_traffic(dname.split("+")[0], _lib.load().wunet_version().decode()) if (precision == "bf16" and B == 256) else (None, None)
    roof.update({"kernel": dname, "kernel_ms": d["ms"], "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": dbytes,
                 "algorithmic_flops": dflops, "peak_source": peaks["source"],
                 "net_frac": round(sum(l["roof_ms"] for l in levels) / sum(l["ms"] for l in levels), 4),
                 "sum_levels_ms": round(float(sum(blk_ms)), 4)})

    # ---- end to end: public API with HOST buffers (pinned); every step copies ITS inputs H2D and ITS result D2H inside
    # the timed region. (a) streaming API Model.forward_host_stream: two batches in flight, so the copies of step k+1 / k-1
    # overlap the kernels of step k (the way enhancement.py's many chunks are served); (b) one synchronous forward_host per step.
    NH = 4
    xh = [torch.from_numpy(wo.make_input(B, T, seed=99 + i)).pin_memory() for i in range(NH)]
    yh = [torch.empty_like(xh[0]).pin_memory() for _ in range(NH)]
    for i in range(2):
        model.forward_host(xh[i % NH], out=yh[i % NH])
    for _ in model.forward_host_stream([xh[i % NH] for i in range(3)], [yh[i % NH] for i in range(3)]):
        pass
    barrier()
    t0 = time.perf_counter()
    for _ in model.forward_host_stream((xh[i % NH] for i in range(args.steps)), (yh[i % NH] for i in range(args.steps))):
        pass
    torch.cuda.synchronize()
    dt_stream = time.perf_counter() - t0
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        model.forward_host(xh[i % NH], out=yh[i % NH])
    torch.cuda.synchronize()
    dt_sync = time.perf_counter() - t0
    t = torch.tensor([dt_stream, dt_sync], device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = B * world * args.steps / float(t[0].item())
    e2e_sync = B * world * args.steps / float(t[1].item())
    nbytes = B * T * 4

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    cpu = None
    extras = {}
    if world == 1:
        # batch-1 latency, the call shape of enhancement.py:64-66 (one chunk per forward): eager launches and a CUDA graph of
        # the same launch sequence (the shim's launches are stream-ordered and capturable)
        x1 = xs[0][:1].contiguous()
        with torch.no_grad():
            lat = {"eager_ms": round(time_steps(lambda: model(x1), 200), 4)}
            try:
                g = torch.cuda.CUDAGraph()
                model(x1)
                torch.cuda.synchronize()
                with torch.cuda.graph(g):
                    yg = model(x1)
                lat["graph_ms"] = round(time_steps(g.replay, 200), 4)
                lat["graph_matches_eager"] = bool(torch.equal(yg, model(x1)))
            except Exception as e:  # noqa: BLE001 - report, do not hide
                lat["graph_error"] = str(e)[:200]
            lat["launches"] = model.last_launch_count()
            lat["precision"] = precision
        extras["latency_b1"] = lat
        # BASELINE.json configs[1]: fp32 (<= 1e-4 path), batch 64. CUDA-core FFMA: its ceiling is the FFMA rate, not the
        # tensor peak (148 SMs x 128 lanes x 2 flop x sm_max_mhz; theoretical, not driver-measured)
        m32 = make("fp32")
        x64 = xs[0][:64].contiguous()
        with torch.no_grad():
            ms32 = time_steps(lambda: m32(x64), 10)
        flops64 = sum(f for _n, f, _b in block_table(64, 4))
        ffma_peak = 148 * 128 * 2 * 1965e6
        extras["fp32_config2"] = {"workload": "unet_basic forward fp32 (FFMA path, <= 1e-4 vs the reference), batch 64 x 16384 samples",
                                  "value": round(64 / ms32 * 1e3, 1), "unit": "frames/s", "ms_per_step": round(ms32, 4),
                                  "roofline": {"bound": "ffma", "achieved": round(flops64 / (ms32 * 1e-3) / 1e12, 2),
                                               "peak": round(ffma_peak / 1e12, 1), "unit": "TFLOP/s",
                                               "frac": round(flops64 / (ms32 * 1e-3) / ffma_peak, 4),
                                               "peak_source": "theoretical FFMA rate at sm_max_mhz (not driver-measured)"}}
        del m32
        # the same <= 1e-4 contract on the tensor cores: split precision (bf16 hi + lo, three tcgen05 MMAs per product)
        try:
            mtc = make("fp32_tc")
            with torch.no_grad():
                ms_tc64 = time_steps(lambda: mtc(x64), 10)
                ms_tc = time_steps(lambda: mtc(xs[0]), 10)
            extras["fp32_tc"] = {"workload": "unet_basic forward, split-precision tcgen05 path (<= 1e-4 vs the reference)",
                                 "batch64": {"value": round(64 / ms_tc64 * 1e3, 1), "unit": "frames/s", "ms_per_step": round(ms_tc64, 4)},
                                 f"batch{B}": {"value": round(B / ms_tc * 1e3, 1), "unit": "frames/s", "ms_per_step": round(ms_tc, 4)}}
            del mtc
        except Exception as e:  # noqa: BLE001 - report, do not hide
            extras["fp32_tc"] = {"error": str(e)[:200]}
        if not args.no_incumbent:
            extras["incumbent"] = incumbent_run(st, B, dev)
            extras["incumbent"]["speedup_vs_best_mode"] = round(value / max(extras["incumbent"][k]["frames_per_s"]
                                                                             for k in ("fp32", "tf32", "bf16_autocast")), 1)
        if not args.no_cpu_baseline:
            r = cpu_reference_run(iters=20, warmup=2)
            cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "batch1", "batch8")}

    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": f"unet_basic forward, batch {B}/GPU x 16384 samples, {N_LAYERS} levels, {CH_INT} base "
                               f"filters, eval-mode BatchNorm, {precision} path",
                   "global_batch": B * world, "parallelism": f"dp{world} (batch sharded, no collective on the forward)",
                   "kernel_forms": "WUNET_TC_PAIR=%s WUNET_TC_ENC0=%s (defaults: block 1 over pairs of positions, block 0 on CUDA cores)"
                                   % (os.environ.get("WUNET_TC_PAIR", "1"), os.environ.get("WUNET_TC_ENC0", "0")),
                   "l2": f"{NBUF} rotating input batches; per-step activation working set "
                         f"{sum(b for _n, _f, b in tab) / 2**30:.2f} GiB >> 126 MB L2"},
        "clocks": clocks,
        "e2e": {"value": e2e_val, "unit": "frames/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
                "api": "Model.forward_host_stream -> wunet_stream_submit/wait: pinned host buffers in and out every step, "
                       "two batches in flight",
                "sync_value": e2e_sync, "sync_api": "Model.forward_host -> wunet_forward_host (one blocking call per step)"},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roof,
        "levels": levels,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    line.update(extras)
    line["library"] = _lib.load().wunet_version().decode()
    if args.dump_outputs:
        dump_output(args.dump_outputs, y)
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
