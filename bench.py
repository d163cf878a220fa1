#!/usr/bin/env python
"""bench.py -- SDF points/sec of the DISN hot path (BASELINE.json metric: 256^3 grid, 1/2/4/8 x B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 0|1|2|4] [--precision P]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic 137x137 images: encode (resize + VGG-16 + the folds)
then the dense (res+1)^3 SDF grid per image (projection + multi-scale gather + two-stream MLP + /10).

    --config 1 (default; with --gpus N > 1 it is BASELINE config 3): single image, --sdf_res 256 (257^3 points).
    --config 0: single image, --sdf_res 64 (the reference's own CPU-runnable case, 2 chunks of 137 313 points).
    --config 2: batch of 8 images, --sdf_res 128 (8 x 129^3 points), VGG on tcgen05; adds the encoder's images/s.
    --config 4: single image, --sdf_res 512 (513^3 points) + CUDA marching-cubes post-pass on rank 0 inside the step.

With N GPUs the grid's z-slabs are sharded across ranks (strong scaling: total work fixed), every rank re-encodes the
image; for `value` every rank's kernel stores its slab straight into rank 0's HBM over NVLink (CUDA IPC peer stores from the
epilogue; `--gather nccl` uses an NCCL gather instead), inside the timed region.

`value`  : device-resident throughput (image + camera already in HBM; CUDA events on the launch stream, max over ranks).
`e2e`    : the same metric through the public host-buffer API -- disn_encode(host image) + disn_eval_grid(host grid) with
           caller-pinned buffers: the image crosses PCIe inside the step and the kernel's epilogue stores the SDF straight
           into the pinned host grid (no device staging, no trailing copy).  With N > 1 every rank writes its slab into one
           shared pinned host grid (POSIX shared memory registered with cudaHostRegister), each over its own PCIe link.
`--dump-outputs DIR`: after the timed steps, what the last one returned is written as .npy files (see dump_outputs); the
           inputs are seeded, so two builds run with the same arguments can be compared output for output.
`--impl reference`: the CPU oracle restating the reference's TF graph (TF itself is not installable here), all host
           threads, reference loop structure (whole graph incl. VGG per chunk).  Each step is a bounded sample of the SAME
           workload: one full chunk as the reference executes it (config 0: the whole 2-chunk job).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_ALG = 2164480.0          # algorithmic FLOP per SDF point (SURVEY.md 8d / DESIGN.md)
METRIC = "sdf_points_per_sec"
UNIT = "points/s"
CONFIGS = {0: dict(batch=1, res=64), 1: dict(batch=1, res=256), 2: dict(batch=8, res=128), 4: dict(batch=1, res=512)}


def workload_string(cfg_id: int) -> str:
    c = CONFIGS[cfg_id]
    R = c["res"] + 1
    return "%s 137x137 image%s, --sdf_res %d (%s%d^3 = %d points), twostream, encoder included per step" % (
        "single" if c["batch"] == 1 else "batch of %d" % c["batch"], "" if c["batch"] == 1 else "s", c["res"],
        "" if c["batch"] == 1 else "%d x " % c["batch"], R, c["batch"] * R ** 3)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_burst=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"],
                    source="measured")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0, period_ms=100):
        self.rows, self.proc, self.gpu, self.period_ms = [], None, gpu_index, period_ms

    def start(self):
        if self.period_ms <= 0:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if not self.rows:       # region shorter than one sampling period (or no background sampler): take one sample now
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=10).stdout
                self.rows = [[c.strip() for c in line.split(",")] for line in o.splitlines() if line.strip()]
            except Exception:
                pass
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "power_w": float(np.median(pw)) if pw else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
SAMPLE_DIV = 8      # reference arm, configs other than 0: 1/8 of a chunk's points per step (plus the chunk's VGG pass)


def cpu_reference_step(cfg_id: int, state: dict):
    """One bounded sample of the workload on the host cores, structured as the reference runs it
    (test/create_sdf.py:262-275): per chunk, the whole graph including VGG.
      config 0: the complete job (2 chunks of 137 313 points, VGG per chunk) -- nothing extrapolated;
      other configs: chunk 0's VGG pass + the first 1/SAMPLE_DIV of its points; the chunk time is
        t_vgg + SAMPLE_DIV * t_points  (the per-point graph is the same work for every point, and all SPLIT_SIZE chunks
        are the same work), which keeps a K-step run within minutes where one full chunk costs 10-20 s.
    Returns (points_represented, seconds_represented, seconds_in_encoder, seconds_spent, description)."""
    import torch
    from disn_b200 import synth
    from oracle import disn_oracle as orc
    c = CONFIGS[cfg_id]
    if not state:
        torch.set_num_threads(os.cpu_count() or 1)
        state["W"] = synth.make_weights(seed=7, init="he")
        state["imgs"] = synth.synthetic_images(c["batch"])
        state["tm"] = synth.synthetic_trans_mats(c["batch"]) if c["batch"] > 1 else synth.DEMO_TRANS_MAT
        R, total, split, nsp = orc.chunking(c["res"])
        pts = orc.grid_points(synth.DEMO_SDF_PARAMS[0], R)
        pad = np.zeros((split * nsp - total, 3), np.float32)
        state["chunks"] = np.concatenate([pts, pad], 0).reshape(split, 1, nsp, 3)
        state["geom"] = (R, total, split, nsp)
    R, total, split, nsp = state["geom"]
    B = c["batch"]
    t0 = time.perf_counter()
    if cfg_id == 0:
        t_enc = 0.0
        for sp in range(split):
            te = time.perf_counter()
            enc = orc.encode(state["imgs"], state["W"], dtype=np.float32)    # VGG re-run per chunk, like the reference
            t_enc += time.perf_counter() - te
            pc = np.repeat(state["chunks"][sp], B, 0)
            orc.decode(enc, pc, pc, state["tm"], state["W"], dtype=np.float32)
        spent = time.perf_counter() - t0
        return B * total, spent, t_enc, spent, "the complete job: %d chunks of %d points, VGG re-run per chunk" % (split, nsp)
    n = (nsp + SAMPLE_DIV - 1) // SAMPLE_DIV
    enc = orc.encode(state["imgs"], state["W"], dtype=np.float32)
    t_enc = time.perf_counter() - t0
    pc = np.repeat(state["chunks"][0][:, :n], B, 0)
    orc.decode(enc, pc, pc, state["tm"], state["W"], dtype=np.float32)
    spent = time.perf_counter() - t0
    t_chunk = t_enc + (spent - t_enc) * (nsp / n)
    desc = ("chunk 0 of %d: its VGG pass + the first %d of its %d points per image; chunk time = t_vgg + %.3f x t_points" %
            (split, n, nsp, nsp / n))
    return B * nsp, t_chunk, t_enc, spent, desc


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    state = {}
    cpu_reference_step(args.config, state)                      # one warm-up sample (thread pools, allocator)
    rates, hoisted, spent = [], [], []
    desc = ""
    for _ in range(max(1, args.steps)):
        n, dt, t_enc, sp_s, desc = cpu_reference_step(args.config, state)
        rates.append(n / dt)
        hoisted.append(n / max(dt - t_enc, 1e-9))
        spent.append(sp_s)
    value = float(np.median(rates))
    c = CONFIGS[args.config]
    total_pts = c["batch"] * (c["res"] + 1) ** 3
    cores = os.cpu_count() or 1
    out = {"metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.median(spent)) * 1e3,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": workload_string(args.config),
                      "note": "PyTorch/NumPy CPU restatement of the TF graph (TF 1.x not installable); each step = " + desc +
                              "; ms_per_step is the duration of that sample; the whole job takes %.0f s at this rate" % (total_pts / value)},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc,
                            "encoder_hoisted_value": float(np.median(hoisted)), "runs": len(rates),
                            "min": float(min(rates)), "max": float(max(rates))},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    if args.config != 0:      # BASELINE config 0 (the reference's own CPU-runnable case) complete, nothing extrapolated
        st0 = {}
        runs = [cpu_reference_step(0, st0) for _ in range(3)]      # thread pools are warm from the steps above
        r = sorted(x[0] / x[1] for x in runs)
        h = sorted(x[0] / max(x[1] - x[2], 1e-9) for x in runs)
        out["config0_full"] = {"workload": workload_string(0), "value": r[1], "unit": UNIT, "encoder_hoisted_value": h[1],
                               "seconds": sorted(x[1] for x in runs)[1], "runs": 3, "min": r[0], "max": r[2], "cores": cores,
                               "note": runs[0][4] + "; median of 3"}
    print(json.dumps(out))


# --------------------------------------------------------------------------------------------------
DUMP_FULL_BYTES = 32 << 20      # a grid up to this size is dumped whole; a larger one as a sample
DUMP_SAMPLE = 1 << 21           # values in that sample (8 MiB, plus 16 MiB of indices)


def dump_outputs(out_dir: str, grid: np.ndarray, mesh_counts=None):
    """Writes the SDF grid [B, R, R, R] (float32) of the last timed step under out_dir, at most 64 MB in all:
      sdf.npy                        the whole grid, when it is at most DUMP_FULL_BYTES;
      sdf_sample.npy                 otherwise its values at DUMP_SAMPLE flat indices drawn with a fixed seed (sorted,
      sdf_sample_index.npy           repeats possible), and those indices as float64;
      mesh_counts.npy                config 4: [vertices, faces] of the mesh the step extracted (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    grid = np.ascontiguousarray(grid, dtype=np.float32)
    if grid.nbytes <= DUMP_FULL_BYTES:
        np.save(os.path.join(out_dir, "sdf.npy"), grid)
    else:
        idx = np.sort(np.random.default_rng(0).integers(0, grid.size, DUMP_SAMPLE))
        np.save(os.path.join(out_dir, "sdf_sample.npy"), grid.reshape(-1)[idx])
        np.save(os.path.join(out_dir, "sdf_sample_index.npy"), idx.astype(np.float64))
    if mesh_counts is not None:
        np.save(os.path.join(out_dir, "mesh_counts.npy"), np.asarray(mesh_counts, dtype=np.float64))


def shared_pinned_grid(nfloats: int, rank: int, world: int, barrier):
    """One host float32 buffer visible to every rank, page-locked in every rank's CUDA context.  Returns (tensor, cleanup)."""
    import torch
    if world == 1:
        t = torch.empty(nfloats, dtype=torch.float32).pin_memory()
        return t, (lambda: None)
    path = "/dev/shm/disn_bench_%s_%s" % (os.environ.get("MASTER_PORT", "0"), os.environ.get("TORCHELASTIC_RUN_ID", "x"))
    if rank == 0:
        with open(path, "wb") as f:
            f.truncate(nfloats * 4)
    barrier()
    t = torch.from_file(path, shared=True, size=nfloats, dtype=torch.float32)
    rt = torch.cuda.cudart()
    rc = rt.cudaHostRegister(t.data_ptr(), nfloats * 4, 0)
    if int(getattr(rc, "value", rc)) != 0:
        raise RuntimeError("cudaHostRegister failed: %s" % rc)

    def cleanup():
        rt.cudaHostUnregister(t.data_ptr())
        barrier()
        if rank == 0 and os.path.exists(path):
            os.remove(path)
    return t, cleanup


def run_ours(args):
    import torch
    import torch.distributed as dist
    from disn_b200 import sharding, synth
    from disn_b200.engine import Engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d" % args.gpus
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg = CONFIGS[args.config]
    B, res = cfg["batch"], cfg["res"]
    R = res + 1
    total_pts = B * R ** 3
    z_bounds = sharding.z_bounds(R, world)
    z0, z1 = sharding.slab(R, world, rank)
    max_planes = sharding.max_planes(R, world)
    planes = z1 - z0

    eng = Engine(device=local_rank, precision=args.precision, max_batch=B)
    W = synth.make_weights(seed=7, init="he")
    eng.load_weights(W)
    del W
    # an explicit (non-default) stream: torch's default stream has handle 0, which the C ABI reads as
    # "use the context's own stream" -- events must be recorded on the stream the kernels run on
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    eng.set_stream(stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    imgs_np = synth.synthetic_images(B)
    tm_np = (synth.synthetic_trans_mats(B) if B > 1 else synth.DEMO_TRANS_MAT).copy()
    sp = np.tile(synth.DEMO_SDF_PARAMS, (B, 1))
    img_host = torch.from_numpy(imgs_np).pin_memory()
    tm_host = torch.from_numpy(tm_np).pin_memory()
    img_dev, tm_dev = img_host.to(dev), tm_host.to(dev)
    # device-resident result.  One GPU: the [B,R,R,R] grid in this process.  N GPUs (B == 1): the whole grid lives in rank 0's
    # HBM (disn_shared_alloc); the other ranks map it through CUDA IPC and their kernels store their z-slab into it over
    # NVLink while they compute -- no gather collective (--gather nccl keeps the NCCL gather for comparison).
    peer = world > 1 and args.gather == "peer"
    slab = torch.empty((B, max_planes, R, R), dtype=torch.float32, device=dev)
    gathered = [torch.empty_like(slab) for _ in range(world)] if (world > 1 and rank == 0 and not peer) else None
    shared_ptr = 0
    if peer:
        hbuf = torch.zeros(64, dtype=torch.uint8, device=dev)
        if rank == 0:
            shared_ptr, handle = eng.shared_alloc(R ** 3 * 4)
            hbuf.copy_(torch.frombuffer(bytearray(handle), dtype=torch.uint8))
        dist.broadcast(hbuf, src=0)
        if rank != 0:
            shared_ptr = eng.shared_open(bytes(hbuf.cpu().numpy().tobytes()))
    out_ptr = (shared_ptr + z0 * R * R * 4) if peer else slab.data_ptr()
    host_grid, host_cleanup = shared_pinned_grid(B * R ** 3, rank, world, barrier)
    host_np = host_grid.numpy().reshape(B, R, R, R)
    do_mc = args.config == 4
    mesh = {}

    def slab_view():        # [B, planes, R, R] contiguous view of this rank's result
        return slab if planes == max_planes else slab[:, :planes]

    def result_grid():      # rank 0: the whole [B, R, R, R] grid the last step left in HBM, copied to the host
        if world == 1:
            return slab.cpu()
        if peer:
            return torch.from_numpy(eng.fetch(shared_ptr, (B, R, R, R)))
        return torch.cat([g[:, :z_bounds[r + 1] - z_bounds[r]].cpu() for r, g in enumerate(gathered)], 1)

    assert B == 1 or world == 1, "config 2 (batch of 8) runs on one GPU; shard images, not slabs, to scale it out"

    def grid_and_gather():
        eng.eval_grid_device(sp, tm_dev.data_ptr(), res, z0, z1, out_ptr)     # [B, planes, R, R] (peer: rank 0's grid)
        if world > 1 and not peer:
            dist.gather(slab, gather_list=gathered, dst=0)
        elif do_mc and peer:
            dist.barrier()          # rank 0 meshes the grid: every slab must have landed

    def mc_on_rank0(fetch):
        if rank != 0:
            return
        if world == 1:
            src_ptr = slab.data_ptr()
        elif peer:
            src_ptr = shared_ptr
        else:
            src = torch.cat([g[0, :z_bounds[r + 1] - z_bounds[r]] for r, g in enumerate(gathered)], 0)
            src_ptr = src.data_ptr()
        r = eng.marching_cubes(None, sp[0], mesh.get("iso", 0.0), device_ptr=src_ptr, R=R, fetch=fetch)
        mesh["nv"], mesh["nf"] = (len(r[0]), len(r[1])) if fetch else r

    def step_device():
        eng.encode_device(img_dev.data_ptr(), B, 137, 137, 3)
        grid_and_gather()
        if do_mc:
            mc_on_rank0(fetch=False)

    def step_e2e():
        eng.encode(img_host.numpy())                                         # H2D of the image inside disn_encode
        if do_mc:      # config 4's deliverable is the mesh: grid stays in HBM, the welded mesh comes back to the host
            grid_and_gather()
            mc_on_rank0(fetch=True)
        elif B == 1:   # this rank's z-slab of the one shared pinned host grid, written by the kernel's epilogue
            eng.eval_grid(sp, tm_np, res, z0=z0, z1=z1, out=host_np[0, z0:z1].reshape(1, planes, R, R))
        else:
            eng.eval_grid(sp, tm_np, res, out=host_np)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        if world > 1:
            dist.barrier()          # the step is complete when every rank's slab has landed
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    if do_mc:       # iso = median of the field (random weights need not cross zero), fixed before timing
        eng.encode_device(img_dev.data_ptr(), B, 137, 137, 3)
        eng.eval_grid_device(sp, tm_dev.data_ptr(), res, z0, z1, slab.data_ptr())       # local copy of this rank's slab
        torch.cuda.synchronize(dev)
        mesh["iso"] = float(slab_view().float().median().item())
        if world > 1:
            t = torch.tensor([mesh["iso"]], device=dev)
            dist.broadcast(t, src=0)
            mesh["iso"] = float(t.item())
    warm = max(3, args.warmup)
    for _ in range(warm):
        step_device()
    sampler = ClockSampler(local_rank, args.clock_period_ms)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count
    ms_total = timed(step_device, args.steps)
    launches = eng.launch_count - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        if rank == 0:
            dump_outputs(args.dump_outputs, result_grid().numpy(), (mesh["nv"], mesh["nf"]) if do_mc else None)
        barrier()           # no rank writes the shared grid again before rank 0 has read it
    ms_step = ms_total / args.steps
    value = total_pts / (ms_step * 1e-3)

    # kernel-only duration of the dominant kernel (fused point kernel) on this rank's slab, and of the encoder
    def ev_time(fn, reps):
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream)
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / reps
    # the dominant kernel's duration, measured INSIDE steps (events around the point kernel of encode + grid steps): timed
    # alone and back to back it runs in a different power / thermal state (+-3 % on this power-capped part)
    kreps = max(1, min(args.steps, 5))
    k_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(kreps)]
    torch.cuda.synchronize(dev)
    for a_, b_ in k_ev:
        eng.encode_device(img_dev.data_ptr(), B, 137, 137, 3)
        a_.record(stream)
        eng.eval_grid_device(sp, tm_dev.data_ptr(), res, z0, z1, slab.data_ptr())
        b_.record(stream)
    torch.cuda.synchronize(dev)
    k_ms = float(np.mean([a_.elapsed_time(b_) for a_, b_ in k_ev]))
    enc_ms = ev_time(lambda: eng.encode_device(img_dev.data_ptr(), B, 137, 137, 3), max(3, kreps))
    slab_pts = B * planes * R * R
    mc = None
    if rank == 0 and world == 1 and args.config in (1, 4):          # marching-cubes post-pass on the resident grid
        iso = mesh.get("iso", float(slab.float().median().item()))
        eng.marching_cubes(None, sp[0], iso, device_ptr=slab.data_ptr(), R=R, fetch=False)     # warm-up: sizes the scratch
        t_mc = ev_time(lambda: eng.marching_cubes(None, sp[0], iso, device_ptr=slab.data_ptr(), R=R, fetch=False), 3)
        nv, nf = eng.marching_cubes(None, sp[0], iso, device_ptr=slab.data_ptr(), R=R, fetch=False)
        alg = R ** 3 * 4 + nv * 12 + nf * 12
        peaks = load_peaks()
        mc = {"ms": t_mc, "verts": int(nv), "faces": int(nf), "iso": iso, "algorithmic_bytes": int(alg),
              "achieved_gbs": alg / (t_mc * 1e-3) / 1e9, "peak_gbs": peaks["hbm"], "frac": alg / (t_mc * 1e-3) / 1e9 / peaks["hbm"],
              "note": "classify + 2 scans + emit incl. the one host sync that sizes the output; scratch traffic (12 B/point of "
                      "edge ids + 4 B/cell, read and written by the scans) is not algorithmic"}

    # end-to-end through the host-buffer API
    for _ in range(2):
        step_e2e()
    e2e_steps = max(1, min(args.steps, 5))
    ms_e2e = timed(step_e2e, e2e_steps) / e2e_steps
    e2e_value = total_pts / (ms_e2e * 1e-3)
    # the host grid now holds the e2e result: cross-check it against the device-resident one
    e2e_ok = None
    if rank == 0 and B == 1 and not do_mc:
        e2e_ok = bool(torch.equal(host_grid.view(B, R, R, R), result_grid()))

    if rank == 0:
        peaks = load_peaks()
        achieved = slab_pts * F_ALG / (k_ms * 1e-3) / 1e12
        peak = peaks["bf16_sustained"]
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "point_kernel_traffic.json")
        if os.path.exists(tpath) and world == 1:
            t = json.load(open(tpath)).get(args.precision)
            if t and t.get("sdf_res") == res and B == 1:
                traffic = t["dram_bytes_read"] + t["dram_bytes_write"]
        passes = {"bf16x3": 3.0, "f16f8": 58.0 / 33.0}.get(args.precision, 1.0)     # bf16-rate MMA units per product (f16f8: 1.5 in fold2/conv1, 2 elsewhere)
        dtype_s = {"fp32": "f32",
                   "bf16x3": "bf16x3 (bf16 hi/lo split operands, 3 MMAs/product, fp32 accumulate)",
                   "f16f8": "f16+e5m2 (fp16 product + e5m2 correction products at 2x rate: two per layer, one in fold2/conv1; fp32 accumulate)"}[args.precision]
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None,
            "dtype": dtype_s,
            "data": "synthetic",
            "config": {"workload": workload_string(args.config), "baseline_config": args.config if world == 1 or args.config != 1 else 3,
                       "precision": args.precision, "parallelism": ("z-slab x%d, every rank's kernel stores its slab into rank 0's HBM over NVLink (CUDA IPC peer "
                                                                 "stores, no collective)" if peer else "z-slab x%d, slabs gathered to rank 0 (NCCL gather)") % world
                       if world > 1 else "z-slab x1",
                       "l2": "inputs larger than L2: each step streams 554 MB of VGG weights + writes %.0f MB of SDF" % (total_pts * 4 / 1e6)},
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": traffic, "kernel": "fused point kernel (%s)" % args.precision,
                         "kernel_ms": k_ms, "flop_per_point": F_ALG,
                         "algorithmic_bytes": int(slab_pts * 4),
                         "executed_tflops": achieved * passes,
                         "note": "frac counts the algorithmic FLOPs once; the split-operand scheme spends %.2fx that in bf16-rate tensor-pipe time"
                                 % passes if passes > 1 else "CUDA-core fp32 path reported against the tensor roofline",
                         "peak_source": "%s bf16 sustained (MEASURED_PEAKS.json)" % peaks["source"]},
            "encoder": {"ms": enc_ms, "images_per_s": B / (enc_ms * 1e-3), "batch": B,
                        "note": "resize + VGG-16 (tcgen05 convs) + fc6-8 + global/local folds, CUDA-graph replay"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(img_host.numel() * 4 + tm_host.numel() * 4),
                    "d2h_bytes_per_step": int(total_pts * 4) if not do_mc else int((mesh.get("nv", 0) + mesh.get("nf", 0)) * 12),
                    "ms_per_step": ms_e2e,
                    "path": "disn_encode(host) + disn_eval_grid(host, pinned): epilogue stores into the pinned host grid"
                            if not do_mc else "disn_encode(host) + resident grid + marching cubes + mesh fetched to the host",
                    "equals_device_result": e2e_ok},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if mc:
            out["marching_cubes"] = mc
        if do_mc:
            out["mesh"] = {"verts": int(mesh.get("nv", 0)), "faces": int(mesh.get("nf", 0)), "iso": mesh.get("iso"),
                           "in_timed_region": True}
        if world == 1 and not args.no_cpu_baseline and args.config in (0, 1):
            st = {}
            cpu_reference_step(args.config, st)               # warm-up
            runs = [cpu_reference_step(args.config, st) for _ in range(3)]
            r = sorted(x[0] / x[1] for x in runs)
            out["cpu_baseline"] = {"value": r[1], "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                                   "sample": runs[0][4] + "; 1 warm-up + median of 3", "min": r[0], "max": r[2],
                                   "encoder_hoisted_value": sorted(x[0] / max(x[1] - x[2], 1e-9) for x in runs)[1]}
        print(json.dumps(out))
    host_cleanup()
    if peer:
        barrier()
        if rank != 0:
            eng.shared_close(shared_ptr, owner=False)
        barrier()
        if rank == 0:
            eng.shared_close(shared_ptr, owner=True)
    if world > 1:
        dist.destroy_process_group()
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS))
    ap.add_argument("--precision", default=os.environ.get("DISN_PRECISION", "f16f8"), choices=["fp32", "bf16x3", "f16f8"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--clock-period-ms", type=int, default=100, dest="clock_period_ms",
                    help="nvidia-smi sampling period during the timed region (0 = one sample right after it)")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how the z-slabs reach rank 0's HBM (peer = stores from the kernel epilogue over NVLink)")
    ap.add_argument("--dump-outputs", metavar="DIR", dest="dump_outputs",
                    help="write the SDF grid of the last timed step under DIR as .npy (a seeded sample when it is large)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a sample of the job and keeps no grid")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
