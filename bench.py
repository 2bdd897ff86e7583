#!/usr/bin/env python
"""Benchmark of the vMAP vectorised per-object training step (BASELINE.json metric:
training-step rays/s at n_obj x n_rays x n_samples).

    python bench.py --gpus N --steps K --warmup W            # this framework on N GPUs
    python bench.py --impl reference --steps K --warmup W    # CPU reference arm (oracle port)

A "step" is one optimisation step of train.py:293-326 for the whole stack of objects: mask counts, fused
PE/MLP/render/loss/backward, ordered gradient reduction and AdamW -- ONE kernel launch (k_step_fused) per step.
N=1 workload = BASELINE cfg 2 (20 objects x 1200 rays x 10 samples, hidden 32).
N>1 = cfg 4, weak scaling: 20 objects per GPU, objects sharded across ranks, no collective in the step
(per-GPU independent Adam) -- only the timing barrier.  Every run also reports, as extra fields of the same JSON
line: BASELINE configs[4] (iMAP H=256, 4800 rays x 32 samples, rays sharded over the N ranks, ONE packed NCCL
all-reduce per step), the train.py-shaped drop-in loop and the captured frame loop at the shipped shape.
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

N_OBJ, N_RAYS, N_SAMPLES, HIDDEN = 20, 1200, 10, 32
FLOP_PER_POINT = 6 * (4 * HIDDEN * HIDDEN + 220 * HIDDEN + 63)      # SURVEY.md 8(d): 67,194 @ H=32
METRIC = "training-step rays/sec at n_obj x n_rays x n_samples"
IMAP_RAYS, IMAP_SAMPLES, IMAP_HIDDEN = 4800, 32, 256                # BASELINE configs[4]
IMAP_FLOP_PER_POINT = 6 * (4 * IMAP_HIDDEN * IMAP_HIDDEN + 220 * IMAP_HIDDEN + 63)

# tcgen05.mma cycles (M=128, K=16, both operands from shared memory) measured by tools/umma_bench2.cu on this pool's
# B200 (profiles/r02_umma_bench2.txt), and the fused kernel's MMA mix per 128-lane tile (k_step_fused.cuh: forward 23 x
# N32 + 4 x N16, dgrad 10 x N32 + 4 x N96 + 2 x N48, wgrad 40 x N32 + 16 x N16): the tensor-pipe time floor of THIS
# decomposition, i.e. the shape-limited peak the achieved FLOP/s is also reported against.
MMA_CYCLES = {16: 36.0, 32: 40.0, 48: 44.0, 96: 56.0}
MMA_MIX = {32: 73, 16: 20, 96: 4, 48: 2}


def log(msg):
    """Progress on stderr (stdout carries exactly one JSON line)."""
    print(f"[bench rank {os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


def workload_name(world):
    """The SAME string in both arms (the driver compares configs)."""
    return f"vMAP {N_OBJ} objects per GPU x {N_RAYS} rays x {N_SAMPLES} samples, hidden {HIDDEN} (BASELINE cfg 2 per GPU)"


def k1_dram_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the step kernel, from this round's committed
    `ncu --set full` summary of the same command (a profiler cannot run inside the timed benchmark)."""
    f = os.path.join(ROOT, "profiles", "r02_k_step_fused_ncu_summary.txt")
    if not os.path.isfile(f):
        return None
    tot, seen = 0.0, 0
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for ln in open(f):
        for key in ("dram__bytes_read.sum [", "dram__bytes_write.sum ["):
            if ln.startswith(key):
                unit = ln[len(key):ln.index("]")]
                tot += float(ln.split("=")[1]) * mult.get(unit, 1.0)
                seen += 1
    return tot if seen == 2 else None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return (d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0),
                d.get("sm_max_mhz", 1965.0), "measured")
    return 1590.0, 1400.0, 6650.0, 1965.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        rows = [l for (t, l) in self.lines if t0 - 0.05 <= t <= t1 + 0.05] or [l for _, l in self.lines]
        sm, mx, reasons = [], None, set()
        for l in rows:
            f = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_reference_rate(steps, warmup, bounded=True):
    """Times the CPU oracle port (oracle/vmap_oracle.py: the reference's functorch step
    restated op for op) with every host thread.  Returns (rays/s, ms/step, cores, sample)."""
    import torch
    from oracle import vmap_oracle as vo
    total = os.cpu_count() or 1
    rays = N_RAYS
    if bounded and steps * 0.5 > 120.0:          # keep the whole run within a few minutes
        rays = max(60, int(N_RAYS * 120.0 / (steps * 0.5)) // 12 * 12)
    params = vo.init_params(N_OBJ, HIDDEN, seed=0)
    ens = vo.OracleEnsemble(params, 2.0)
    batches = [vo.synthetic_batch(N_OBJ, rays, N_SAMPLES, seed=i) for i in range(2)]
    # "all the host threads it can use": these small batched GEMMs get SLOWER when oversubscribed, so pick the
    # fastest thread count on this box -- by the MEDIAN of three steps each, one noisy step must not decide it.
    best, cores = None, total
    for n in sorted({total, max(1, total // 2), 64, 32, 16, 8}, reverse=True):
        if n > total:
            continue
        torch.set_num_threads(n)
        ens.step(batches[0])
        ts = []
        for i in range(3):
            t = time.perf_counter()
            ens.step(batches[(i + 1) % 2])
            ts.append(time.perf_counter() - t)
        t = sorted(ts)[1]
        if best is None or t < best:
            best, cores = t, n
    torch.set_num_threads(cores)
    for i in range(warmup):
        ens.step(batches[i % 2])
    t0 = time.perf_counter()
    for i in range(steps):
        ens.step(batches[i % 2])
    dt = time.perf_counter() - t0
    sample = (f"{steps} full optimisation steps of {N_OBJ} obj x {rays} rays x {N_SAMPLES} samples, fp32, "
              f"{cores} threads (fastest median-of-3 among the thread counts tried on a {total}-core host)")
    return N_OBJ * rays * steps / dt, dt / steps * 1e3, cores, sample


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rate, ms, cores, sample = cpu_reference_rate(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.gpus),
                   "note": "reference is pure Python/PyTorch and cannot travel to the GPU box; this arm times the CPU port "
                           "of its functorch step (oracle/vmap_oracle.py), validated against the reference's own modules, "
                           "on ONE GPU's share of the workload (the reference is single-process, train.py:20)"},
        "cpu_baseline": {"value": rate, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# extra arms (same JSON line): configs[4], drop-in loop, frame loop
# ------------------------------------------------------------------------------------------------------------------
def bench_imap_cfg4(dev, world, rank, K, W, barrier, max_over_ranks):
    """BASELINE configs[4]: whole-scene MLP (hidden 256) replicated on every rank, 4800 rays x 32 samples per step,
    rays sharded over the ranks, ONE packed NCCL all-reduce (gradients + loss terms + next step's mask counts) per
    step, then AdamW on every rank.  Device-timed, max over ranks; rank 0 also times the full batch on one GPU."""
    import torch
    import torch.distributed as dist
    from vmap_b200 import synth as vo
    from vmap_b200.dist import ReplicatedStep
    from vmap_b200.ensemble import VmapEnsemble
    R_loc = IMAP_RAYS // world
    params = vo.init_params(1, IMAP_HIDDEN, seed=77)
    n_pool = 4

    def make(rays, lo):
        ens = VmapEnsemble(1, hidden=IMAP_HIDDEN, scale=5.0, device=dev)
        ens.load_stacked(params)
        full = [vo.synthetic_batch(1, IMAP_RAYS, IMAP_SAMPLES, seed=900 + i, n_cam2surf=5) for i in range(n_pool)]
        pool = [{k: v[:, lo:lo + rays].contiguous().to(dev) for k, v in b.items()} for b in full]
        return ens, ReplicatedStep(ens), pool

    def timed(rs, pool, use_graph, sync_all):
        for i in range(max(W, 3)):                                # eager warm-up (allocations, NCCL channels)
            rs.step(pool[i % n_pool], next_batch=pool[(i + 1) % n_pool])
        torch.cuda.synchronize()
        graphs = None
        if use_graph:
            try:
                graphs = []
                for i in range(n_pool):
                    g = torch.cuda.CUDAGraph()
                    rs._counts_for = id(pool[i])                  # counts arrive with the previous step's collective
                    with torch.cuda.graph(g):
                        rs.step(pool[i], next_batch=pool[(i + 1) % n_pool])
                    graphs.append(g)
                rs._counts_for = None                             # captures did not execute: recompute, then chain
                rs.step(pool[0], next_batch=pool[1])              # eager step establishes pool[1]'s counts on the device
                i0 = 1
            except Exception as e:                                # NCCL capture unsupported here: time eager launches
                graphs = None
                torch.cuda.synchronize()
                print(f"[bench] iMAP graph capture unavailable ({type(e).__name__}: {e}); eager", file=sys.stderr)
        if graphs is None:
            i0 = 0
        if sync_all:
            barrier()
        else:
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            j = (i0 + i) % n_pool
            if graphs is not None:
                graphs[j].replay()
            else:
                rs.step(pool[j], next_batch=pool[(j + 1) % n_pool])
        e1.record()
        if sync_all:
            barrier()
        else:
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / K
        return (max_over_ranks(ms) if sync_all else ms), graphs is not None

    ens, rs, pool = make(R_loc, rank * R_loc)
    ms, graphed = timed(rs, pool, use_graph=os.environ.get("VMB_GRAPHS", "1") == "1", sync_all=True)
    ens.check_status()
    out = {"workload": f"iMAP whole-scene MLP hidden {IMAP_HIDDEN}, {IMAP_RAYS} rays x {IMAP_SAMPLES} samples per step "
                       f"(BASELINE configs[4]), rays sharded {R_loc}/GPU over {world} GPU(s)",
           "ms_per_step": ms, "rays_per_s": IMAP_RAYS / (ms * 1e-3),
           "collectives_per_step": 1 if world > 1 else 0, "allreduce_bytes": rs.allreduce_bytes() if world > 1 else 0,
           "launch": "CUDA graph (step kernels + NCCL all-reduce + AdamW)" if graphed else "eager launches",
           "algorithmic_tflops": IMAP_FLOP_PER_POINT * IMAP_RAYS * IMAP_SAMPLES / (ms * 1e-3) / 1e12,
           "l2": "the layer-wise activation workspace (hundreds of MB per step) is rewritten every step, nothing stays in L2"}
    if world > 1:
        single = None
        if rank == 0:                                             # one GPU, full batch, same code path, no collective
            ens1 = VmapEnsemble(1, hidden=IMAP_HIDDEN, scale=5.0, device=dev)
            ens1.load_stacked(params)

            class _Solo(ReplicatedStep):
                def _world(self):
                    return 1
            full = [vo.synthetic_batch(1, IMAP_RAYS, IMAP_SAMPLES, seed=900 + i, n_cam2surf=5) for i in range(n_pool)]
            pool1 = [{k: v.to(dev) for k, v in b.items()} for b in full]
            single, _ = timed(_Solo(ens1), pool1, use_graph=os.environ.get("VMB_GRAPHS", "1") == "1", sync_all=False)
        barrier()
        if rank == 0:
            out["single_gpu_ms_per_step"] = single
            out["vs_single_gpu"] = single / ms
    return out


def bench_dropin(dev, K):
    """The train.py-shaped loop (train.py:293-326 written against the mirror API: vmap(pe) -> vmap(fc) ->
    loss.step_batch_loss -> backward -> optimiser.step -> zero_grad) at the shipped shape 20 objects x 120 rays:
    what the Python layer of the drop-in costs per step (two launches: fused step kernel, AdamW kernel)."""
    import torch
    import vmap_b200.loss as loss
    import vmap_b200.utils as utils
    from vmap_b200 import embedding, model
    from vmap_b200 import synth as vo
    from vmap_b200.optim import AdamW
    from vmap_b200.utils import vmap
    B, R, S = N_OBJ, 120, N_SAMPLES
    fcs = [model.OccupancyMap(87, 42, hidden_size=HIDDEN).apply(model.init_weights).to(dev) for _ in range(B)]
    pes = [embedding.UniDirsEmbed(max_deg=5, scale=2.0).to(dev) for _ in range(B)]
    opt = AdamW([torch.zeros(1)], lr=1e-3, weight_decay=0.013)
    fc_model, fc_param, fc_buffer = utils.update_vmap(fcs, opt)
    pe_model, pe_param, pe_buffer = utils.update_vmap(pes, opt)
    frame = {k: v.to(dev) for k, v in vo.synthetic_batch(B, R * 20, S, seed=4242).items()}

    def loop(n):
        for i in range(n):
            idx = slice((i % 20) * R, (i % 20 + 1) * R)
            emb = vmap(pe_model)(pe_param, pe_buffer, frame["pcs"][:, idx, ...])
            alpha, color = vmap(fc_model)(fc_param, fc_buffer, emb)
            batch_loss, _ = loss.step_batch_loss(alpha, color, frame["gt_depth"][:, idx], frame["gt_colour"][:, idx],
                                                 frame["sem"][:, idx], frame["mask_depth"][:, idx], frame["z"][:, idx])
            batch_loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
    loop(20)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    loop(K)
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / K * 1e3
    ms = e0.elapsed_time(e1) / K
    return {"workload": f"train.py-shaped loop, {B} objects x {R} rays x {S} samples (shipped Replica vMAP shape)",
            "ms_per_step": ms, "host_ms_per_step": wall, "rays_per_s": B * R / (ms * 1e-3), "launches_per_step": 2}


def bench_frame_loop(dev):
    """One mapping frame as ONE CUDA graph (vmap_b200/frame.py): batched sampler + the frame's 20 optimisation steps
    at the shipped shape (20 objects x 2400 rays per frame, 120 rays per step), Replica-sized keyframes."""
    import torch
    from vmap_b200 import synth as vo
    from vmap_b200.ensemble import VmapEnsemble
    from vmap_b200.frame import FrameLoop
    from vmap_b200.sampler import BatchedSampler, KeyframeSet
    B, KF, W, H = N_OBJ, 4, 1200, 680
    g = torch.Generator(device=dev).manual_seed(0)
    objs = []
    for b in range(B):
        rgbs = torch.randint(0, 256, (KF, W, H, 4), generator=g, dtype=torch.uint8, device=dev)
        rgbs[..., 3] = (torch.rand(KF, W, H, generator=g, device=dev) * 3).to(torch.uint8).clamp(0, 2)
        depth = torch.rand(KF, W, H, generator=g, device=dev) * 4 + 0.5
        depth[torch.rand(KF, W, H, generator=g, device=dev) < 0.1] = 0
        twc = torch.eye(4, device=dev).repeat(KF, 1, 1)
        twc[:, :3, 3] = torch.rand(KF, 3, generator=g, device=dev) - 0.5
        u0 = torch.randint(0, W - 300, (KF,), generator=g, device=dev).float()
        v0 = torch.randint(0, H - 250, (KF,), generator=g, device=dev).float()
        objs.append(KeyframeSet(rgbs, depth, twc, torch.stack([u0, u0 + 300, v0, v0 + 250], 1), KF, [KF - 2, KF - 1]))
    ii, jj = torch.meshgrid(torch.arange(W, dtype=torch.float32), torch.arange(H, dtype=torch.float32), indexing="ij")
    rays = torch.stack([(ii - 599.5) / 600.0, (jj - 339.5) / 600.0, torch.ones_like(ii)], -1).to(dev)   # vmap.py:31-41 (z-forward)
    smp = BatchedSampler(dev, n_bins_cam2surface=1, n_bins=9)
    ens = VmapEnsemble(B, hidden=HIDDEN, scale=2.0, device=dev)
    ens.load_stacked(vo.init_params(B, HIDDEN, seed=0))
    n_frames, n_pix, n_iter = 100, 24, 20
    fl = FrameLoop(ens, smp, n_frames, n_pix, n_iter, rays, seed=3)
    fl.set_objects(objs)
    fl.capture()
    for _ in range(3):
        fl.run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20
    e0.record()
    for _ in range(n):
        fl.set_objects(objs)              # per-frame host work: refill the pinned tables
        fl.run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    ens.check_status()
    return {"workload": f"frame graph: sampler + {n_iter} steps, {B} objects x {n_frames * n_pix} rays per frame "
                        f"({n_frames * n_pix // n_iter} rays per step), {W}x{H} keyframes",
            "frame_ms": ms, "ms_per_step": ms / n_iter, "rays_per_s": B * n_frames * n_pix / (ms * 1e-3)}


def dump_outputs(out_dir, ens):
    """What the last timed step hands its caller: the per-object loss terms it computed and the parameters after
    its AdamW update, one float32 ``<name>.npy`` per array (20 objects at hidden 32: under 1 MB).

    The inputs are the same in every run.  The outputs are only as reproducible as the step: by default the fused
    kernel sums weight-gradient MMAs in arrival order, and AdamW amplifies that rounding over the run (two runs of
    ``--steps 200 --warmup 10`` on a B200 at 1000 W: loss terms within ~1e-3 relative, parameters within ~2 % rel-L2).
    With ``VMB_DETERMINISTIC=1`` the step is bitwise reproducible (tests/test_umma_gpu.py::test_step_is_reproducible),
    so two builds can be compared bit for bit."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss_terms": ens.loss_terms}
    arrays.update({"params." + k: v for k, v in ens.stacked().items()})
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
    log(f"wrote {len(arrays)} arrays of the last timed step to {out_dir}")


def run_ours(args):
    import torch
    import torch.distributed as dist
    from vmap_b200 import synth as vo             # product-side input generator (oracle/ is only used by the cpu legs)
    from vmap_b200.ensemble import VmapEnsemble

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the vMAP step)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    impl = os.environ.get("VMB_IMPL", "auto")
    fused = impl in ("auto", "umma")
    log(f"world {world}, device {dev}, impl {impl}")

    sampler = ClockSampler(local)                 # runs for the whole process; windowed to the timed arms below
    if rank == 0:
        sampler.start()
    B, R, S = N_OBJ, N_RAYS, N_SAMPLES            # per GPU (weak scaling)
    params = vo.init_params(B, HIDDEN, seed=1000 + rank)
    ens = VmapEnsemble(B, hidden=HIDDEN, scale=2.0, device=dev, impl=impl)
    ens.load_stacked(params)

    # input pool larger than L2 (126 MB): every step reads a different, cold batch.  One flat
    # buffer per batch (pinned on the host) so a step's inputs move with a single H2D copy.
    from vmap_b200.ensemble import StepInputs
    step_bytes = B * R * S * 16 + B * R * 18
    n_pool = max(8, int(140e6 // step_bytes) + 1)
    host_pool = []
    for i in range(n_pool):
        host_pool.append(StepInputs(B, R, S, pinned=True).fill(vo.synthetic_batch(B, R, S, seed=rank * 100003 + i)))
    dev_pool = [StepInputs(B, R, S, device=dev).copy_from(h, non_blocking=False) for h in host_pool]
    stage = [StepInputs(B, R, S, device=dev).copy_from(host_pool[i], non_blocking=False) for i in range(2)]
    loss_host = torch.zeros(B, 4, dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()
    use_graphs = os.environ.get("VMB_GRAPHS", "1") == "1"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    K, W = args.steps, max(args.warmup, 3)
    log(f"input pool of {n_pool} batches ready")
    for i in range(3):                               # eager warm-up (sets kernel attributes, allocates scratch)
        ens.step(dev_pool[i % n_pool].views)
    if use_graphs:                                   # one captured step per input buffer
        pool_graphs = [ens.capture_step(d.views) for d in dev_pool]
        stage_graphs = [ens.capture_step(d.views) for d in stage]

    def run_step(i, pool, graphs):
        if use_graphs:
            graphs[i].replay()
        else:
            ens.step(pool[i].views)

    # ---- device-resident arm ("value"): inputs already in HBM ---------------------------------
    for i in range(W):
        run_step(i % n_pool, dev_pool, pool_graphs if use_graphs else None)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    for i in range(K):
        run_step((W + i) % n_pool, dev_pool, pool_graphs if use_graphs else None)
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    ens.check_status()
    log(f"device-resident arm: {ms_total / K * 1e3:.1f} us/step")
    if args.dump_outputs and rank == 0:           # before the arms below take more steps on the same ensemble
        dump_outputs(args.dump_outputs, ens)

    # ---- same steps launched eagerly with CUDA events around the step kernel (roofline) ----
    k1_events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for i in range(K):
        ens.forward_backward(dev_pool[(W + i) % n_pool].views, k1_events=k1_events[i], fuse_adam=True)
    barrier()
    k1_ms = sorted(a.elapsed_time(b) for a, b in k1_events)
    k1_avg_ms = sum(k1_ms) / len(k1_ms)

    # ---- end-to-end arm: pinned host inputs -> H2D -> step -> D2H loss terms --------------------
    # double-buffered: the copy of step i+1's inputs (copy stream) overlaps step i's kernels.
    cur, cs = torch.cuda.current_stream(), torch.cuda.Stream(device=dev)
    ev_copied = [torch.cuda.Event(), torch.cuda.Event()]
    ev_done = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_loop(n, base):
        for i in range(n):
            j = i % 2
            with torch.cuda.stream(cs):
                cs.wait_event(ev_done[j])                      # staging buffer j is free again
                stage[j].copy_from(host_pool[(base + i) % n_pool])
                ev_copied[j].record(cs)
            cur.wait_event(ev_copied[j])
            run_step(j, stage, stage_graphs if use_graphs else None)
            loss_host.copy_(ens.loss_terms, non_blocking=True)  # the step's result goes back to the host
            ev_done[j].record(cur)

    e2e_loop(4, 0)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    e2e_loop(K, 4)
    f1.record()
    barrier()
    e2e_ms = max_over_ranks(f0.elapsed_time(f1))
    ens.check_status()
    assert bool(torch.isfinite(loss_host).all())
    # keep the GPU under the same load a little longer so that nvidia-smi (>= 50 ms period) sees it
    t_hold = time.time()
    while time.time() - t_hold < 0.35:
        e2e_loop(50, 0)
        torch.cuda.synchronize()
    clocks = sampler.stop(t_wall0, time.time()) if rank == 0 else None

    # ---- extra arms -------------------------------------------------------------------------------------------------
    log(f"end-to-end arm: {e2e_ms / K * 1e3:.1f} us/step")
    extras = {}
    if not args.no_extras:
        try:
            extras["imap_cfg4"] = bench_imap_cfg4(dev, world, rank, max(20, min(K, 100)), W, barrier, max_over_ranks)
        except Exception as e:
            extras["imap_cfg4"] = {"error": f"{type(e).__name__}: {e}"}
        if rank == 0 and fused:
            for name, fn in (("dropin", lambda: bench_dropin(dev, 200)), ("frame_loop", lambda: bench_frame_loop(dev))):
                try:
                    extras[name] = fn()
                except Exception as e:
                    extras[name] = {"error": f"{type(e).__name__}: {e}"}
        barrier()

    if rank == 0:
        bf16_burst, bf16_sust, hbm, sm_max_mhz, src = peaks()
        rays_total = world * B * R * K
        flop_k1 = FLOP_PER_POINT * B * R * S
        achieved = flop_k1 / (k1_avg_ms * 1e-3) / 1e12
        # tensor-pipe floor of this decomposition: tiles/SM x MMA cycles per tile at the measured issue cost
        rpw = 32 // S
        tiles = B * ((R + 4 * rpw - 1) // (4 * rpw))
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        cyc_tile = sum(MMA_CYCLES[n] * c for n, c in MMA_MIX.items())
        floor_us = (tiles / n_sm) * cyc_tile / (sm_max_mhz * 1e6) * 1e6
        peak_shape = flop_k1 / (floor_us * 1e-6) / 1e12
        line = {
            "metric": METRIC, "value": rays_total / (ms_total * 1e-3), "unit": "rays/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": {
                "workload": workload_name(world),
                "global_objects": world * B, "parallelism": f"object-sharded x{world}, no collective in the step",
                "precision": "fp16 tensor-core operands, fp32 accumulate, fp32 master weights / Adam / render / loss",
                "impl": impl, "l2": f"input pool of {n_pool} distinct batches ({n_pool * step_bytes / 1e6:.0f} MB > 126 MB L2)",
                "launch": ("CUDA graph of the step (one kernel) per input buffer" if fused else "CUDA graph of K0+K1+K2 per input buffer")
                          if use_graphs else "eager launches",
                "d2h": "per-object loss terms copied to pinned host memory every step (async), one sync at the end",
            },
            "e2e": {"value": rays_total / (e2e_ms * 1e-3), "unit": "rays/s", "ms_per_step": e2e_ms / K,
                    "h2d_bytes_per_step": host_pool[0].nbytes, "d2h_bytes_per_step": B * 16,
                    "pipeline": "double-buffered staging: H2D of step i+1 on a copy stream overlaps step i"},
            "gpu_launches": (1 if fused else 3) * K,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": bf16_burst, "unit": "TFLOP/s",
                         "frac": achieved / bf16_burst,
                         "traffic": k1_dram_traffic() if fused and world == 1 else None,
                         "traffic_source": "profiles/r02_k_step_fused_ncu_summary.txt (ncu --set full of this command)",
                         "peak_source": src + " bf16 burst",
                         "peak_sustained": bf16_sust, "kernel": "k_step_fused" if fused else ("k_step_fp32" if impl == "fp32" else "layer-wise"),
                         "kernel_does": "mask counts + PE + MLP + render + loss + backward + ordered gradient reduction + AdamW" if fused else "K1 only",
                         "kernel_us": k1_avg_ms * 1e3, "kernel_us_median": k1_ms[len(k1_ms) // 2] * 1e3,
                         "flop_per_launch": flop_k1,
                         "peak_shape_limited": peak_shape, "frac_shape_limited": achieved / peak_shape,
                         "shape_limited_note": f"{tiles} tiles of 128 lanes over {n_sm} SMs x {cyc_tile:.0f} tensor-pipe cycles per tile "
                                               f"(tcgen05.mma M128 K16: N32 {MMA_CYCLES[32]:.0f}, N16 {MMA_CYCLES[16]:.0f}, N96 {MMA_CYCLES[96]:.0f}, N48 {MMA_CYCLES[48]:.0f} "
                                               f"cycles, profiles/r02_umma_bench2.txt) at {sm_max_mhz:.0f} MHz = {floor_us:.1f} us floor",
                         "hbm_algorithmic_GBps": (B * R * S * 16 + B * R * 18 + 24 * B * 11363) / (k1_avg_ms * 1e-3) / 1e9, "hbm_peak": hbm},
            "clocks": clocks,
        }
        line.update(extras)
        if world == 1 and not args.no_cpu:
            n_cpu = 12
            rate, ms, cores, sample = cpu_reference_rate(n_cpu, 2, bounded=False)
            line["cpu_baseline"] = {"value": rate, "unit": "rays/s", "cores": cores, "kind": "port",
                                    "ms_per_step": ms, "sample": sample}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[4] / drop-in / frame-loop arms")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss terms and updated parameters of the last "
                    "timed step (rank 0's objects) as DIR/<name>.npy; inputs are seeded, and with VMB_DETERMINISTIC=1 "
                    "so is the result, so runs compare array by array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the GPU arm only")
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
