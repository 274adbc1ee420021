#!/usr/bin/env python
"""bench.py -- fwd+bwd Mpixel/s (and train iters/s) of the Gaussian-splat render path on B200.

    python bench.py --gpus N --steps K --warmup W            # ours (sm_100a kernels via the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU back end (oracle/_ref)

Workload (BASELINE.json configs[1]): 1M synthetic Gaussians, 1920x1080, SH degree 3, fp32, one camera
view per GPU (data-parallel over views; weak scaling).  A "step" is one pass of the hot path over one
view: SH fwd -> project fwd -> bin/sort/pack -> blend fwd -> MSE -> blend bwd -> project bwd -> SH bwd
(+ the cross-GPU gradient exchange when N > 1).  Prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n, W, H, scale, opacity range)
    "c2_1M_1080p_sh3": (1_000_000, 1920, 1080, 0.02, (0.05, 0.95)),
    "c3_3M_4k_sh3": (3_000_000, 3840, 2160, 0.01, (0.05, 0.95)),        # same pixel footprints as c2 (focal doubles)
    "c5_5M_1440p_dense": (5_000_000, 2560, 1440, 0.023, (0.05, 0.95)),   # ~200 blended-candidate splats / pixel
    "c1_1k_256": (1_000, 256, 256, 0.5, (0.05, 0.95)),
}


# kernels of OURS launched per fwd+bwd step (counted from the C-ABI implementations, fast binning path):
#   sh_fwd(+clamp) 1, project_fwd 1, bin_count 1, count_scan 1, tile_scan 1, tile_order 1, bucket_emit 1, tile_dsort_pack 1,
#   tile_sort_pack (fallback pass) 1, blend_fwd 1, mse 1, blend_bwd 1, row_reduce 1, project_bwd 1, sh_bwd 1
#   (N>1 fused exchange: mask 1 + exchange 1 instead of sh_bwd; the two cross-rank barriers are torch's kernels)
def launches_per_step(world=1, fused=True, train=False):
    n = 14 + (2 if (world > 1 and fused) else 1)
    return n + (1 if train else 0)


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
def cpu_reference_run(workload, steps, warmup, budget_s):
    """Times the reference's own CPU back end (oracle/_ref: the unmodified gsplat_cpu.cpp + operator .cpp files
    compiled where they lie) on the FULL workload -- same Gaussians, same image size, same fwd+bwd step as the
    GPU arm.  `steps` timed repetitions after `warmup` untimed ones, cut short once `budget_s` seconds of timed
    work have been spent (at least one timed step always runs).  Returns (Mpixel/s, info)."""
    import numpy as np
    import torch
    from oracle import ref
    from opensplat_b200.scene import make_scene
    n, W, H, scale, opac = WORKLOADS[workload]
    sc = make_scene(n, W, H, scale=scale, sh_degree=3, opacity=opac, seed=0)
    o = ref.ops()
    # all the host threads the reference can use (torchrun exports OMP_NUM_THREADS=1 to its workers)
    torch.set_num_threads(max(torch.get_num_threads(), min(os.cpu_count() or 1, 64)))
    t = lambda a, g=False: torch.from_numpy(np.ascontiguousarray(a)).requires_grad_(g)
    target = torch.zeros(H, W, 3)
    times = []
    for it in range(warmup + steps):
        means, scales, quats = t(sc["means"], True), t(sc["scales"], True), t(sc["quats"], True)
        coeffs, opacity = t(sc["coeffs"], True), t(sc["opacities"], True)
        t0 = time.perf_counter()
        rgbs = torch.clamp_min(o.sh_cpu(3, t(sc["viewdirs"]), coeffs) + 0.5, 0.0)
        p = o.project_cpu(means, scales, 1.0, quats, t(sc["viewmat"]), t(sc["projmat"]), sc["fx"], sc["fy"],
                          sc["cx"], sc["cy"], H, W, 0.01)
        img = o.rasterize_cpu(p[0], p[1], p[2], rgbs, opacity, p[3], p[4].contiguous(), H, W, torch.zeros(3))
        loss = torch.nn.functional.mse_loss(img, target)
        loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
            if sum(times) >= budget_s:
                break
    sec = sum(times) / len(times)
    info = {"cores": int(o.num_threads()), "kind": "reference", "steps_timed": len(times), "warmup_done": warmup,
            "sample": f"the full workload ({n} Gaussians at {W}x{H}, SH degree 3, fwd+bwd), {len(times)} timed "
                      f"step(s) after {warmup} warm-up; raster loops of the reference are single-threaded, ATen ops "
                      f"use {int(o.num_threads())} threads; host has {os.cpu_count()} cpus",
            "seconds_per_step": sec}
    return W * H / sec / 1e6, info


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warmup = max(0, min(args.warmup, 1))   # a CPU loop has nothing to warm beyond the allocator: one step at most
    v, info = cpu_reference_run(args.workload, steps=max(1, args.steps), warmup=warmup, budget_s=args.ref_budget_s)
    n, W, H, scale, opac = WORKLOADS[args.workload]
    out = {"impl": "reference", "metric": "fwd_bwd_mpixel_per_s", "value": v, "unit": "Mpixel/s",
           "n_gpus": args.gpus, "steps": info["steps_timed"], "warmup": info["warmup_done"],
           "ms_per_step": info["seconds_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": args.workload, "gaussians": n, "width": W, "height": H, "sh_degree": 3,
                      "note": f"full workload; {info['steps_timed']} step(s) timed of {args.steps} requested "
                              f"(time budget {args.ref_budget_s:.0f} s of CPU work), {info['warmup_done']} warm-up"},
           "cpu_baseline": {"value": v, "unit": "Mpixel/s", "cores": info["cores"], "kind": "reference",
                            "sample": info["sample"]},
           "e2e": {"value": v, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------
def _setup_pipe(workload, dev, rank, world, stage_timing=True):
    import numpy as np
    import torch
    from opensplat_b200.pipeline import SplatPipeline
    from opensplat_b200.scene import make_scene, cube_view_camera
    n, W, H, scale, opac = WORKLOADS[workload]
    sc = make_scene(n, W, H, scale=scale, sh_degree=3, opacity=opac, seed=0)  # same Gaussians on every rank
    pipe = SplatPipeline(n, W, H, sh_degree=3, device=dev, stage_timing=stage_timing)
    pipe.load_scene(sc)
    cam = None
    if world > 1:  # one camera view per GPU (config C4): the eight cube-symmetry views (comparable work per rank)
        cam = cube_view_camera(W, H, rank)
        pipe.set_camera(cam)
        vd = sc["means"] - cam["cam_pos"]
        vd = (vd / np.linalg.norm(vd, axis=-1, keepdims=True)).astype(np.float32)
        pipe.viewdirs.copy_(torch.from_numpy(vd).to(dev))
    rng = np.random.default_rng(1 + rank)
    target_host = torch.from_numpy(rng.uniform(0, 1, (H, W, 3)).astype(np.float32)).pin_memory()
    pipe.target.copy_(target_host, non_blocking=True)
    return pipe, sc, cam, target_host


def _pair_counts(pipe):
    """Untimed diagnostic pass: work units of the blend kernels for the frame currently in the pipeline's buffers."""
    import torch
    from opensplat_b200 import capi
    L, P = capi.lib(), capi.ptr
    cnt = torch.zeros(4, dtype=torch.int64, device=pipe.dev)
    out = torch.empty_like(pipe.out_img)
    fT, fI = torch.empty_like(pipe.final_Ts), torch.empty_like(pipe.final_idx)
    capi.check(L.gsb_rasterize_forward_count(pipe.H, pipe.W, pipe.tb[0], pipe.tb[1], pipe.m_raster, P(pipe.tile_bins),
                                             P(pipe.background), P(pipe.records), P(out), P(fT), P(fI), P(cnt),
                                             capi.stream()))
    torch.cuda.synchronize()
    assert torch.equal(out, pipe.out_img), "counting instantiation must reproduce the production image"
    rec, slots, ev, bl = (int(v) for v in cnt.tolist())
    return {"records_processed": rec, "pixel_tests": slots * 32, "pairs_evaluated": ev, "pairs_blended": bl}


def _traffic_for(workload, kernel):
    """dram__bytes_read+write of one launch from this round's `ncu --set full` capture, if one exists for exactly
    this workload and kernel (profiles/dram_traffic.json); null otherwise -- never a number from another config."""
    tfile = os.path.join(ROOT, "profiles", "dram_traffic.json")
    try:
        d = json.load(open(tfile))
        return d.get(workload, {}).get(kernel)
    except Exception:
        return None


def _ncu_counter(workload, kernel, key):
    """Per-launch counter of this round's ncu capture of exactly this workload / kernel (profiles/ncu_counters.json)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_counters.json"))).get(workload, {}).get(kernel, {}).get(key)
    except Exception:
        return None


def _roofline(pipe, stage_ms, ms_step, workload, pairs):
    peak, peak_src = peaks()
    alg, passes = pipe.algorithmic_bytes()
    alg_stage = dict(alg)
    alg_stage["bucket_sort_pack"] = alg["emit"] + alg["sort"] + alg["bins"]   # the fused stage stands for the three rows
    dom = max(stage_ms, key=lambda k: stage_ms[k]) if stage_ms else "raster_bwd"
    dom_key = dom if dom in alg_stage else "raster_bwd"
    ach = alg_stage[dom_key] / (stage_ms.get(dom_key, ms_step) * 1e-3) / 1e9
    path_bytes = sum(v for k, v in alg.items())
    path_ach = path_bytes / (ms_step * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": dom_key, "achieved": ach, "peak": peak, "unit": "GB/s",
            "frac": ach / peak, "traffic": _traffic_for(workload, dom_key), "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg_stage[dom_key], "ms_per_launch": stage_ms.get(dom_key),
            "note": "both blend kernels are instruction-issue bound (SURVEY R6); their work units are pixel pairs, "
                    "see `pairs`"}
    if pairs:
        f, b = stage_ms.get("raster_fwd"), stage_ms.get("raster_bwd")
        roof["pairs"] = dict(pairs)
        if f:
            roof["pairs"]["fwd_blended_pairs_per_s"] = pairs["pairs_blended"] / (f * 1e-3)
            roof["pairs"]["fwd_evaluated_pairs_per_s"] = pairs["pairs_evaluated"] / (f * 1e-3)
        if b:   # the backward pass replays the same blended set (up to each pixel's final index)
            roof["pairs"]["bwd_blended_pairs_per_s"] = pairs["pairs_blended"] / (b * 1e-3)
            roof["pairs"]["bwd_evaluated_pairs_per_s"] = pairs["pairs_evaluated"] / (b * 1e-3)
        # warp-instructions per blended pair: instruction totals from the committed ncu capture of THIS workload
        # (null without one), pair count from this run
        for key, st in (("fwd", "raster_fwd"), ("bwd", "raster_bwd")):
            ins = _ncu_counter(workload, st, "warp_instructions")
            roof["pairs"][f"{key}_warp_instructions_per_blended_pair"] = (ins / pairs["pairs_blended"]) if ins else None
            roof["pairs"][f"{key}_warp_instructions_per_record"] = (ins / pairs["records_processed"]) if ins else None
    roof_path = {"achieved": path_ach, "peak": peak, "unit": "GB/s", "frac": path_ach / peak,
                 "algorithmic_bytes_per_step": path_bytes, "generic_sort_passes_modelled": passes}
    return roof, roof_path


DUMP_GAUSSIANS = 1 << 16   # Gaussians whose gradients --dump-outputs keeps
DUMP_PIXELS = 1 << 21      # pixels it keeps of a larger image: a dump stays below 64 MB at every workload


def _dump_rows(t, k):
    """Rows of t at a fixed, seeded set of k indices; all of t when it has no more than k rows."""
    import numpy as np
    import torch
    if t.shape[0] <= k:
        return t
    rows = np.sort(np.random.default_rng(0).choice(t.shape[0], size=k, replace=False))
    return t.index_select(0, torch.from_numpy(rows).to(t.device))


def dump_outputs(out_dir, pipe):
    """Writes what the timed step hands its caller -- the rendered image, the loss and the gradient of every Gaussian
    parameter -- as float32 DIR/<name>.npy, so that two builds can be compared output for output.  The gradients are
    kept for DUMP_GAUSSIANS Gaussians, an image of more than DUMP_PIXELS pixels for that many (as [k, 3]); both
    samples are the same rows in every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    img = pipe.out_img
    if img.shape[0] * img.shape[1] > DUMP_PIXELS:
        img = _dump_rows(img.reshape(-1, 3), DUMP_PIXELS)
    arrays = {"image": img, "loss": pipe.loss}
    arrays.update({"grad_" + k: _dump_rows(v, DUMP_GAUSSIANS) for k, v in pipe.g.items()})
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def _side_config(workload, dev, steps=5, warmup=3):
    """One-shot sub-record for another BASELINE config (C3 / C5) on this GPU: value, stages, roofline."""
    import torch
    pipe, sc, cam, tgt = _setup_pipe(workload, dev, 0, 1, stage_timing=False)
    for _ in range(warmup):
        pipe.forward_backward()

    def region():
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            pipe.forward_backward()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    ms = region()                       # value: no instrumentation between the kernels
    pipe.stage_timing = True            # stage times / roofline: the same steps with per-stage events
    pipe.stage_ms.clear(); pipe._steps_ev = []
    ms_instr = region()
    stage_ms = pipe.resolve_stage_times()
    pairs = _pair_counts(pipe)
    roof, roof_path = _roofline(pipe, stage_ms, ms, workload, pairs)
    n, W, H, _, _ = WORKLOADS[workload]
    rec = {"value": W * H / (ms * 1e-3) / 1e6, "unit": "Mpixel/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
           "gaussians": n, "width": W, "height": H, "intersections_binned": pipe.m,
           "intersections_reference": int(pipe.nth.sum()), "longest_tile_list": pipe.max_len,
           "tile_occupancy": pipe.tile_occupancy(),
           "stages_ms": {k: round(v, 4) for k, v in stage_ms.items()}, "ms_per_step_instrumented": ms_instr,
           "roofline": roof, "roofline_path": roof_path}
    del pipe
    torch.cuda.empty_cache()
    return rec


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from opensplat_b200 import capi, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    capi.lib()  # fail loudly if the CUDA library is missing

    n, W, H, scale, opac = WORKLOADS[args.workload]
    pipe, sc, cam, target_host = _setup_pipe(args.workload, dev, rank, world)
    fused = world > 1 and args.exchange == "fused"
    exchange_check = None
    if fused:
        # The fused exchange is verified ONCE, outside every timed region, against the plain path (sh_backward +
        # one NCCL all-reduce of the flat buffer) on this very scene; if it cannot be set up or disagrees, every rank
        # falls back to the NCCL exchange and the line says so.
        ok_local, geo_rel, sh_rel, why = 1, None, None, None
        try:
            from opensplat_b200.multigpu import ViewParallelExchange
            pipe.exchange = ViewParallelExchange(pipe, cam["cam_pos"])
            pipe.forward(); pipe.backward()
            got = pipe.grad_flat.clone()
            ex, pipe.exchange = pipe.exchange, None
            pipe.forward(); pipe.backward()
            dist.all_reduce(pipe.grad_flat, op=dist.ReduceOp.SUM)
            ref = pipe.grad_flat * (1.0 / world)
            pipe.exchange = ex
            geo = pipe.geom_numel
            geo_rel = float((ref[:geo] - got[:geo]).norm() / ref[:geo].norm())
            sh_rel = float((ref[geo:] - got[geo:]).norm() / ref[geo:].norm())
            ok_local = int(geo_rel < 1e-5 and sh_rel < 1e-4)
            del got, ref
        except Exception as exn:   # e.g. symmetric memory / multicast not available on this box
            ok_local, why = 0, str(exn)[:200]
        flag = torch.tensor([ok_local], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        exchange_check = {"verified_against_nccl": bool(flag[0]), "geometry_rel_l2": geo_rel, "sh_rel_l2": sh_rel,
                          "multicast": bool(getattr(pipe.exchange, "multicast_ptr", 0)), "error": why}
        if not bool(flag[0]):
            pipe.exchange = None
            fused = False

    def step_fwd_bwd():
        pipe.forward()
        pipe.backward()       # with pipe.exchange: fused multi-view SH backward + gradient all-reduce inside
        if world > 1 and pipe.exchange is None:
            dist.all_reduce(pipe.grad_flat, op=dist.ReduceOp.SUM)
        pipe._collect()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms[0])

    for _ in range(max(args.warmup, 3)):
        step_fwd_bwd()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # the headline region: K steps, no instrumentation between the kernels
    pipe.stage_timing = False
    ms_total = timed(step_fwd_bwd, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pipe)
    # the same K steps again with a CUDA event at every stage boundary (stage times, roofline): the ~20 timing events
    # per step cost 1-2 % (each one drains the launch pipeline for a moment), which is why they are not in the
    # headline region; `ms_per_step_instrumented` says what the step took with them
    pipe.stage_timing = True
    pipe.stage_ms.clear(); pipe._steps_ev = []
    ms_instr = timed(step_fwd_bwd, args.steps) / args.steps
    stage_ms = pipe.resolve_stage_times()
    m_timed = pipe.m
    ms_step = ms_total / args.steps
    value = world * W * H / (ms_step * 1e-3) / 1e6
    pairs = _pair_counts(pipe)
    m_ref = int(pipe.nth.sum())
    occupancy = pipe.tile_occupancy()

    # per-rank work and compute time (separates view skew from the exchange): every rank's binned M, longest tile
    # list and the sum of its own stages without the exchange stage
    compute_ms = sum(v for k, v in stage_ms.items() if k != "sh_bwd")
    mine = {"rank": rank, "intersections_binned": m_timed, "intersections_reference": m_ref,
            "longest_tile_list": pipe.max_len, "compute_ms_without_exchange": round(compute_ms, 4),
            "exchange_stage_ms": round(stage_ms.get("sh_bwd", 0.0), 4)}
    per_rank = [mine]
    if world > 1:
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)

    # ---- train iters/s: + fused Adam (and the all-reduce average) ----
    pipe.stage_timing = False
    for _ in range(2):
        pipe.train_step(world_size=world)
    ms_train = timed(lambda: pipe.train_step(world_size=world), args.steps) / args.steps

    # ---- e2e: through the reference-facing autograd operators, host buffers in the timed region ----
    from opensplat_b200 import cpp_ops
    use_cpp = cpp_ops.available()
    cops = cpp_ops.ops() if use_cpp else None
    names = ("means", "scales", "quats", "coeffs", "opacities")
    P = {k: pipe.p[k].detach().clone().requires_grad_() for k in names}
    # the operators' gradients accumulate IN PLACE into views of one flat buffer (AccumulateGrad adds into an existing
    # .grad), so the data-parallel exchange of this arm is the single NCCL all-reduce of north_star
    gflat = torch.zeros(sum(t.numel() for t in P.values()), device=dev)
    gviews, o = {}, 0
    for k in names:
        gviews[k] = gflat[o:o + P[k].numel()].view_as(P[k]); o += P[k].numel()
    view_host = pipe.viewmat.cpu().pin_memory()
    proj_host = pipe.projmat.cpu().pin_memory()
    fx, fy, cx, cy = pipe.intr
    bg = torch.zeros(3, device=dev)

    # H2D of every step's inputs (target image + camera) from pinned memory runs on a copy stream, one step
    # ahead of the compute (double buffer); the step's result (the loss) is copied D2H every step into one of two
    # pinned slots and consumed on the host two steps later (when its slot comes round again), so neither direction
    # stalls the GPU or drains the launch queue.  All inside the timed region.
    copy_stream = torch.cuda.Stream(device=dev)
    slots = [dict(tgt=torch.empty_like(pipe.target), vm=torch.empty_like(pipe.viewmat),
                  pm=torch.empty_like(pipe.projmat), ev=torch.cuda.Event(), used=torch.cuda.Event(),
                  loss=torch.zeros(1).pin_memory(), loss_ev=torch.cuda.Event()) for _ in range(2)]
    state = {"i": 0, "last_loss": None}

    def prefetch(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(slot["used"])      # the compute that last read this slot has finished
            slot["tgt"].copy_(target_host, non_blocking=True)
            slot["vm"].copy_(view_host, non_blocking=True)
            slot["pm"].copy_(proj_host, non_blocking=True)
            slot["ev"].record(copy_stream)

    for sl in slots:
        sl["used"].record(torch.cuda.current_stream())
    prefetch(slots[0])

    def step_e2e():
        i = state["i"]
        cur, nxt = slots[i % 2], slots[(i + 1) % 2]
        if i > 1:                                                # the result of step i-2 (this slot's previous use),
            cur["loss_ev"].synchronize()                         # read on the host before the slot is written again:
            state["last_loss"] = float(cur["loss"][0])           # the host never waits for the step still in flight
        prefetch(nxt)                                            # next step's inputs, overlapped
        state["i"] = i + 1
        torch.cuda.current_stream().wait_event(cur["ev"])       # this step's H2D has landed
        tgt, vm, pm = cur["tgt"], cur["vm"], cur["pm"]
        if world > 1 and fused:
            # gradients of the geometry tensors accumulate in place into the symmetric flat buffer the fused exchange
            # all-reduces; the colour gradient lands in the symmetric v_rgb buffer the peers pull from
            pipe.grad_flat[:pipe.geom_numel].zero_()
            pipe.exchange.v_rgb.zero_()
            for k in ("means", "scales", "quats", "opacities"):
                P[k].grad = pipe.g[k]
            P["coeffs"].grad = None
        elif world > 1:
            gflat.zero_()
            for k in names:
                P[k].grad = gviews[k]
        else:
            for t in P.values():
                t.grad = None
        if world > 1 and fused:
            # SH colours through the operator (forward); their backward + the cross-GPU reduction happen in the fused
            # exchange launch, which expands every view's colour gradient into the coefficient gradient
            with torch.no_grad():
                rgbs = torch.clamp_min((cops.spherical_harmonics(3, pipe.viewdirs, P["coeffs"]) if use_cpp else
                                        ops.compute_sh_forward(3, 3, pipe.viewdirs, P["coeffs"])) + 0.5, 0.0)
            rgbs.requires_grad_()
            rgbs.grad = pipe.exchange.v_rgb
        elif use_cpp:   # the libtorch autograd operators a C++ caller of the reference API uses
            rgbs = torch.clamp_min(cops.spherical_harmonics(3, pipe.viewdirs, P["coeffs"]) + 0.5, 0.0)
        else:
            rgbs = torch.clamp_min(ops.SphericalHarmonics.apply(3, pipe.viewdirs, P["coeffs"]) + 0.5, 0.0)
        if use_cpp:
            xys, depths, radii, conics, nth, _ = cops.project_gaussians(
                P["means"], P["scales"], 1.0, P["quats"], vm, pm, fx, fy, cx, cy, H, W, 0.01)
            img = cops.rasterize_gaussians(xys, depths, radii, conics, nth, rgbs, P["opacities"], H, W, bg)
        else:
            xys, depths, radii, conics, nth, _ = ops.ProjectGaussians.apply(
                P["means"], P["scales"], 1.0, P["quats"], vm, pm, fx, fy, cx, cy, H, W, pipe.tb)
            img = ops.RasterizeGaussians.apply(xys, depths, radii, conics, nth, rgbs, P["opacities"], H, W, bg)
        loss = torch.nn.functional.mse_loss(img, tgt)
        loss.backward()
        if world > 1 and fused:
            pipe.rgbs = rgbs.detach()                            # the clamp mask of the exchange
            pipe.exchange.exchange(average=False)               # ONE fused launch: SH bwd of all views + all-reduce
        elif world > 1:
            dist.all_reduce(gflat, op=dist.ReduceOp.SUM)        # ONE flat all-reduce of all per-Gaussian gradients
        cur["used"].record(torch.cuda.current_stream())
        cur["loss"].copy_(loss.detach().reshape(1), non_blocking=True)  # D2H: the step's result
        cur["loss_ev"].record(torch.cuda.current_stream())

    for _ in range(3):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = world * W * H / (ms_e2e * 1e-3) / 1e6

    roof, roof_path = _roofline(pipe, stage_ms, ms_step, args.workload, pairs)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    side = {}
    if world == 1 and args.workload == "c2_1M_1080p_sh3" and not args.no_side_configs:
        del P, gflat
        for wl in ("c3_3M_4k_sh3", "c5_5M_1440p_dense"):
            try:
                side[wl] = _side_config(wl, dev, steps=args.steps, warmup=max(args.warmup, 3))
            except Exception as ex:   # a sub-record must never cost the headline line
                side[wl] = {"error": str(ex)[:300]}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            v, info = cpu_reference_run(args.workload, steps=2, warmup=0, budget_s=30.0)
            cpu = {"value": v, "unit": "Mpixel/s", "cores": info["cores"], "kind": info["kind"],
                   "sample": info["sample"]}
        except Exception as ex:  # the checker is optional for the number; say why it is missing
            cpu = {"value": None, "unit": "Mpixel/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {ex}"}

    exch = ("fused launch: multi-view SH bwd over NVLink peer loads + two-shot all-reduce of the geometry gradients ("
            + ("NVSwitch multimem" if getattr(pipe.exchange, "multicast_ptr", 0) else "peer pointers") + ")") \
        if fused else "nccl all-reduce(flat grads)"
    out = {
        "metric": "fwd_bwd_mpixel_per_s", "value": value, "unit": "Mpixel/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "gaussians": n, "width": W, "height": H, "sh_degree": 3,
                   "intersections_M": m_timed, "intersections_reference": m_ref,
                   "binning": "conservative cull at bin time: (Gaussian, tile) pairs whose alpha>=1/255 extent box "
                              "misses the tile are never sorted or streamed (results unchanged)",
                   "views_per_gpu": 1, "parallelism": f"dp{world}-views",
                   "views": "cube-symmetry view set (comparable work per rank)" if world > 1 else "front view",
                   "step": "sh+project+bin/sort/pack+blend fwd, mse, blend+project+sh bwd"
                           + (", " + exch if world > 1 else ""),
                   "l2_policy": "inputs larger than L2 (>300 MB of parameters/records per step vs 126 MB L2)"},
        "train_iters_per_s": 1e3 / ms_train, "train_ms_per_iter": ms_train,
        "e2e": {"value": e2e_value, "unit": "Mpixel/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(target_host.numel() * 4 + 128), "d2h_bytes_per_step": 4 + 16,
                "last_loss_read_on_host": state["last_loss"],
                "api": ("C++ libtorch autograd operators ProjectGaussians/RasterizeGaussians/SphericalHarmonics "
                        "(libopensplat_b200_ops.so via torch.ops)") if use_cpp else
                       "opensplat_b200.ops python autograd operators",
                "exchange": (("the fused exchange launch (as the device-timed arm)" if fused else
                              "one NCCL all-reduce of the flat gradient buffer") if world > 1 else None)},
        "gpu_launches": launches_per_step(world, fused) * args.steps,
        "clocks": clocks,
        "roofline": roof, "roofline_path": roof_path,
        "stages_ms": {k: round(v, 4) for k, v in stage_ms.items()},
        "ms_per_step_instrumented": ms_instr,
        "per_rank": per_rank,
        "tile_occupancy": occupancy,
        "exchange_check": exchange_check,
        "other_configs": side or None,
        "cpu_baseline": cpu,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def _watchdog(seconds):
    """A bench run that stalls (hung kernel / collective) must not block the driver: exit hard after `seconds`."""
    def fire():
        sys.stderr.write(f"bench.py watchdog: no result after {seconds}s, aborting\n")
        sys.stderr.flush()
        os._exit(3)
    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()


if __name__ == "__main__":
    _watchdog(1500)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every measured region (>= 1)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2_1M_1080p_sh3", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-configs", action="store_true", help="skip the C3 / C5 one-shot sub-records (N=1)")
    ap.add_argument("--ref-budget-s", type=float, default=150.0,
                    help="--impl reference: stop after this many seconds of timed CPU work (>= 1 step always runs)")
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"],
                    help="N>1: fused multi-view SH backward + all-reduce launch over peer memory (default) or plain "
                         "NCCL all-reduce of the flat gradient buffer")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (image, loss, sampled gradients) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours only")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
