#!/usr/bin/env python
"""bench.py — rays/sec of the eval-mode MultiPly forward on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # the reference algorithm on the host CPU
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's pixels as DIR/*.npy

A "step" is one pass of the hot path (Multiply.forward, eval) over one batch of synthetic rays:
BASELINE.json configs[1] = 2-person synthetic SMPL scene, 4096 rays x 128 samples (S/E/X = 128/256/64),
1 x B200.  With N GPUs every rank renders its own 4096-ray block of a 4096*N-ray batch (weak scaling)
and the rendered pixels are all-gathered over NCCL; `value` = all rays / max-over-ranks device time.

`value`  : inputs (rays, hit lists, posed bodies) resident on the device, engine.Renderer.render.
`e2e`    : the drop-in call — multiply_b200.model.multiply.Multiply.forward(input_dict) with the reference's input dict
           in PINNED HOST memory: per step H2D of uv / pose / intrinsics / smpl_* / idx, SMPL server, posed-grid rebuild,
           GPU ray/box culling, sampling, MLPs, compositing, D2H of rgb_values.
Sub-records (same JSON line, `extras`): strong scaling of one 16 384-ray x 256-sample frame (configs[3]),
person-sharded fields (configs[4]), a chunked 512x512 frame (configs[2]), dense SDF grid queries, precision modes.
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

import numpy as np
import torch

# algorithmic FLOPs per sample point (SURVEY.md §8d / BASELINE.md §2)
F_SDF, B_SDF, F_RGB, F_BG = 1084416, 918016, 532992, 1146880
RAYS_PER_GPU = 4096
S_SAMPLES = 128
PERSONS = 2
CPU_SAMPLE_RAYS = 512          # cpu_baseline leg of the GPU arm (timed once)
REF_SAMPLE_RAYS = 128          # --impl reference: rays per step


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_sustained=d.get("bf16_tflops_sustained", 1400.0), bf16_burst=d.get("bf16_tflops", 1590.0),
                    hbm=d.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_sustained=1400.0, bf16_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def config_dict(world):
    return {"workload": "configs[1]: 2-person synthetic SMPL scene, %d rays x %d samples per GPU "
                        "(S/E/X = 128/256/64, n = 193 main-pass samples), eval forward: sampler + deformer + "
                        "SDF/colour MLPs + composite + background" % (RAYS_PER_GPU, S_SAMPLES),
            "rays_per_gpu": RAYS_PER_GPU, "persons": PERSONS, "N_samples": S_SAMPLES,
            "global_rays": RAYS_PER_GPU * world,
            "precision": "fp16 hi/lo split x3 tcgen05 MMAs, fp32 accumulate (parity mode, RGB/SDF within 1e-4)",
            "scene": "bodies from the device SMPL server (mp_smpl_forward) on a synthetic SMPL-shaped model, "
                     "geometric-init networks (multiply_b200/scene.py:make_smpl_scene)",
            "rays": "uniform in the persons' image-space bounding rectangle; `value`: hit lists resident (host slab test, "
                    "as in BASELINE.md); `e2e`: culled on the GPU inside the timed region",
            "l2_flush": "256 MB device write between timed steps (outside the timed events)",
            "cpu_sample_rays": {"cpu_baseline": CPU_SAMPLE_RAYS, "reference_arm_per_step": REF_SAMPLE_RAYS},
            "parallelism": "ray blocks sharded over %d GPU(s), one NCCL all_gather of pixels" % world}


def best_cpu_threads(fn):
    """The oracle is many small torch ops: using every host thread is often slower than a moderate count.
    Time one call at a few settings and keep the fastest ("all the host threads it can use")."""
    cores = os.cpu_count() or 1
    best = None
    for t in sorted({min(cores, 8), min(cores, 32), cores}):
        torch.set_num_threads(t)
        t0 = time.time()
        fn()
        dt = time.time() - t0
        if best is None or dt < best[1]:
            best = (t, dt)
    torch.set_num_threads(best[0])
    return best[0]


def cpu_scene():
    """The benchmark scene built WITHOUT this repo's kernels (reference arm): same networks, same SMPL inputs, the
    bodies from the oracle's restatement of SMPLServer.forward (lib/model/smpl.py:50-95) instead of mp_smpl_forward —
    the two agree to 5e-6 (tests/test_gpu_mirror.py::test_smpl_server_and_culling)."""
    import math
    from oracle import port
    from multiply_b200 import scene as S
    si = S.smpl_scene_inputs(PERSONS)
    nets, rest = S.smpl_scene_networks(PERSONS, S_SAMPLES, 42)
    persons = []
    for p in range(PERSONS):
        sm = S.make_smpl_model(300 + p, body_seed=100 + p)
        tinv, vc = port.smpl_canonical_tfs_inv(sm, torch.zeros(10))
        o = port.smpl_server_forward(sm, tinv, si["smpl_params"][0, p, :1], si["smpl_trans"][0, p], si["smpl_pose"][0, p],
                                     torch.zeros(10))
        persons.append(dict(verts_c=vc, weights=sm["lbs_weights"], verts_p=o["smpl_verts"], tfs=o["smpl_tfs"],
                            smpl_pose=si["smpl_pose"][:, p].clone(), cond=si["smpl_pose"][:, p, 3:] / math.pi, scale=0.5,
                            implicit=nets[p]["implicit"], render=nets[p]["render"]))
    return dict(rest, persons=persons)


def run_reference(args, rank, world):
    """The reference algorithm on the host CPU (oracle/port.py — pinned against the unmodified reference
    modules by tests/golden; the reference itself needs the absent SMPL pkl / trimesh / nerfacc / pytorch3d)."""
    if rank != 0:
        return
    from oracle import port
    from multiply_b200 import scene as S
    sc = cpu_scene()
    n_sample = REF_SAMPLE_RAYS
    inp = S.make_rays(sc, RAYS_PER_GPU, seed=1234, region="boxes")
    sub = dict(uv=inp["uv"][:, :n_sample].contiguous(), pose=inp["pose"], intrinsics=inp["intrinsics"])
    hits = S.make_hit_lists(sc, sub)
    tiny = dict(uv=inp["uv"][:, :8].contiguous(), pose=inp["pose"], intrinsics=inp["intrinsics"])
    thits = S.make_hit_lists(sc, tiny)
    cores = best_cpu_threads(lambda: port.multiply_forward(sc, tiny, thits))
    times = []
    for i in range(args.warmup + args.steps):
        t = time.time()
        o = port.multiply_forward(sc, sub, hits)
        dt = time.time() - t
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, host_copy(o))
    tot = sum(times)
    val = n_sample * len(times) / tot
    line = {"impl": "reference", "metric": "rays/sec", "value": val, "unit": "rays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * tot / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(config_dict(world), precision="fp32 (torch CPU)", parallelism="host CPU, %d torch threads" % cores),
            "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cores, "kind": "port",
                             "sample": "%d of the %d rays of the same batch per step (full per-ray work: "
                                       "2 persons, S/E/X=128/256/64, background)" % (n_sample, RAYS_PER_GPU)},
            "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


class Timer:
    """K steps bracketed by barrier + synchronize, CUDA events per step on the current stream, L2 flush between
    steps (outside the events), max over ranks."""

    def __init__(self, dev, world, lib):
        self.dev, self.world, self.lib = dev, world, lib
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run(self, fn, steps, warmup, profile=False):
        import torch.distributed as dist
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        self.lib.mp_launch_count(1)
        if profile:
            self.lib.mp_profile_enable(1)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            self.flush.fill_(i & 0xFF)          # L2 flush, outside the timed events
            ev[i][0].record()
            fn()
            ev[i][1].record()
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        launches = self.lib.mp_launch_count(0)
        if profile:
            self.lib.mp_profile_enable(0)
        ms = sum(a.elapsed_time(b) for a, b in ev)
        t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), int(launches)


def linf(a, b):
    return float((a.double().cpu() - b.double().cpu()).abs().max())


def host_copy(out):
    """float32 host copies of the pixel outputs (parallel.PIXEL_KEYS) of one step."""
    from multiply_b200 import parallel
    return {k: out[k].detach().float().cpu().numpy() for k in parallel.PIXEL_KEYS}


def dump_outputs(path, arrays):
    """--dump-outputs: one DIR/<name>.npy per output array, so that two builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def extras_strong(timer, dev, rank, world, steps):
    """BASELINE configs[3]: ONE 16 384-ray x 256-sample frame (2 persons, S/E/X = 256/512/128, n = 385) sharded N ways
    over ray blocks (strong scaling): frame time, rays/s, and the gathered frame against the same frame rendered on
    one GPU (bit-equal when the sampler's batch-global trip counts agree, SURVEY §0-10)."""
    import torch.distributed as dist
    from multiply_b200 import engine, parallel, scene as S
    total = 16384
    sc = S.make_scene(P=2, S=256, seed=42)
    full = S.make_rays(sc, total, seed=77, region="boxes")
    lo, hi = parallel.shard_bounds(total, rank, world)
    mine = dict(uv=full["uv"][:, lo:hi].contiguous(), pose=full["pose"], intrinsics=full["intrinsics"])
    hits = [h.to(dev) for h in S.make_hit_lists(sc, mine)]
    d_in = {k: v.to(dev) for k, v in mine.items()}
    r = engine.Renderer(sc, device=dev)
    Rl = hi - lo
    buf = parallel.PixelBuffer(Rl, 2, dev)
    gathered = torch.empty(world, Rl * 12, device=dev) if world > 1 else None

    def step():
        r.render(d_in, hits, out=buf.views)
        if world > 1:
            dist.all_gather_into_tensor(gathered, buf.flat)

    ms, _ = timer.run(step, steps, 3)
    rec = {"config": "configs[3]: one %d-ray x 256-sample frame (2 persons, S/E/X = 256/512/128), %d rays per GPU" % (total, Rl),
           "frame_ms": ms / steps, "rays_per_s": total * steps / (ms / 1000.0), "scaling": "strong"}
    if world > 1:
        frame = parallel.PixelBuffer.frame(gathered, world, Rl, 2)
        if rank == 0:
            fh = [h.to(dev) for h in S.make_hit_lists(sc, full)]
            one = r.render({k: v.to(dev) for k, v in full.items()}, fh)
            torch.cuda.synchronize()
            rec["vs_single_gpu_frame"] = {"bit_equal": all(torch.equal(frame[k], one[k]) for k in parallel.PIXEL_KEYS),
                                          "rgb_linf": linf(frame["rgb_values"], one["rgb_values"])}
    return rec


def extras_person_sharded(timer, dev, rank, world, steps):
    """BASELINE configs[4]: 6 persons, 4096 rays x 128 samples, one canonical field per GPU (person p on rank p mod N),
    all-to-all of sample rows by ray block, block compositing, pixel all-gather; against the fused single-GPU frame."""
    import torch.distributed as dist
    from multiply_b200 import engine, parallel, scene as S
    P, R = 6, 4096
    sc = S.make_scene(P=P, S=S_SAMPLES, seed=42)
    inp = S.make_rays(sc, R, seed=1234, region="boxes")
    hits = S.make_hit_lists(sc, inp)
    d_in = {k: v.to(dev) for k, v in inp.items()}
    pr = parallel.PersonShardedRenderer(sc, device=dev)
    out = {}

    def step():
        out["o"] = pr.render(d_in, hits)

    ms, _ = timer.run(step, steps, 3)
    n = sc["cfg"]["N_samples"] + sc["cfg"]["N_samples_extra"] + 1
    # rows that leave their owner: every row of a person's hit list whose ray block is another rank's
    plan = parallel.exchange_plan(parallel.normalize_hits(hits), R, world)
    moved = sum(plan[p][b][1] - plan[p][b][0] for p in range(P) for b in range(world) if b != parallel.person_owner(p, world))
    rec = {"config": "configs[4]: %d persons, %d rays x %d samples, field p on GPU p mod %d" % (P, R, S_SAMPLES, world),
           "frame_ms": ms / steps, "rays_per_s": R * steps / (ms / 1000.0),
           "all_to_all_bytes_per_frame": int(moved * (8 * n + 1) * 4), "persons_per_gpu": [len([p for p in range(P) if parallel.person_owner(p, world) == g]) for g in range(world)]}
    if world > 1:
        # time of the exchange alone (same rows, same plan)
        rows = pr.person_rows(d_in, parallel.normalize_hits(hits))
        pr._plan = plan

        def xchg():
            parallel.exchange_person_rows(rows, plan, pr.width, rank, world, dev, None)

        xms, _ = timer.run(xchg, steps, 2)
        rec["all_to_all_ms"] = xms / steps
    if rank == 0:
        one = engine.Renderer(sc, device=dev).render(d_in, [h.to(dev) for h in hits])
        torch.cuda.synchronize()
        rec["vs_single_gpu_frame"] = {"bit_equal": all(torch.equal(out["o"][k], one[k]) for k in parallel.PIXEL_KEYS),
                                      "rgb_linf": linf(out["o"]["rgb_values"], one["rgb_values"])}
    return rec


def extras_full_frame(dev, rank, world):
    """BASELINE configs[2]: 3 persons, 512 x 512 pixels, 256 samples/ray (S/E/X = 256/512/128), chunked in 16 384-ray
    pieces through the drop-in Multiply.forward (idr_utils.split_input / merge_output, multiply_model.py:1235-1270);
    with N GPUs the chunks are dealt round-robin.  One warm-up chunk, then the whole frame is timed once."""
    import torch.distributed as dist
    from multiply_b200 import scene as S
    from multiply_b200.utils import idr_utils
    res, chunk = 512, 16384
    sc, model, smpl_in = S.make_smpl_scene(P=3, S=256, seed=42, device=dev)
    frame = S.grid_rays(res=res)
    # the synthetic camera looks down the world z axis from (0, 0, 2.5): the ray of the central pixel passes through the
    # origin, where depth2pts_outside's rotation axis cross(o, p_sphere) is 0/0 — NaN in the reference too
    # (multiply.py:712-714).  Shift the camera a hair so that the frame statistic below is finite.
    frame["pose"] = frame["pose"].clone()
    frame["pose"][0, 0, 3] = 0.013
    inputs = {k: v.to(dev) for k, v in dict(frame, **smpl_in).items()}
    chunks = idr_utils.split_input(inputs, res * res, n_pixels=chunk)
    mine = chunks[rank::world]
    with torch.no_grad():
        model(mine[0])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res_list = [model(c) for c in mine]
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    merged = idr_utils.merge_output(res_list, len(mine) * chunk, 1)
    model._renderer.check_status()
    return {"config": "configs[2]: 3 persons, %dx%d frame, 256 samples/ray, %d-ray chunks (%d chunks, %d per GPU)"
                      % (res, res, chunk, len(chunks), len(mine)),
            "frame_ms": float(ms.item()), "rays_per_s": res * res / (float(ms.item()) / 1000.0),
            "rgb_mean": float(merged["rgb_values"].mean()), "acc_mean": float(merged["acc_map"].mean())}


def extras_sdf_grid(dev):
    """f3: canonical SDF on the dense 257^3 lattice of generate_mesh (lib/utils/mesh.py:78-105) in one mp_sdf_grid call,
    and the same number of points in 10 000-point query_oc batches (point_batch of the reference's mesh refresh)."""
    from multiply_b200 import engine, scene as S
    sc = S.make_scene(P=1, S=16, seed=42)
    p0 = sc["persons"][0]
    f = engine.Field(p0["implicit"], p0["render"], device=dev)
    f.set_cond(p0["cond"])
    res = 256
    f.sdf_grid([0.0, 0.0, 0.0], 1.8, 32)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    f.sdf_grid([0.0, 0.0, 0.0], 1.8, res)
    e1.record()
    torch.cuda.synchronize()
    n = (res + 1) ** 3
    dense = n / (e0.elapsed_time(e1) / 1000.0)
    pts = (torch.rand(10000, 3, device=dev) - 0.5) * 2.0
    f.implicit_forward(pts, want_feat=False)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(100):
        f.implicit_forward(pts, want_feat=False)
    e1.record()
    torch.cuda.synchronize()
    return {"dense_res": res, "dense_points": n, "dense_points_per_s": dense,
            "dense_tflops_algorithmic": dense * F_SDF / 1e12,
            "batch_10k_points_per_s": 100 * 10000 / (e0.elapsed_time(e1) / 1000.0)}


def extras_precision(timer, r, d_inp, d_hits, R, steps, oracle_check):
    """The tcgen05 precision modes side by side (mp_set_precision): `parity` (three split terms everywhere, the headline),
    `colour1` (single-term colour layers), `throughput` (one fp16 term everywhere): rays/s of the resident-input step and,
    when the oracle sample is available, the measured L-inf of each mode against it."""
    from multiply_b200 import engine
    out = {}
    try:
        for mode in ("parity", "colour1", "throughput"):
            engine.set_precision(mode)
            ms, _ = timer.run(lambda: r.render(d_inp, d_hits), steps, 3)
            rec = {"rays_per_s": R * steps / (ms / 1000.0), "ms_per_step": ms / steps}
            if oracle_check is not None:
                rec.update(oracle_check())
            out[mode] = rec
    finally:
        engine.set_precision("parity")
    out["terms"] = {"parity": "A_hi.W_hi + A_lo.W_hi + A_hi.W_lo in every layer (fp16 hi/lo operands, fp32 accumulate)",
                    "colour1": "colour layers A_hi.W_hi only; SDF net and reverse sweep as parity",
                    "throughput": "A_hi.W_hi in every layer (plain fp16 tensor-core inference; outside the 1e-4 gate)"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--engine", default=os.environ.get("MP_ENGINE", "tc"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--precision", default="parity", choices=["parity", "colour1", "throughput"],
                    help="tcgen05 precision mode of the main measurement (default parity: RGB/SDF within 1e-4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the pixel outputs of the last timed step as DIR/<name>.npy (float32; rank 0, whole frame)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    assert args.warmup >= 3 or args.steps <= 2, "timing rules: at least 3 warm-up steps"
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    from multiply_b200 import engine, parallel, scene as S, _lib as L
    lib = L.lib()
    engine.set_engine(args.engine)
    engine.set_precision(args.precision)
    # ---- workload: the drop-in scene (bodies from the device SMPL server) --------------------------------
    sc, model, smpl_in = S.make_smpl_scene(P=PERSONS, S=S_SAMPLES, seed=42, device=dev)
    full = S.make_rays(sc, RAYS_PER_GPU * world, seed=1234, region="boxes")
    lo, hi = rank * RAYS_PER_GPU, (rank + 1) * RAYS_PER_GPU
    inp = dict(uv=full["uv"][:, lo:hi].contiguous(), pose=full["pose"], intrinsics=full["intrinsics"])
    hits = S.make_hit_lists(sc, inp)
    R = inp["uv"].shape[1]
    r = engine.Renderer(sc, device=dev)
    d_inp = {k: v.to(dev) for k, v in inp.items()}
    d_hits = [h.to(dev) for h in hits]
    h_inp = {k: v.pin_memory() for k, v in dict(inp, **smpl_in).items()}
    h_out = torch.empty(R, 3).pin_memory()
    buf = parallel.PixelBuffer(R, PERSONS, dev)
    gathered = torch.empty(world, R * (10 + PERSONS), device=dev) if world > 1 else None
    timer = Timer(dev, world, lib)
    model.output_buffers = buf.views          # the drop-in call writes its pixels straight into the gather buffer

    def step_resident():
        r.render(d_inp, d_hits, out=buf.views)
        if world > 1:
            dist.all_gather_into_tensor(gathered, buf.flat)

    def step_e2e():
        di = {k: v.to(dev, non_blocking=True) for k, v in h_inp.items()}
        o = model(di)
        if world > 1:
            dist.all_gather_into_tensor(gathered, buf.flat)
        h_out.copy_(o["rgb_values"], non_blocking=True)

    clocks = ClockSampler(local)
    clocks.start()
    ms_value, launches = timer.run(step_resident, args.steps, args.warmup)
    # the later passes below render into the same buffers: keep what the last timed step returned
    last_step = None
    if args.dump_outputs and rank == 0:
        last_step = host_copy(parallel.PixelBuffer.frame(gathered, world, R, PERSONS) if world > 1 else buf.views)
    with torch.no_grad():
        ms_e2e, launches_e2e = timer.run(step_e2e, args.steps, args.warmup)
    model._renderer.check_status()
    # Per-launch timing of the dominant kernel (roofline): CUDA events on the launching stream around every
    # tc_chain_kernel launch, in a pass of the same workload on the single-stream schedule.  (In the multi-stream
    # schedule the persons' launches queue behind each other INSIDE their event brackets, which would charge the
    # wait to the kernel.)
    prof_steps = max(1, min(args.steps, 20))
    L.check(lib.mp_set_streams(0), "mp_set_streams")
    ms_serial, _ = timer.run(step_resident, prof_steps, 2, profile=True)
    import ctypes as C
    pms = (C.c_double * 4)()
    pl = (C.c_longlong * 4)()
    pp = (C.c_double * 4)()
    L.check(lib.mp_profile_read(pms, pl, pp, 1), "mp_profile_read")
    L.check(lib.mp_set_streams(1), "mp_set_streams")
    clocks.stop_flag = True
    clocks.join(timeout=2)

    # one instrumented pass for trip counts (outside timing)
    o = r.render(d_inp, d_hits, debug=True)
    torch.cuda.synchronize()
    trips = o["trips"].cpu().tolist()

    # ---- the same resident-input step replayed from a CUDA graph (one graph launch instead of ~60 kernel launches)
    graph_rec = None
    try:
        gr = engine.GraphedRender(r, d_inp, d_hits)

        def step_graph():
            gr.replay()
            if world > 1:
                buf.flat.copy_(torch.cat([gr.out[k].reshape(-1) for k in parallel.PIXEL_KEYS]))
                dist.all_gather_into_tensor(gathered, buf.flat)

        ms_graph, _ = timer.run(step_graph, args.steps, args.warmup)
        torch.cuda.synchronize()
        graph_rec = {"rays_per_s": R * world * args.steps / (ms_graph / 1000.0), "ms_per_step": ms_graph / args.steps,
                     "bit_equal_to_eager": all(torch.equal(gr.out[k], o[k]) for k in parallel.PIXEL_KEYS),
                     "what": "engine.GraphedRender: mp_render_rays (63 launches, fork/join over 3 streams) captured once, "
                             "replayed per step; inputs resident"}
    except Exception as e:
        graph_rec = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---- parity at every N: the gathered frame against the same rays rendered on ONE GPU, and the drop-in call against
    # the resident-input renderer on this rank's shard
    parity = {}
    with torch.no_grad():
        o_drop = model({k: v.to(dev) for k, v in h_inp.items()})
    torch.cuda.synchronize()
    parity["drop_in_vs_resident_rgb_linf"] = linf(o_drop["rgb_values"], o["rgb_values"])
    if world > 1:
        step_resident()
        torch.cuda.synchronize()
        frame = parallel.PixelBuffer.frame(gathered, world, R, PERSONS)
        if rank == 0:
            fh = [h.to(dev) for h in S.make_hit_lists(sc, full)]
            one = r.render({k: v.to(dev) for k, v in full.items()}, fh)
            torch.cuda.synchronize()
            parity["gathered_vs_single_gpu"] = {"bit_equal": all(torch.equal(frame[k], one[k]) for k in parallel.PIXEL_KEYS),
                                                "rgb_linf": linf(frame["rgb_values"], one["rgb_values"]),
                                                "normal_linf": linf(frame["normal_values"], one["normal_values"]),
                                                "rays": R * world}

    extras = {}
    if not args.no_extras:
        xs = max(3, min(args.steps, 10))
        for name, fn in (("strong", lambda: extras_strong(timer, dev, rank, world, xs)),
                         ("person_sharded", lambda: extras_person_sharded(timer, dev, rank, world, xs)),
                         ("full_frame", lambda: extras_full_frame(dev, rank, world))):
            try:
                extras[name] = fn()
            except Exception as e:          # a sub-record must never take the headline line down
                extras[name] = {"error": "%s: %s" % (type(e).__name__, e)}
                if world > 1:
                    raise
        if rank == 0:
            try:
                extras["sdf_grid"] = extras_sdf_grid(dev)
            except Exception as e:
                extras["sdf_grid"] = {"error": "%s: %s" % (type(e).__name__, e)}

    if rank == 0:
        total_rays = R * world
        value = total_rays * args.steps / (ms_value / 1000.0)
        e2e = total_rays * args.steps / (ms_e2e / 1000.0)
        peaks = measured_peaks()
        # roofline of the dominant kernel (tc_chain_kernel): algorithmic FLOPs of the points it processed
        flops = pp[0] * F_SDF + pp[1] * F_SDF + pp[2] * (F_SDF + B_SDF + F_RGB) + pp[3] * F_BG
        mlp_ms = sum(pms)
        n_l = sum(pl)
        ach = flops / (mlp_ms / 1000.0) / 1e12 if mlp_ms > 0 else 0.0
        # all-samples formula of SURVEY.md §8d (no outlier skipping), for reference
        n = S_SAMPLES + S_SAMPLES // 2 + 1
        E = 2 * S_SAMPLES
        all_flops = 0.0
        for p in range(PERSONS):
            all_flops += hits[p].numel() * (trips[p] * E * F_SDF + n * (F_SDF + B_SDF + F_RGB))
        all_flops += R * 32 * F_BG
        h2d = sum(v.numel() * v.element_size() for v in h_inp.values())
        traffic, traffic_src = None, None
        for tag in ("r2", "r1"):
            tp = os.path.join(ROOT, "profiles", tag + "_traffic.json")
            if os.path.exists(tp):
                tj = json.load(open(tp))
                traffic = tj["tc_chain_kernel_dram_bytes_per_step"]
                traffic_src = "profiles/%s_traffic.json (%s)" % (tag, tj.get("captured", "ncu --set full capture of this workload"))
                break
        line = {
            "metric": "rays/sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_value / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (fp16 hi/lo split tensor-core operands, fp32 accumulate)",
            "data": "synthetic", "config": config_dict(world),
            "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(R * 3 * 4),
                    "ms_per_step": ms_e2e / args.steps,
                    "path": "multiply_b200.model.multiply.Multiply.forward(input_dict): pinned-host inputs -> H2D -> "
                            "SMPL server x%d -> posed-grid rebuild -> GPU ray/box culling -> sampler / deformer / MLPs / "
                            "composite / background -> D2H rgb_values; no host synchronisation inside the call" % PERSONS,
                    "gpu_launches_per_step": launches_e2e / args.steps},
            "gpu_launches": launches,
            "clocks": clocks.summary(),
            "roofline": {"bound": "tensor", "achieved": ach, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                         "frac": ach / peaks["bf16_sustained"], "traffic": traffic, "traffic_source": traffic_src,
                         "traffic_note": "DRAM bytes of the kernel's launches of one step; achieved is likewise aggregated over "
                                         "the step's launches.  Algorithmic bytes are ~6.6 MB of weights per field plus "
                                         "~100 B of I/O per point",
                         "kernel": "tc_chain_kernel (fused SDF/grad/colour MLP chain)",
                         "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                         "kernel_timing": "CUDA events per launch, %d-step pass on the single-stream schedule "
                                          "(%.3f ms/step; the timed region above overlaps persons and background on "
                                          "separate streams)" % (prof_steps, ms_serial / prof_steps),
                         "kernel_ms_per_step": mlp_ms / prof_steps, "kernel_launches_per_step": n_l / prof_steps,
                         "kernel_share_of_step": mlp_ms / ms_serial,
                         "points_per_step": {"sdf_only": pp[0] / prof_steps, "forward": pp[1] / prof_steps,
                                             "shade": pp[2] / prof_steps, "background": pp[3] / prof_steps},
                         "issued_tensor_tflops": None,
                         "all_samples_formula_tflops_per_step": all_flops / 1e12,
                         "effective_all_samples_tflops": all_flops * args.steps / (ms_value / 1000.0) / 1e12,
                         "ms_per_step_single_stream": ms_serial / prof_steps},
            "sampler_trips": trips, "engine": args.engine,
        }
        # issued tensor FLOPs: every step of every tile is 3 MMAs of 128x256x(64*nk)
        # 64-wide K chunks per tile of each program (mlp_tc.cu:tc_pack); the shade and background chains carry one
        # extra K-block for the colour net's extra inputs
        steps_nk = {0: 29, 1: 33, 2: 78, 3: 35}
        issued = 0.0
        for k in range(4):
            tiles = pp[k] / 128.0
            issued += tiles * steps_nk[k] * 3 * 2.0 * 128 * 256 * 64
        line["roofline"]["issued_tensor_tflops"] = issued / (mlp_ms / 1000.0) / 1e12 if mlp_ms > 0 else 0.0
        line["roofline"]["issued_frac_of_peak"] = line["roofline"]["issued_tensor_tflops"] / peaks["bf16_sustained"]
        line["roofline"]["note"] = ("parity mode issues three fp16 MMAs per product (A_hi.W_hi + A_lo.W_hi + A_hi.W_lo) and "
                                    "pads K / N to 64 / 256: `frac` counts the ALGORITHMIC FLOPs once, so its ceiling in "
                                    "this mode is ~1/3; `issued_frac_of_peak` is the tensor work actually issued against "
                                    "the same measured peak")
        if not args.no_cpu_baseline:
            from oracle import port
            n_sample = CPU_SAMPLE_RAYS
            sub = dict(uv=inp["uv"][:, :n_sample].contiguous(), pose=inp["pose"], intrinsics=inp["intrinsics"])
            shits = S.make_hit_lists(sc, sub)
            tiny = dict(uv=inp["uv"][:, :8].contiguous(), pose=inp["pose"], intrinsics=inp["intrinsics"])
            thits = S.make_hit_lists(sc, tiny)
            cores = best_cpu_threads(lambda: port.multiply_forward(sc, tiny, thits))
            t0 = time.time()
            ref = port.multiply_forward(sc, sub, shits)
            dt = time.time() - t0
            line["cpu_baseline"] = {"value": n_sample / dt, "unit": "rays/s", "cores": cores, "kind": "port",
                                    "sample": "first %d rays of this rank's 4096-ray batch, timed once, full per-ray work "
                                              "(oracle/port.py, torch CPU fp32, %d threads)" % (n_sample, cores)}
            # parity of the same rays rendered inside the full batch is not comparable (batch-global sampler
            # flag, SURVEY §0-10): render the sample on the GPU and compare
            og = r.render(sub, shits)
            torch.cuda.synchronize()
            parity.update({"rgb_linf_vs_oracle": linf(og["rgb_values"], ref["rgb_values"]),
                           "normal_linf_vs_oracle": linf(og["normal_values"], ref["normal_values"]),
                           "acc_linf_vs_oracle": linf(og["acc_map"], ref["acc_map"]), "rays": n_sample})
        if not args.no_extras and world == 1:
            chk = None
            if not args.no_cpu_baseline:
                def chk():
                    og2 = r.render(sub, shits, debug=True)
                    torch.cuda.synchronize()
                    return {"rgb_linf_vs_oracle": linf(og2["rgb_values"], ref["rgb_values"]),
                            "normal_linf_vs_oracle": linf(og2["normal_values"], ref["normal_values"]),
                            "acc_linf_vs_oracle": linf(og2["acc_map"], ref["acc_map"])}
            try:
                extras["precision_modes"] = extras_precision(timer, r, d_inp, d_hits, R, max(3, min(args.steps, 10)), chk)
            except Exception as e:
                extras["precision_modes"] = {"error": "%s: %s" % (type(e).__name__, e)}
        extras["cuda_graph"] = graph_rec
        line["parity"] = parity
        line["extras"] = extras
        if last_step is not None:
            dump_outputs(args.dump_outputs, last_step)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
