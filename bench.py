#!/usr/bin/env python
"""Benchmark of the DM-NeRF render hot path (BASELINE.json metric: rays/sec, 64 coarse + 128 fine samples).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--scaling weak|strong]
                    [--dump-outputs DIR]

One "step" = one full 640x480 synthetic frame (307 200 rays) per GPU through the complete pipeline
(coarse net -> composite -> importance sampling -> fine net -> composite, object head included), i.e.
BASELINE.json configs[1] (DM-SR 'study').  Under torchrun (N > 1) every rank renders its own frame of the
synthetic trajectory (rays shard with no data-path collective; weak scaling) and the rendered images are
all-gathered once per step over NCCL, inside the timed region.

Timed quantities (ours):
  value      rays/s, device-timed (CUDA events on the launch stream), inputs already resident in HBM
  e2e        rays/s through the C-ABI host entry point (dmnerf_render_forward_host): pinned HOST rays in,
             HOST rgb/depth/acc/ins out, H2D + D2H inside the timed region
  roofline   the dominant kernel (fine-network MLP): algorithmic FLOPs / its CUDA-event duration vs the measured
             tensor peak in MEASURED_PEAKS.json
  cpu_baseline  the oracle port (torch CPU restatement of the reference) on this box's host cores, bounded sample

--scaling strong (BASELINE configs[4], the per-pose loop of tester.py:55-85): ONE frame per step, its pixels split by
contiguous range over the N ranks; every rank generates the rays of its range on its own device from K / c2w (a new pose
of the synthetic trajectory every step), renders them with the fused kernel, and one NCCL all-gather assembles the image
on every rank; `value` = frame rays / max-over-ranks time, `allgather` = that collective's share.

--impl reference times that same CPU path alone (the reference is pure Python/torch and cannot travel to the GPU
box; the oracle is its bit-for-bit restatement, see oracle/dmnerf_oracle.py).

--dump-outputs DIR writes the per-ray maps the last timed step returned (rgb_fine, depth_fine, acc_fine, ins_fine) as
DIR/<name>.npy in float32, so that two builds run with the same arguments (same seeded weights and rays) can be compared
map by map.  Above 60 MiB in all, every map keeps the same seeded sample of rays.
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

import numpy as np   # noqa: E402
import torch         # noqa: E402

N_COARSE, N_IMPORTANCE = 64, 128
_CPU_THREADS = None


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="dmsr_study")
    ap.add_argument("--mlp", default="auto", choices=["auto", "simt", "umma"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the informational training-step block")
    ap.add_argument("--cpu-procs", type=int, default=0,
                    help="cpu_baseline: also run this many concurrent CPU workers (whole-box figure); 0 = cores // 16")
    ap.add_argument("--cpu-worker", type=int, default=0, help=argparse.SUPPRESS)    # internal: one whole-box worker, N threads
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's per-ray maps as DIR/<name>.npy")
    return ap.parse_args()


WORKLOAD_TEXT = {
    "dmsr_study": "DM-SR 'study' 640x480 full render, 64+128 hierarchical, coarse+fine+object head",
    "replica_room0": "Replica room0 640x480, 59-object instance logits, 64+128 samples",
    "replica_room0_93": "Replica room_0 640x480, 93-object instance logits (data/color_dict.json), 64+128 samples",
    "replica_office2": "Replica office2 640x480 trajectory frames, 69-object instance logits, 64+128 samples",
}


def workload_text(name, ins_num, n_rays, scaling, world):
    per = "one frame (%d rays) per GPU per step" % n_rays if scaling == "weak" else \
        "one frame (%d rays) per step, pixels split over %d GPU(s)" % (n_rays, world)
    return "%s (ins_num=%d), %s" % (WORKLOAD_TEXT.get(name, name), ins_num, per)


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_rate(workload, seconds, chunk=1024, threads=None):
    """rays/s of the oracle port on the host cores: full dm_nerf pipeline, 1024-ray chunks (BASELINE configs[0]
    chunk size), repeated until `seconds` of CPU work have elapsed (at least 2 chunks after 1 warm-up)."""
    from oracle import dmnerf_oracle as O
    from dmnerf_b200 import synth
    wl = synth.workload(workload)
    cores = os.cpu_count() or 1
    pc = O.to_torch(synth.make_weights(101, wl["ins_num"]))
    pf = O.to_torch(synth.make_weights(202, wl["ins_num"]))
    ro, rd = torch.from_numpy(wl["rays_o"]), torch.from_numpy(wl["rays_d"])
    z = O.z_val_sample(chunk, wl["near"], wl["far"], N_COARSE)
    n_total = ro.shape[0]
    with torch.no_grad():
        # the reference would run with torch's default (= all cores); on many-core hosts that oversubscribes these
        # small GEMMs badly, so give the CPU arm its best thread count (quick calibration on 256 rays)
        global _CPU_THREADS
        if threads is not None:
            _CPU_THREADS = threads
        if _CPU_THREADS is None:
            best = None
            for th in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
                torch.set_num_threads(th)
                O.render(ro[:256], rd[:256], pc, pf, z[:256], perturb=0.0, n_importance=N_IMPORTANCE)
                t0 = time.perf_counter()
                O.render(ro[256:512], rd[256:512], pc, pf, z[:256], perturb=0.0, n_importance=N_IMPORTANCE)
                dt = time.perf_counter() - t0
                if best is None or dt < best[0]:
                    best = (dt, th)
            _CPU_THREADS = best[1]
        torch.set_num_threads(_CPU_THREADS)
        O.render(ro[:chunk], rd[:chunk], pc, pf, z, perturb=0.0, n_importance=N_IMPORTANCE)     # warm-up
        done, t0 = 0, time.perf_counter()
        pos = chunk
        while True:
            O.render(ro[pos:pos + chunk], rd[pos:pos + chunk], pc, pf, z, perturb=0.0, n_importance=N_IMPORTANCE)
            done += chunk
            pos = (pos + chunk) % (n_total - chunk)
            el = time.perf_counter() - t0
            if el >= seconds and done >= 2 * chunk:
                break
    return done / el, cores, torch.get_num_threads(), done, el


def cpu_whole_box_rate(workload, seconds, procs, threads):
    """Whole-box CPU figure: `procs` concurrent workers of `threads` threads each (one 16-thread process leaves most of a
    128-core host idle: small GEMMs stop scaling there), rates summed."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload, "--cpu-worker", str(threads),
           "--cpu-seconds", str(seconds)]
    ps = [subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=dict(os.environ, RANK="0"))
          for _ in range(procs)]
    rates = []
    for pr in ps:
        out, _ = pr.communicate()
        try:
            rates.append(float(json.loads(out.strip().splitlines()[-1])["rays_per_s"]))
        except Exception:
            pass
    return sum(rates), len(rates)


def cpu_c1_coarse_only(workload="dmsr_study", reps=3):
    """BASELINE configs[0] exactly as named: one 1024-ray chunk, 64 coarse samples, coarse MLP only (embed -> network ->
    composite), CPU torch fp32, with autograd recording as in the reference's training forward and its global anomaly mode
    (networks/dm_nerf.py:5) off and on."""
    from oracle import dmnerf_oracle as O
    from dmnerf_b200 import synth
    wl = synth.workload(workload)
    pc = {k: v.requires_grad_(True) for k, v in O.to_torch(synth.make_weights(101, wl["ins_num"])).items()}
    ro, rd = torch.from_numpy(wl["rays_o"][:1024]), torch.from_numpy(wl["rays_d"][:1024])
    z = O.z_val_sample(1024, wl["near"], wl["far"], N_COARSE)
    res = {}

    def once():
        viewdirs = rd / torch.norm(rd, dim=-1, keepdim=True)
        x, shp = O._net_inputs(ro, rd, viewdirs, z)
        raw = O.mlp_forward(pc, x).reshape(*shp, -1)
        return O.composite(raw, z, rd)

    for tag, flag in (("anomaly_off", False), ("anomaly_on", True)):
        torch.autograd.set_detect_anomaly(flag)
        once()
        t0 = time.perf_counter()
        for _ in range(reps):
            once()
        res[tag + "_rays_per_s"] = 1024 * reps / (time.perf_counter() - t0)
    torch.autograd.set_detect_anomaly(False)
    res["what"] = "1024-ray chunk, 64 coarse samples, embed + coarse DM_NeRF + render_train, torch CPU fp32, %d threads" % torch.get_num_threads()
    return res


def cpu_train_step(workload="dmsr_study", anomaly=False):
    """BASELINE configs[3] on the CPU: dm_nerf(perturb=1) on 1024 random rays + the benchmark loss + backward (oracle port)."""
    from oracle import dmnerf_oracle as O
    from dmnerf_b200 import synth
    wl = synth.workload(workload)
    n_rays = wl["rays_o"].shape[0]
    pc = {k: v.requires_grad_(True) for k, v in O.to_torch(synth.make_weights(101, wl["ins_num"])).items()}
    pf = {k: v.requires_grad_(True) for k, v in O.to_torch(synth.make_weights(202, wl["ins_num"])).items()}
    sel = np.random.Generator(np.random.PCG64(0)).choice(n_rays, 1024, replace=False)
    ro, rd = torch.from_numpy(wl["rays_o"][sel]), torch.from_numpy(wl["rays_d"][sel])
    z = O.z_val_sample(1024, wl["near"], wl["far"], N_COARSE)
    gen = torch.Generator().manual_seed(0)
    tgt = torch.rand(1024, 3, generator=gen)
    torch.autograd.set_detect_anomaly(anomaly)
    t0 = time.perf_counter()
    out = O.render(ro, rd, pc, pf, z, perturb=1.0, n_importance=N_IMPORTANCE, t_rand=torch.rand(1024, N_COARSE, generator=gen),
                   u=torch.rand(1024, N_IMPORTANCE, generator=gen), is_train=True)
    loss = ((out["rgb_fine"] - tgt) ** 2).mean() + ((out["rgb_coarse"] - tgt) ** 2).mean() + out["ins_fine"].mean()
    loss.backward()
    dt = time.perf_counter() - t0
    torch.autograd.set_detect_anomaly(False)
    return 1024 / dt, dt


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from dmnerf_b200 import synth
    if args.cpu_worker:                                # internal: one worker of the whole-box measurement
        r, _, _, _, _ = cpu_reference_rate(args.workload, args.cpu_seconds, threads=args.cpu_worker)
        print(json.dumps({"rays_per_s": r}))
        return
    wl = synth.workload(args.workload)
    rates = []
    per_step = max(2.0, min(20.0, 100.0 / max(1, args.steps + args.warmup)))
    for i in range(args.warmup + args.steps):
        r, cores, threads, rays, el = cpu_reference_rate(args.workload, per_step)
        if i >= args.warmup:
            rates.append((r, rays, el))
    tot_rays = sum(x[1] for x in rates)
    tot_t = sum(x[2] for x in rates)
    value = tot_rays / tot_t
    line = {
        "impl": "reference", "metric": "rays/sec (64c+128f samples)", "value": value, "unit": "rays/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, args.steps),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args.workload, wl["ins_num"], wl["rays_o"].shape[0], args.scaling, args.gpus),
                   "name": args.workload, "rays_per_step_per_gpu": int(wl["rays_o"].shape[0]) // (args.gpus if args.scaling == "strong" else 1),
                   "note": "CPU arm: each step renders a bounded sample of that frame (1024-ray chunks, as the reference's "
                           "tester.py chunk loop would) and reports rays/s"},
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port",
                         "sample": "%d rays per step in 1024-ray chunks, torch CPU fp32, %d threads" % (rates[-1][1], threads)},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 and len(r) >= 7] or [r for (_, r) in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[0]) for r in rows)
        reasons = []
        for i, name in ((3, "hw_slowdown"), (4, "hw_thermal_slowdown"), (5, "sw_thermal_slowdown"), (6, "sw_power_cap")):
            if any(r[i].lower().startswith("active") for r in rows):
                reasons.append(name)
        try:
            pw = max(float(r[2]) for r in rows)
        except ValueError:
            pw = None
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "power_w_max": pw, "samples": len(rows),
                "reasons": reasons}


# --------------------------------------------------------------------------------------------- outputs
DUMP_BYTES = 60 << 20          # keeps a dump below 64 MB with room for the .npy headers


def dump_outputs(out, n_rays, ins_num, path):
    """Write one step's result as path/<map>.npy (float32).  `out` is render_rays' dict of per-ray maps, or on N > 1 ranks
    the all-gathered [N, rays, 5 + ins_num] image slab, whose first `n_rays` rows are unpacked into the same maps.  When the
    maps exceed DUMP_BYTES they all keep the same rays: a sorted sample drawn from a fixed seed."""
    from dmnerf_b200.parallel import unpack_image
    if torch.is_tensor(out):
        out = unpack_image(out.reshape(-1, out.shape[-1])[:n_rays], ins_num)
    maps = {k: v.float().contiguous().cpu().numpy() for k, v in out.items()}
    total = sum(a.nbytes for a in maps.values())
    if total > DUMP_BYTES:
        keep = np.random.Generator(np.random.PCG64(0)).choice(n_rays, DUMP_BYTES * n_rays // total, replace=False)
        maps = {k: a[np.sort(keep)] for k, a in maps.items()}
    os.makedirs(path, exist_ok=True)
    for k, a in maps.items():
        np.save(os.path.join(path, k + ".npy"), a)


# --------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import ctypes as C
    from dmnerf_b200 import synth, _lib
    from dmnerf_b200.engine import get_context
    from dmnerf_b200.testing import make_models

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (ours) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    impl = {"auto": _lib.IMPL_AUTO, "simt": _lib.IMPL_SIMT, "umma": _lib.IMPL_UMMA}[args.mlp]

    wl = synth.workload(args.workload, frame=rank)                  # each rank: its own frame of the trajectory
    ins_num = wl["ins_num"]
    n_rays = wl["rays_o"].shape[0]
    nc, nf, _, _ = make_models(101, 202, ins_num, dev)
    ctx = get_context(dev)
    ctx.bind(0, nc); ctx.bind(1, nf)
    from dmnerf_b200.render import render_rays
    from dmnerf_b200.parallel import gather_image
    ro, rd = torch.from_numpy(wl["rays_o"]).to(dev), torch.from_numpy(wl["rays_d"]).to(dev)
    z = (torch.linspace(0, 1, N_COARSE) * (wl["far"] - wl["near"]) + wl["near"]).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    strong = args.scaling == "strong"
    gather_ev = []
    if strong:
        # BASELINE configs[4]: ONE frame per step (a new pose of the synthetic trajectory each step), pixel range per rank,
        # rays generated on the device from K / c2w for that range only, one all-gather of the packed image.
        from dmnerf_b200.parallel import shard_range
        from dmnerf_b200.helpers import get_rays_at
        lo, hi, per = shard_range(n_rays, world, rank, multiple=128)
        pix = torch.arange(lo, hi, device=dev, dtype=torch.int64)
        poses = [torch.from_numpy(synth.workload(args.workload, frame=f)["c2w"]).to(dev) for f in range(8)]
        step_no = [0]

    def step_device():
        if strong:
            c2w = poses[step_no[0] % len(poses)]
            step_no[0] += 1
            ro_r, rd_r = get_rays_at(wl["H"], wl["W"], wl["K"], c2w, pix)
            out = render_rays(ro_r, rd_r, nc, nf, z, want_raw=False, want_coarse=False, want_samples=False, impl=impl)
            if world > 1:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                full = gather_image(out, world, pad_to=per)
                e1.record()
                gather_ev.append((e0, e1))
                return full
            return out
        out = render_rays(ro, rd, nc, nf, z, want_raw=False, want_coarse=False, want_samples=False, impl=impl)
        if world > 1:
            return gather_image(out, world)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- warm-up
    with torch.no_grad():
        for _ in range(max(3, args.warmup)):
            step_device()
        barrier()
        # ---- timed: K steps, per-step CUDA events (L2 flushed, untimed, between steps)
        launches0 = _lib.launch_count()
        del gather_ev[:]
        lib = ctx.lib
        _lib.check(lib.dmnerf_profile_enable(ctx.handle, 1), "profile_enable")
        sampler = ClockSampler(local)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        stage_ms = np.zeros(6)
        barrier()
        t_wall0 = time.perf_counter()
        for s in range(args.steps):
            flush.fill_(s & 0xFF)
            evs[s][0].record()
            if s + 1 < args.steps:
                step_device()
            else:
                last = step_device()             # only the last step's result is kept, for --dump-outputs
            evs[s][1].record()
            ms = (C.c_float * 6)()
            _lib.check(lib.dmnerf_profile_read(ctx.handle, ms, 6), "profile_read")
            stage_ms += np.array(list(ms))
        barrier()
        t_wall1 = time.perf_counter()
        clocks = sampler.stop(t_wall0, t_wall1)
        _lib.check(lib.dmnerf_profile_enable(ctx.handle, 0), "profile_enable")
        launches = _lib.launch_count() - launches0
        dev_ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
        gather_ms = sum(a.elapsed_time(b) for a, b in gather_ev) if gather_ev else 0.0
        if args.dump_outputs and rank == 0:
            dump_outputs(last, n_rays * (1 if strong else world), ins_num, args.dump_outputs)
        del last

        # ---- end to end through the C ABI with HOST buffers (pinned), H2D + D2H inside the timed region
        h = {k: torch.empty(shape, dtype=torch.float32).pin_memory() for k, shape in
             (("rgb_fine", (n_rays, 3)), ("depth_fine", (n_rays,)), ("acc_fine", (n_rays,)), ("ins_fine", (n_rays, ins_num)))}
        hro, hrd = torch.from_numpy(wl["rays_o"]).pin_memory(), torch.from_numpy(wl["rays_d"]).pin_memory()
        hz = z.cpu().pin_memory()
        io = _lib.RenderIO()
        io.rays_o, io.rays_d, io.z_coarse, io.z_row_stride = _lib.ptr(hro), _lib.ptr(hrd), _lib.ptr(hz), 0
        for k, v in h.items():
            setattr(io, k, _lib.ptr(v))
        h2d = hro.numel() * 4 + hrd.numel() * 4 + hz.numel() * 4
        d2h = sum(v.numel() * 4 for v in h.values())

        if strong:
            # the call a trajectory renderer makes: dmnerf_render_frame_host on this rank's pixel range (rays generated on the
            # device: 84 bytes of camera in, the range's maps out to pinned host memory) + the all-gather of the image
            Kf = (C.c_float * 9)(*[float(v) for v in np.asarray(wl["K"], dtype=np.float32).reshape(-1)])
            cfs = [(C.c_float * 12)(*[float(v) for v in synth.workload(args.workload, frame=f)["c2w"][:3, :4].reshape(-1)]) for f in range(8)]
            hs = {k: torch.empty((hi - lo,) + shape, dtype=torch.float32).pin_memory() for k, shape in
                  (("rgb_fine", (3,)), ("depth_fine", ()), ("acc_fine", ()), ("ins_fine", (ins_num,)))}
            io = _lib.RenderIO()
            for k, v in hs.items():
                setattr(io, k, _lib.ptr(v))
            h2d = (9 + 12) * 4
            d2h = sum(v.numel() * 4 for v in hs.values())
            hstep = [0]

        def step_host():
            if strong:
                cf = cfs[hstep[0] % len(cfs)]
                hstep[0] += 1
                _lib.check(lib.dmnerf_render_frame_host(ctx.handle, Kf, cf, wl["H"], wl["W"], float(wl["near"]), float(wl["far"]),
                                                        lo, hi - lo, N_COARSE, N_IMPORTANCE, 0, impl, C.byref(io), ctx.stream()),
                           "dmnerf_render_frame_host")
                if world > 1:
                    gather_image({k: v.to(dev, non_blocking=True) for k, v in hs.items()}, world, pad_to=per)
                return
            _lib.check(lib.dmnerf_render_forward_host(ctx.handle, io, n_rays, N_COARSE, N_IMPORTANCE, 0, impl, ctx.stream()),
                       "dmnerf_render_forward_host")

        for _ in range(2):
            step_host()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw0 = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            step_host()
        e1.record()
        barrier()
        tw1 = time.perf_counter()
        e2e_ms = max(e0.elapsed_time(e1), 1e3 * (tw1 - tw0))        # host-synchronous call: wall clock is the honest one
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peaks = json.load(open(peaks_path))
        peak_tf, peak_src = float(peaks["bf16_tflops_sustained"]), "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
    else:
        peak_tf, peak_src = 1400.0, "fallback (B200_PROFILING.md sustained)"

    # ---- BASELINE configs[3]: training step, 1024 random rays, forward + backward through the native path + Adam
    train = None
    if world == 1 and not args.no_train:
        import types
        from dmnerf_b200.render import dm_nerf
        from dmnerf_b200.embedder import get_embedder
        from dmnerf_b200.helpers import get_select_full
        from dmnerf_b200.evaluator import ins_criterion, img2mse
        from dmnerf_b200.penalizer import ins_penalizer
        sel = torch.from_numpy(np.random.Generator(np.random.PCG64(0)).choice(n_rays, 1024, replace=False)).to(dev)
        rays = torch.stack([ro[sel], rd[sel]], 0)
        targs = types.SimpleNamespace(perturb=1.0, N_importance=N_IMPORTANCE, is_train=True, N_ins=None, tolerance=0.05, deta_w=0.05)
        pe, ve = get_embedder(10)[0], get_embedder(4)[0]
        zc = z[None].expand(1024, N_COARSE)
        tgt = torch.rand(1024, 3, device=dev)
        nc.train(); nf.train()
        opt = torch.optim.Adam(list(nc.parameters()) + list(nf.parameters()), lr=5e-4)

        def train_step():
            out = dm_nerf(rays, pe, ve, nc, nf, zc, targs)
            loss = ((out["rgb_fine"] - tgt) ** 2).mean() + ((out["rgb_coarse"] - tgt) ** 2).mean() + out["ins_fine"].mean()
            opt.zero_grad()
            loss.backward()
            opt.step()

        # the reference's whole iteration (train_dmsr.py:23-64) through the same call surface: ray selection, both Hungarian
        # instance losses (assignment on the device), both emptiness penalizers, backward, Adam
        gt_rgb = torch.rand(wl["H"], wl["W"], 3, device=dev)
        gt_lab = (torch.arange(n_rays, device=dev).reshape(wl["H"], wl["W"]) * min(7, ins_num) // n_rays).to(torch.int16)
        pose = torch.from_numpy(wl["c2w"]).to(dev)

        def full_iteration():
            target_c, target_i, batch_rays = get_select_full(gt_rgb, pose, wl["K"], gt_lab, 1024)
            info = dm_nerf(batch_rays, pe, ve, nc, nf, zc, targs)
            total = img2mse(info["rgb_coarse"], target_c) + img2mse(info["rgb_fine"], target_c) \
                + ins_criterion(info["ins_coarse"], target_i, ins_num)[0] + ins_criterion(info["ins_fine"], target_i, ins_num)[0] \
                + ins_penalizer(info["raw_coarse"], info["z_vals_coarse"], info["depth_coarse"], batch_rays[1], targs) \
                + ins_penalizer(info["raw_fine"], info["z_vals_fine"], info["depth_fine"], batch_rays[1], targs)
            opt.zero_grad()
            total.sum().backward()
            opt.step()

        def timed(fn, reps):
            for _ in range(3):
                fn()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize(dev)
            return 1e3 * (time.perf_counter() - t0) / reps, e0.elapsed_time(e1) / reps

        launches_t0 = _lib.launch_count()
        tms, tms_dev = timed(train_step, 10)
        launches_train = (_lib.launch_count() - launches_t0) // 13
        train_flops = 3.0 * synth.flops_per_ray(ins_num) * 1024          # SURVEY 8(d): forward + dX + dW, recompute / split not credited
        train = {"rays_per_step": 1024, "ms_per_step": tms, "device_ms_per_step": tms_dev, "rays_per_s": 1024 / (tms * 1e-3),
                 "native_launches_per_step": int(launches_train),
                 "roofline": {"bound": "tensor", "achieved": train_flops / (tms_dev * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                              "frac": train_flops / (tms_dev * 1e-3) / 1e12 / peak_tf,
                              "note": "algorithmic 3 x forward FLOPs (1.065 GFLOP/ray) over the whole step incl. Adam; CUDA events"},
                 "what": "dm_nerf(perturb=1) forward + backward through the native kernels + Adam step on 1024 random rays"}
        try:
            fms, fms_dev = timed(full_iteration, 5)
            train["full_iteration"] = {"ms_per_step": fms, "device_ms_per_step": fms_dev,
                                       "what": "train_dmsr.py:23-64 through the drop-in call surface: get_select_full (the reference's "
                                               "np.random.choice draw: a host-side shuffle of all H*W pixel indices, 3-4 ms, bounds "
                                               "this number), dm_nerf, 2 x MSE, 2 x ins_criterion (Hungarian assignment on the device, "
                                               "no host hop), 2 x ins_penalizer, backward, Adam"}
            os.environ["DMNERF_SELECT"] = "device"
            try:
                fms2, fms2_dev = timed(full_iteration, 10)
            finally:
                del os.environ["DMNERF_SELECT"]
            train["full_iteration_device_select"] = {"ms_per_step": fms2, "device_ms_per_step": fms2_dev,
                                                     "what": "the same iteration with DMNERF_SELECT=device (pixels drawn by the native "
                                                             "keyed-bijection kernel: uniform without replacement, not numpy's stream)"}
        except Exception as exc:                       # informational block: never fail the bench line because of it
            train["full_iteration"] = {"error": str(exc)}
        # SURVEY 8(f2): the emptiness penalizer on the fine network's per-sample outputs (forward + backward), HBM-streaming
        try:
            pargs = types.SimpleNamespace(tolerance=0.05, deta_w=0.05)
            praw = torch.randn(1024, N_COARSE + N_IMPORTANCE, 4 + ins_num + 1, device=dev, requires_grad=True)
            pz = (torch.rand(1024, N_COARSE + N_IMPORTANCE, device=dev).sort(-1).values * 11 + 4)
            pdep = pz[:, 100].clone()
            for _ in range(3):
                praw.grad = None
                ins_penalizer(praw, pz, pdep, rays[1], pargs).sum().backward()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(20):
                praw.grad = None
                ins_penalizer(praw, pz, pdep, rays[1], pargs).sum().backward()
            ev1.record()
            torch.cuda.synchronize(dev)
            pus = 1e3 * ev0.elapsed_time(ev1) / 20
            k1 = ins_num + 1
            pbytes = 1024 * (N_COARSE + N_IMPORTANCE) * (4 * (2 * k1 + k1) + 3 * 4)
            train["penalizer"] = {"us_per_fwd_bwd": pus, "algorithmic_GBps": pbytes / (pus * 1e-6) / 1e9,
                                  "what": "ins_penalizer on raw_fine [1024,192,%d] forward + backward; algorithmic bytes = raw logits "
                                          "read twice + gradient written once + z_vals three times" % (4 + k1)}
        except Exception as exc:
            train["penalizer"] = {"error": str(exc)}
        nc.eval(); nf.eval()
        if not args.no_cpu_baseline:
            try:
                r_off, _ = cpu_train_step(args.workload, anomaly=False)
                r_on, _ = cpu_train_step(args.workload, anomaly=True)
                train["cpu_reference"] = {"rays_per_s_anomaly_off": r_off, "rays_per_s_anomaly_on": r_on, "kind": "port",
                                          "what": "oracle port: dm_nerf(perturb=1) + the same loss + backward on 1024 rays, one step each, "
                                                  "torch CPU fp32, %d threads; the reference ships with anomaly mode ON (dm_nerf.py:5)" % torch.get_num_threads()}
            except Exception as exc:
                train["cpu_reference"] = {"error": str(exc)}

    total_rays = n_rays * (1 if strong else world) * args.steps
    value = total_rays / (dev_ms * 1e-3)
    e2e_value = total_rays / (e2e_ms * 1e-3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (fine network: F = 192 samples per ray)
    rays_rank = (hi - lo) if strong else n_rays
    fused = stage_ms[4] < 0.05 * stage_ms[0]                    # single-kernel pipeline: only stage 0 carries time
    if fused:
        fine_ms = stage_ms[0] / args.steps
        fine_flops = synth.flops_per_ray(ins_num) * rays_rank
        kname = "fused render kernel (coarse 64 + fine 192 network evaluations per ray, composite, sampling)"
    else:
        fine_ms = stage_ms[4] / args.steps
        fine_flops = 2.0 * (N_COARSE + N_IMPORTANCE) * synth.macs_per_sample(ins_num) * rays_rank
        kname = "fine-network MLP kernel (192 samples/ray)"
    achieved_tf = fine_flops / (fine_ms * 1e-3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch") if fused else None
    roofline = {"bound": "tensor", "kernel": kname, "achieved": achieved_tf,
                "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf, "traffic": traffic,
                "peak_source": peak_src,
                "note": "algorithmic FLOPs (2*693504 MACs per network evaluation, the reference's layer shapes); the kernel issues 3 bf16 "
                        "tensor passes (hi/lo operand split for fp32 parity) over 563200 padded+folded MACs per sample, so "
                        "frac cannot exceed 693504/(3*563200) = 0.410 of the bf16 peak",
                "stage_ms_per_step": {k: float(v / args.steps) for k, v in
                                      zip(("coarse_z_or_fused_kernel", "coarse_mlp", "coarse_composite", "hier_sample", "fine_mlp",
                                           "fine_composite"), stage_ms)}}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        r, cores, threads, rays, el = cpu_reference_rate(args.workload, args.cpu_seconds)
        cpu_baseline = {"value": r, "unit": "rays/s", "cores": cores, "kind": "port",
                        "sample": "%d rays (1024-ray chunks, full 64+128 pipeline) in %.1f s, torch CPU fp32, %d threads"
                                  % (rays, el, threads)}
        try:
            procs = args.cpu_procs or max(1, cores // max(threads, 1))
            if procs > 1:
                wr, got = cpu_whole_box_rate(args.workload, min(args.cpu_seconds, 10.0), procs, threads)
                cpu_baseline["whole_box"] = {"value": wr, "unit": "rays/s", "processes": got, "threads_each": threads,
                                             "what": "the same sample run by %d concurrent processes (all host cores busy), rates summed" % got}
            cpu_baseline["c1_coarse_only"] = cpu_c1_coarse_only(args.workload)
        except Exception as exc:
            cpu_baseline["extras_error"] = str(exc)

    line = {
        "metric": "rays/sec (64c+128f samples)", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32 (bf16x3 split operands on tcgen05, fp32 accumulate)" if args.mlp != "simt" else "f32",
        "data": "synthetic",
        "config": {"workload": workload_text(args.workload, ins_num, n_rays, args.scaling, world),
                   "name": args.workload, "rays_per_step_per_gpu": rays_rank, "l2": "256 MiB write between timed steps",
                   "mlp_impl": args.mlp,
                   "parallelism": ("one frame's pixels sharded by contiguous range, dp%d, rays generated per rank on the device, "
                                   "one NCCL all-gather of the image per frame" % world) if strong else
                                  ("rays sharded by frame, dp%d, one NCCL all-gather of the image per step" % world)},
        "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / args.steps,
                "api": ("dmnerf_render_frame_host on the rank's pixel range (C ABI, camera in, pinned host maps out) + all-gather"
                        if strong else "dmnerf_render_forward_host (C ABI, pinned host buffers)")},
        "gpu_launches": int(launches), "roofline": roofline, "clocks": clocks,
    }
    if strong:
        line["allgather"] = {"ms_per_frame": gather_ms / args.steps, "share_of_step": gather_ms / max(dev_ms, 1e-9),
                             "bytes_per_rank": int(per * (5 + ins_num) * 4) if world > 1 else 0,
                             "what": "NCCL all_gather_into_tensor of the packed [rays, 5 + ins_num] image slab, CUDA events on rank 0"}
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
    if train:
        line["train_step"] = train
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
