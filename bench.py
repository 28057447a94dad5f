#!/usr/bin/env python
"""Benchmark of the dense-BA update hot path (BASELINE.json metric: "BA-update iters/sec (512 edges, 344x64x48) at
1/2/4/8 B200; corr HBM GB/s vs peak").

One STEP = the droid_backends work of one FactorGraph.update (SURVEY.md section 8d): a 4-level radius-3
corr_index_forward over all edges + ba(iterations=2, lm=1e-4, ep=0.1) on a synthetic 512-edge / 72-keyframe graph at
48x64 (fp16 correlation volumes as in the live system).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--dump-outputs DIR]

* our arm: `value` times the step with all inputs resident in HBM, launched through the C ABI (ctypes); `e2e` goes
  through the pybind `droid_backends` API from pinned HOST buffers (per-step inputs H2D, BA results D2H inside the timed
  region; the correlation volumes are persistent device state exactly as in the reference, where they are produced on
  the GPU once per edge and never cross PCIe).
* N > 1 (torchrun, one rank per GPU): weak scaling in edges -- the graph has 512*N edges over the same 72-keyframe
  window, sharded by source frame (droid_slam_b200/sharded.py); one NCCL all-reduce of the reduced pose system per
  Gauss-Newton iteration; `value` = 512-edge-equivalents per second = N / step time (max over ranks).
* --impl reference: the UNMODIFIED reference CUDA kernels (oracle/_ref/droid_backends_ref: /root/reference/src built for
  sm_100a against the dense-LLT Eigen stand-in) on the same tensors, same protocol; corr_index is issued in chunks of
  128 edges because the reference's 32-bit accessors cannot address a 512-edge level-0 volume.  Falls back to the CPU
  oracle port when that build is absent.  Rank 0 only.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

EDGES_PER_GPU = 512
FRAMES = 72
HT, WD = 48, 64
RADIUS, LEVELS = 3, 4
BA_ITERS, LM, EP = 2, 1e-4, 0.1
CFG_NAME, SCALING, STEREO, WITH_CORR, RGBD = "metric", "weak", False, True, False

# BASELINE.json `configs` (SURVEY section 8d).  `metric` is the configuration the metric is quoted on (and the default); the others
# are selected with --config.  weak: `edges` per GPU (the graph grows with the GPU count over the same window); strong: `edges` in
# total, sharded by source frame over the GPUs.
CONFIGS = {
    "metric": dict(edges=512, frames=72, ht=48, wd=64, dtype="f16", itrs=2, lm=1e-4, ep=0.1, scaling="weak", corr=True, stereo=False),
    "c2": dict(edges=128, frames=25, ht=48, wd=64, dtype="f32", itrs=2, lm=1e-4, ep=0.1, scaling="weak", corr=True, stereo=False),
    "c3": dict(edges=2048, frames=400, ht=48, wd=64, dtype="f16", itrs=10, lm=1e-5, ep=1e-2, scaling="strong", corr=False, stereo=False),
    "c4": dict(edges=256, frames=64, ht=48, wd=64, dtype="f16", itrs=2, lm=1e-4, ep=0.1, scaling="weak", corr=True, stereo=True),
    "c5": dict(edges=8192, frames=1000, ht=72, wd=96, dtype="bf16", itrs=2, lm=1e-4, ep=0.1, scaling="strong", corr=True, stereo=False),
    # one rank's share of c5 on ONE GPU (1024 edges = 130 GB of bf16 volumes, 125 keyframes): the single-GPU proxy of the stress config
    "c5_rank": dict(edges=1024, frames=125, ht=72, wd=96, dtype="bf16", itrs=2, lm=1e-4, ep=0.1, scaling="strong", corr=True, stereo=False),
}


def select_config(args):
    """--config: BASELINE.json configs 2-5 at their stated sizes (the step keeps its definition: lookups over the rank's edges, if the
    config has correlation volumes, + one ba call with the config's iteration count and damping)"""
    global EDGES_PER_GPU, FRAMES, HT, WD, BA_ITERS, LM, EP, CFG_NAME, SCALING, STEREO, WITH_CORR
    c = CONFIGS[args.config]
    CFG_NAME, SCALING, STEREO, WITH_CORR = args.config, c["scaling"], c["stereo"], c["corr"]
    EDGES_PER_GPU, FRAMES, HT, WD, BA_ITERS, LM, EP = c["edges"], c["frames"], c["ht"], c["wd"], c["itrs"], c["lm"], c["ep"]
    if args.dtype is None:
        args.dtype = c["dtype"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 400 for the metric config = a >= 0.5 s timed region; 20 otherwise)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="metric", choices=sorted(CONFIGS.keys()), help="BASELINE.json config (default: the one the metric is quoted on)")
    ap.add_argument("--dtype", default=None, choices=["f16", "f32", "bf16"], help="correlation volume dtype (default: the config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--collective", default="auto", choices=["auto", "p2p", "nccl"], help="N>1: fused peer-to-peer reduction inside the solve kernel, or a NCCL all-reduce of the pose system; auto = p2p for pose systems up to 1024 unknowns (the metric window), nccl for the large global-BA systems (only 16 SMs pull peer data in the fused kernel)")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a captured CUDA graph (N=1)")
    ap.add_argument("--dropin-lookup", action="store_true", help="time the step with the four drop-in corr_index_forward launches on reference-layout volumes (round-1 definition) instead of the fused one-launch lookup on tiled volumes")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary kernels (update operator, volume build, altcorr, geometry, solve) timed for `rooflines`")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32): poses, disps, dx, dz of ba and "
                         "a fixed sample (seed 0) of the correlation lookup; rank 0, --impl ours")
    args = ap.parse_args()
    select_config(args)
    if args.steps is None:
        args.steps = 400 if (args.config == "metric" and args.impl == "ours") else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs is supported for --impl ours only")
    return args


# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, index):
        self.index = index; self.proc = None; self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def roofline_traffic():
    """dram bytes per step of the corr_index kernels from the committed ncu capture (profiles/), or None"""
    p = os.path.join(ROOT, "profiles", "corr_index_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


# ---------------------------------------------------------------------------------------------------------
def build_problem(args, rank, world, dev):
    """the rank's shard of the (512*world)-edge graph: BA tensors, correlation pyramid, lookup coordinates"""
    from droid_slam_b200 import sharded, synth
    cfg = dict(E=EDGES_PER_GPU * (world if SCALING == "weak" else 1), N=FRAMES, ht=HT, wd=WD, stereo=STEREO, itrs=BA_ITERS, lm=LM, ep=EP)
    on_device = cfg["E"] * HT * WD > 16 * 1024 * 1024     # the stress config's scene (57 M pixels x edges) is generated on the GPU: minutes -> seconds
    s = synth.make_scene(cfg, seed=0, device=dev if on_device else "cpu")
    bounds = sharded.partition_frames(s["ii"], FRAMES, world)
    lo, hi = bounds[rank]
    idx = sharded.shard_edges(s["ii"], lo, hi)
    dtype = {"f16": torch.float16, "f32": torch.float32, "bf16": torch.bfloat16}[args.dtype]
    sub = dict(s); sub["ii"] = s["ii"][idx]; sub["jj"] = s["jj"][idx]; sub["coords_gt"] = s["coords_gt"][idx.to(s["coords_gt"].device)]
    if on_device:                                           # keep only this rank's shard, on the host like the CPU-generated scenes
        ix = idx.to(dev)
        s = dict(s, targets=s["targets"][ix].cpu(), weights=s["weights"][ix].cpu(), coords_gt=None, **{k: s[k].cpu() for k in ("poses", "disps", "disps_sens", "intrinsics", "eta", "poses_gt", "disps_gt")})
        idx_local = torch.arange(int(idx.numel()))
    else:
        idx_local = idx
    sub["cfg"] = dict(cfg, E=int(idx.numel()))
    if WITH_CORR:
        need = int(idx.numel()) * (HT * WD) ** 2 * 1.33 * (4 if dtype == torch.float32 else 2)
        free = torch.cuda.mem_get_info(dev)[0]
        if need > 0.9 * free:
            raise SystemExit("config %s: %.0f GB of correlation volumes per GPU do not fit (%.0f GB free); use more GPUs" % (CFG_NAME, need / 1e9, free / 1e9))
        pyr, coords, _ = synth.make_corr_inputs(sub, dtype=dtype, device=dev, edge_chunk=32 if HT * WD <= 3072 else 4)
    else:
        pyr, coords = [], torch.zeros(int(idx.numel()), 2, HT, WD, device=dev)
    kx = torch.unique(torch.cat([torch.arange(s["t0"], s["t1"]), s["ii"]]))
    eta_f = torch.zeros(FRAMES, HT, WD); eta_f[kx] = s["eta"]
    host = dict(poses=s["poses"], disps=s["disps"], disps_sens=s["disps_sens"], intrinsics=s["intrinsics"], targets=s["targets"][idx_local].contiguous(),
                weights=s["weights"][idx_local].contiguous(), eta=s["eta"], eta_by_frame=eta_f, ii=sub["ii"].contiguous(), jj=sub["jj"].contiguous(),
                coords=coords.cpu())
    return dict(scene=s, host=host, bounds=bounds, pyr=pyr, coords=coords, E=int(idx.numel()), dtype=dtype, t0=s["t0"], t1=s["t1"], M=s["M"])


def alg_bytes_corr(E, dtype):
    s = 4 if dtype == torch.float32 else 2
    return E * HT * WD * (LEVELS * ((2 * RADIUS + 2) ** 2 + (2 * RADIUS + 1) ** 2) * s + LEVELS * 8)     # SURVEY 8d: HW*(452 s + 32)


# ---------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, dev):
    import droid_slam_b200
    from droid_slam_b200 import c_api, sharded
    be = droid_slam_b200.install()          # raises if the native extension is missing: no fallback
    L = c_api.load()
    pb = build_problem(args, rank, world, dev)
    h = pb["host"]
    E, dtype = pb["E"], pb["dtype"]
    dcode = {torch.float16: c_api.DBA_F16, torch.float32: c_api.DBA_F32, torch.bfloat16: c_api.DBA_BF16}[dtype]
    d = {k: v.to(dev) for k, v in h.items()}
    pristine_poses, pristine_disps = d["poses"].clone(), d["disps"].clone()
    NL = LEVELS if WITH_CORR else 0
    coords_l = [(pb["coords"] / 2 ** l).contiguous() for l in range(NL)]
    corr_out = [torch.empty(E, 7, 7, HT, WD, dtype=dtype, device=dev) for _ in range(NL)]
    # fused lookup (CorrBlock.__call__ in one launch, droid_slam_b200.modules.install_corr_volume_hook(fused_lookup=True)): levels 0 and 1 of
    # the volumes in the tiled layout corr_volume_pyramid(tiled=True) writes -- same values, same outputs, bit for bit (tests/test_parity_gpu.py)
    FUSED = WITH_CORR and dtype == torch.float16 and WD % 64 == 0 and HT % 8 == 0 and not args.dropin_lookup
    pyr_t, corr196 = None, None
    if FUSED:
        def tile(v, l):
            h2, w2 = HT >> l, WD >> l
            return v.view(E, HT, WD, h2 // 4, 4, w2 // 8, 8).permute(0, 1, 2, 3, 5, 4, 6).contiguous().view(E, HT, WD, h2, w2)
        pyr_t = [tile(pb["pyr"][0], 0), tile(pb["pyr"][1], 1), pb["pyr"][2], pb["pyr"][3]]
        corr196 = torch.empty(E, 196, HT, WD, dtype=dtype, device=dev)
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    spbox = [sp]
    engine = sharded.CApiEngine(dev)
    p2p = None
    if args.collective == "auto":
        args.collective = "p2p" if 6 * (pb["t1"] - pb["t0"]) <= 1024 else "nccl"
    if world > 1 and args.collective == "p2p":
        # every rank first agrees that symmetric memory can be tried at all, so that no rank enters the rendezvous collective alone
        try:
            import torch.distributed._symmetric_memory as _symm  # noqa: F401
            can = 1.0
        except Exception:
            can = 0.0
        okc = torch.tensor([can], device=dev)
        dist.all_reduce(okc, op=dist.ReduceOp.MIN)
        try:
            if float(okc) == 0.0:
                raise RuntimeError("torch.distributed._symmetric_memory is not importable on every rank")
            p2p = sharded.P2PSystem(6 * (pb["t1"] - pb["t0"]), dev)
        except Exception as e:                       # no peer-mapped memory on this box: plain NCCL all-reduce of the pose system
            sys.stderr.write("[bench] rank %d: symmetric memory unavailable (%s); using the NCCL all-reduce path\n" % (rank, str(e)[:160]))
            p2p = None
        okp = torch.tensor([1.0 if p2p is not None else 0.0], device=dev)
        dist.all_reduce(okp, op=dist.ReduceOp.MIN)   # all ranks take the same path
        if float(okp) == 0.0:
            p2p = None
    drv = sharded.ShardedBA(engine, p2p=p2p)

    def lookup_dropin(sp_):
        for l in range(NL):
            v = pb["pyr"][l]
            c_api.check(L.dba_corr_index_forward(ctypes.c_void_p(v.data_ptr()), ctypes.c_void_p(coords_l[l].data_ptr()),
                                                 ctypes.c_void_p(corr_out[l].data_ptr()), E, HT, WD, v.shape[3], v.shape[4], RADIUS, dcode, sp_), "corr")

    def step_resident(ev=None):
        d["poses"].copy_(pristine_poses); d["disps"].copy_(pristine_disps)
        if ev: ev[0].record()
        if FUSED:
            c_api.check(L.dba_corr_lookup_pyramid(*[ctypes.c_void_p(v.data_ptr()) for v in pyr_t], ctypes.c_void_p(pb["coords"].data_ptr()),
                                                  ctypes.c_void_p(corr196.data_ptr()), E, HT, WD, 3, dcode, spbox[0]), "corr_lookup_pyramid")
        else:
            lookup_dropin(spbox[0])
        if ev: ev[1].record()
        drv.run(d["poses"], d["disps"], d["intrinsics"], d["disps_sens"], d["targets"], d["weights"], d["eta_by_frame"], d["ii"], d["jj"],
                pb["t0"], pb["t1"], BA_ITERS, LM, EP, pb["bounds"], exchange_disps=(world > 1))

    def barrier():
        torch.cuda.synchronize()
        if world > 1: dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step_resident()
    barrier()
    # the whole step (4 lookups + prepare + 2 x (build, Schur, [publish,] Cholesky, back-substitution, retraction) [+ depth exchange])
    # is a static launch sequence with no host synchronisation, so it is captured once into a CUDA graph and replayed (the C ABI is
    # capture-safe; for N > 1 the peer-to-peer epoch lives on the device and NCCL's depth all-reduce is captured with the rest)
    use_graph = not args.no_graph and BA_ITERS % 2 == 0
    graph = None
    if use_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    spbox[0] = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
                    step_resident()
                    spbox[0] = sp
            torch.cuda.current_stream().wait_stream(side)
            for _ in range(3):
                graph.replay()
        except Exception as e:                       # capture refused (e.g. a collective that cannot be captured): launch eagerly
            sys.stderr.write("[bench] CUDA graph capture failed on rank %d, falling back to eager launches: %s\n" % (rank, str(e)[:200]))
            spbox[0] = sp
            graph = None
            use_graph = False
        if world > 1:                                # every rank replays the graph or none does
            okf = torch.tensor([1.0 if graph is not None else 0.0], device=dev)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            if float(okf) == 0.0:
                graph, use_graph = None, False
        barrier()
    sampler = ClockSampler(torch.cuda.current_device()); sampler.start()
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_beg.record()
    for k in range(args.steps):
        if graph is not None:
            graph.replay()
        else:
            step_resident()
    t_end.record()
    barrier()
    clocks = sampler.stop()
    ms_total = t_beg.elapsed_time(t_end)
    outputs = snapshot_outputs(d, engine, corr196 if FUSED else corr_out) if args.dump_outputs and rank == 0 else None
    # the dominant kernel on its own stream position: the four corr_index launches of a step, CUDA events around them
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for k in range(args.steps):
        step_resident(evs[k])
    barrier()
    corr_ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps
    t = torch.tensor([ms_total, corr_ms], device=dev, dtype=torch.float64)
    if world > 1: dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t[0]) / args.steps
    corr_ms = float(t[1])
    dropin_ms = None
    if FUSED and world == 1:      # the four drop-in launches on the reference-layout volumes, for comparison (and equality of the results)
        dropin_ms = _time_ms(lambda: lookup_dropin(sp), iters=min(args.steps, 20), warm=3)
        ref196 = torch.cat([c.view(E, 49, HT, WD) for c in corr_out], 1)
        if not torch.equal(ref196, corr196):
            raise RuntimeError("fused tiled lookup and the drop-in corr_index_forward launches disagree")
        del ref196

    # ---- end to end through the public pybind API from pinned host buffers
    pin = {k: h[k].pin_memory() for k in ("coords", "targets", "weights", "eta", "eta_by_frame", "poses", "disps", "disps_sens", "ii", "jj", "intrinsics")}
    P = pb["t1"] - pb["t0"]
    out_pin = dict(poses=torch.empty(FRAMES, 7).pin_memory(), disps=torch.empty(FRAMES, HT, WD).pin_memory(), dx=torch.empty(P, 6).pin_memory())
    h2d = sum(pin[k].numel() * pin[k].element_size() for k in ("coords", "targets", "weights", "poses", "disps", "disps_sens", "ii", "jj", "intrinsics"))
    h2d += pin["eta"].numel() * 4 if world == 1 else pin["eta_by_frame"].numel() * 4
    d2h = sum(v.numel() * v.element_size() for v in out_pin.values())

    copy_stream = torch.cuda.Stream()

    def step_e2e():
        # user-level pipelining: the lookup only needs the coordinates, so the BA inputs travel on a second stream while the
        # four corr_index_forward launches run; everything still happens inside the timed region
        main = torch.cuda.current_stream()
        coords = pin["coords"].to(dev, non_blocking=True)
        copy_stream.wait_stream(main)
        with torch.cuda.stream(copy_stream):
            g = {k: pin[k].to(dev, non_blocking=True) for k in pin if k not in ("eta", "eta_by_frame", "coords")}
            eta = (pin["eta"] if world == 1 else pin["eta_by_frame"]).to(dev, non_blocking=True)
        feats = []
        if FUSED:
            feats.append(be.corr_lookup_pyramid(pyr_t, coords, True))                   # CorrBlock.__call__ through the fused-lookup hook
        for l in range(0 if FUSED else NL):
            corr, = be.corr_index_forward(pb["pyr"][l], coords / 2 ** l, RADIUS)       # reference call pattern, modules/corr.py:46-48
            feats.append(corr)
        main.wait_stream(copy_stream)
        for t in list(g.values()) + [eta]:
            t.record_stream(main)
        if world == 1:
            dx, dz = be.ba(g["poses"], g["disps"], g["intrinsics"], g["disps_sens"], g["targets"], g["weights"], eta, g["ii"], g["jj"],
                           pb["t0"], pb["t1"], BA_ITERS, LM, EP, False)
        else:
            drv.run(g["poses"], g["disps"], g["intrinsics"], g["disps_sens"], g["targets"], g["weights"], eta, g["ii"], g["jj"],
                    pb["t0"], pb["t1"], BA_ITERS, LM, EP, pb["bounds"], exchange_disps=True)
            dx = engine.dx
        out_pin["poses"].copy_(g["poses"], non_blocking=True); out_pin["disps"].copy_(g["disps"], non_blocking=True)
        out_pin["dx"].copy_(dx, non_blocking=True)
        return feats

    def time_e2e(fn):
        for _ in range(3):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1: dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]) / args.steps

    e2e_eager_ms = time_e2e(step_e2e)
    copy_only_ms = time_e2e(lambda: [pin[k].to(dev, non_blocking=True) for k in pin if k != ("eta_by_frame" if world == 1 else "eta")])     # PCIe share of the step
    e2e_ms, e2e_mode = e2e_eager_ms, "eager"
    if use_graph:
        # the same calls captured once: pinned-host -> device copies, the four lookups, ba and the device -> pinned-host reads are all
        # nodes of one CUDA graph (the copies of the BA inputs form a parallel branch), so a step is a single graph launch
        stat = {k: torch.empty_like(pin[k], device=dev) for k in pin if k != ("eta_by_frame" if world == 1 else "eta")}
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        e2e_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(e2e_graph, stream=side):
            main = torch.cuda.current_stream()
            stat["coords"].copy_(pin["coords"], non_blocking=True)
            copy_stream.wait_stream(main)
            with torch.cuda.stream(copy_stream):
                for k in stat:
                    if k != "coords":
                        stat[k].copy_(pin[k], non_blocking=True)
            keep = [be.corr_lookup_pyramid(pyr_t, stat["coords"], True)] if FUSED else [be.corr_index_forward(pb["pyr"][l], stat["coords"] / 2 ** l, RADIUS)[0] for l in range(NL)]
            main.wait_stream(copy_stream)
            if world == 1:
                dx, dz = be.ba(stat["poses"], stat["disps"], stat["intrinsics"], stat["disps_sens"], stat["targets"], stat["weights"], stat["eta"],
                               stat["ii"], stat["jj"], pb["t0"], pb["t1"], BA_ITERS, LM, EP, False)
            else:
                drv.run(stat["poses"], stat["disps"], stat["intrinsics"], stat["disps_sens"], stat["targets"], stat["weights"], stat["eta_by_frame"],
                        stat["ii"], stat["jj"], pb["t0"], pb["t1"], BA_ITERS, LM, EP, pb["bounds"], exchange_disps=True)
                dx = engine.dx
            out_pin["poses"].copy_(stat["poses"], non_blocking=True); out_pin["disps"].copy_(stat["disps"], non_blocking=True)
            out_pin["dx"].copy_(dx, non_blocking=True)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        e2e_ms, e2e_mode = time_e2e(e2e_graph.replay), "cuda graph replay (copies, lookups, ba and result reads captured as one graph)"
        torch.cuda.synchronize()
        # the graph must produce what the eager call sequence produces
        chk_p, chk_d = out_pin["poses"].clone(), out_pin["disps"].clone()
        step_e2e(); torch.cuda.synchronize()
        # (fp64 atomics make the pose system's summation order run-dependent; ten ill-conditioned GN iterations amplify that, hence the
        #  looser bound for the global-BA configs)
        tol = dict(rtol=1e-4, atol=1e-6) if BA_ITERS <= 2 else dict(rtol=1e-2, atol=1e-3)
        if not (torch.allclose(chk_p, out_pin["poses"], **tol) and torch.allclose(chk_d, out_pin["disps"], **tol)):
            raise RuntimeError("e2e graph replay and eager call sequence disagree (poses %.2e, disps %.2e)" % (
                float((chk_p - out_pin["poses"]).abs().max()), float((chk_d - out_pin["disps"]).abs().max())))

    if rank != 0:
        return
    peak, peak_src = measured_peak()
    alg = alg_bytes_corr(E, dtype)
    achieved = alg / (corr_ms * 1e-3) / 1e9 if (WITH_CORR and corr_ms > 0) else 0.0
    traffic = roofline_traffic()
    launches_per_step = (1 if FUSED else NL) + 2 + BA_ITERS * 6        # corr x4, prepare+csr, per GN iter: build, schur x2, chol, backsub, pose_retr
    Ptot = pb["t1"] - pb["t0"]
    sys_bytes = 8 * (36 * Ptot * Ptot + 6 * Ptot)
    mult = world if SCALING == "weak" else 1
    if CFG_NAME == "metric":
        metric, unit = "BA-update iters/sec (512 edges, 344x64x48)", "iters/s (512-edge equivalents)"
        workload = "metric: %d edges/GPU x %d GPU(s) over a %d-keyframe window at %dx%d, 4-level r=3 correlation lookup (%s) + ba(itrs=2, lm=1e-4, ep=0.1)" % (
            EDGES_PER_GPU, world, FRAMES, HT, WD, "one fused launch on the tiled volumes of corr_volume_pyramid(tiled=True); the four drop-in corr_index_forward launches are reported under dropin_lookup" if FUSED else "4 x corr_index_forward")
    else:
        metric, unit = "BA-update iters/sec (BASELINE config %s)" % CFG_NAME, "iters/s (one step = %sba(itrs=%d))" % ("4-level corr_index_forward + " if WITH_CORR else "", BA_ITERS)
        workload = "%s: %d edges %s, %d keyframes at %dx%d, %s volumes, %sba(itrs=%d, lm=%g, ep=%g)%s" % (
            CFG_NAME, EDGES_PER_GPU, "per GPU" if SCALING == "weak" else "in total (sharded over %d GPU(s))" % world, FRAMES, HT, WD, args.dtype,
            "4-level r=3 corr_index_forward + " if WITH_CORR else "no lookup (global BA backend), ", BA_ITERS, LM, EP, ", one (i,i) stereo edge per frame" if STEREO else "")
    line = {
        "metric": metric, "value": mult * 1e3 / ms_step, "unit": unit,
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": SCALING, "vs_baseline": None, "dtype": "f32 (BA solve in f64), %s corr volumes" % args.dtype, "data": "synthetic",
        "impl": "ours",
        "config": {"workload": workload, "name": CFG_NAME,
                   "edges_this_rank": E, "frames": FRAMES, "depth_frames": pb["M"], "pose_system": 6 * Ptot,
                   "parallelism": ("edge-sharded by source frame; the %d-double pose system is reduced once per GN iteration, %s" % (36 * P * P + 6 * P, "fused into the Cholesky kernel (peer-to-peer loads over NVLink, release/acquire flags)" if p2p is not None else "NCCL all-reduce")) if world > 1 else "single GPU",
                   "l2": ("inputs larger than L2: %.1f GB of correlation volumes stream through the 126 MB L2 every step" % (sum(v.numel() * v.element_size() for v in pb["pyr"]) / 1e9)) if WITH_CORR else
                         "BA inputs of %.0f MB per rank; L2 not flushed between steps (the reference keeps them resident too)" % (E * HT * WD * 16 / 1e6)},
        "e2e": {"value": mult * 1e3 / e2e_ms, "unit": unit, "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "launch_mode": e2e_mode, "eager_ms_per_step": e2e_eager_ms, "h2d_copy_only_ms": copy_only_ms,
                "api": "droid_backends." + ("corr_lookup_pyramid" if FUSED else "corr_index_forward x4") + " + droid_backends.ba from pinned host buffers (BA inputs copied on a second stream during the lookups); volumes persistent on device"},
        "gpu_launches": launches_per_step * args.steps, "launch_mode": "cuda graph replay" if graph is not None else "eager",
        "clocks": clocks,
        "ba_ms_per_step": ms_step - corr_ms, "ms_per_gn_iteration": (ms_step - corr_ms) / BA_ITERS,
        "pose_system_reduction": {"bytes_per_gn_iteration": sys_bytes, "nvlink_bytes_per_gn_iteration_per_gpu": (sys_bytes * (world - 1) if p2p is not None else int(2 * sys_bytes * (world - 1) / max(world, 1))) if world > 1 else 0,
                                  "how": ("every rank reads the %d peer copies inside the solve kernel" % (world - 1)) if p2p is not None else ("NCCL ring all-reduce (2(N-1)/N x bytes per GPU)" if world > 1 else "none")},
    }
    if WITH_CORR:
        kname = "corr_lookup_pyramid_f16_kernel<tiled levels 0-1> (1 launch/step: all 4 levels)" if FUSED else "corr_index_fwd_%s_r3_kernel (4 launches/step)" % args.dtype
        line["roofline"] = {"kernel": kname, "bound": "hbm", "achieved": achieved, "peak": peak,
                            "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src, "algorithmic_bytes_per_step": alg,
                            "kernel_ms_per_step": corr_ms, "share_of_step": corr_ms / ms_step,
                            "traffic": (traffic or {}).get("dram_bytes_per_step_" + ("fused_tiled_f16" if FUSED else args.dtype)),
                            "traffic_source": "ncu dram__bytes_read.sum + dram__bytes_write.sum of the four launches, profiles/ (captured once per kernel change, not re-measured by this run)"}
    else:
        alg_ba = BA_ITERS * (16 * E * HT * WD + 16 * pb["M"] * HT * WD + 28 * FRAMES)
        line["roofline"] = {"kernel": "ba (build + Schur + solve + back-substitution per GN iteration)", "bound": "hbm", "achieved": alg_ba / ((ms_step - corr_ms) * 1e-3) / 1e9,
                            "peak": peak, "unit": "GB/s", "frac": alg_ba / ((ms_step - corr_ms) * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                            "algorithmic_bytes_per_step": alg_ba, "traffic": None,
                            "note": "SURVEY 8d BA bytes (16 E HW + 16 M HW + 28 N per iteration); the step is latency / solve bound, not HBM bound"}
    if dropin_ms is not None:
        line["dropin_lookup"] = {"kernel": "corr_index_fwd_f16_r3_kernel (4 launches on reference-layout volumes, the round-1 step)", "kernel_ms_per_step": dropin_ms,
                                 "achieved": alg / (dropin_ms * 1e-3) / 1e9, "frac": alg / (dropin_ms * 1e-3) / 1e9 / peak, "unit": "GB/s",
                                 "step_ms_with_dropin_lookup": ms_step - corr_ms + dropin_ms, "value_with_dropin_lookup": mult * 1e3 / (ms_step - corr_ms + dropin_ms),
                                 "traffic": (traffic or {}).get("dram_bytes_per_step_" + args.dtype), "outputs": "bit-identical to the fused lookup (checked in this run)"}
    if world == 1 and not args.no_extras:
        extras = secondary_kernels(E, dev, ms_step, L, be, cpu_legs=not args.no_cpu_baseline)
        line["update_operator"] = extras.pop("update_operator")
        line["rooflines"] = extras["rooflines"]
    if world == 1 and not args.no_cpu_baseline and CFG_NAME in ("metric", "c2", "c4"):
        line["cpu_baseline"] = cpu_baseline(pb)
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))


CORR_SAMPLE = 4 << 20     # lookup values kept by --dump-outputs (16 MB as float32)


def snapshot_outputs(d, engine, corr):
    """host copies of what the last timed step computed: ba's in-place poses / disps and its dx / dz, and a fixed seeded sample of the
    4-level lookup in the [E, 196, ht, wd] layout of CorrBlock.__call__ (the fused launch writes that layout, the drop-in launches
    are concatenated into it)"""
    out = {k: d[k].float().cpu() for k in ("poses", "disps")}
    out["dx"], out["dz"] = engine.dx.float().cpu(), engine.dz.float().cpu()
    if isinstance(corr, list):
        corr = torch.cat([c.view(c.shape[0], 49, HT, WD) for c in corr], 1) if corr else None
    if corr is not None:
        flat = corr.reshape(-1)
        idx = torch.randint(0, flat.numel(), (min(CORR_SAMPLE, flat.numel()),), generator=torch.Generator().manual_seed(0))
        out["corr_sample"] = flat[idx.to(flat.device)].float().cpu()
    return out


def write_outputs(dirname, outputs):
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(dirname, name + ".npy"), t.numpy().astype(np.float32))


def _time_ms(fn, iters=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def secondary_kernels(E, dev, ms_step, L, be, cpu_legs=True):
    """The other kernels of the path, each timed on its own with CUDA events (not part of `value`): the update operator (row A6,
    tcgen05 convolutions), the correlation-volume build (A7), altcorr (A2), the streaming geometry ops (A8-A11) and the fp64 solve.
    Each entry carries its algorithmic work (SURVEY 8d) and the roofline it is held against.  Failures are reported, never raised."""
    out = {"update_operator": None, "rooflines": []}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    tf_burst, tf_sust = float(peaks.get("bf16_tflops", 1590.0)), float(peaks.get("bf16_tflops_sustained", 1400.0))
    src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
    from droid_slam_b200 import synth
    g = torch.Generator(device=dev).manual_seed(7)
    # ---- update operator: same E edges as the step, 72 source frames
    try:
        from droid_slam_b200.update import UpdateModule
        mod = UpdateModule().to(dev)
        mod.load_state_dict({k: v.to(dev) for k, v in synth.make_update_weights(0).items()})
        net = torch.tanh(torch.randn(1, E, 128, HT, WD, generator=g, device=dev)).half()
        inp = torch.relu(torch.randn(1, E, 128, HT, WD, generator=g, device=dev)).half()
        corr = torch.randn(1, E, 196, HT, WD, generator=g, device=dev).half()
        motn = torch.randn(1, E, 4, HT, WD, generator=g, device=dev)
        ii = torch.arange(E, device=dev) % FRAMES
        with torch.no_grad():
            ms = _time_ms(lambda: mod(net, inp, corr, motn, ii))
        flops = (14.03e9 * E + 1.37e9 * min(E, FRAMES)) * (HT * WD / 3072.0)              # SURVEY 8d
        out["update_operator"] = {"ms": ms, "full_update_ms": ms + ms_step, "edges": E, "tflops": flops / ms / 1e9,
                                  "impl": "droid_slam_b200.UpdateModule: tcgen05 implicit-GEMM convolutions (csrc/update_op.cu), reference-layout (NCHW) inputs, f16 operands / fp32 accumulation; "
                                          "not part of `value`; the reference formula through torch/cuDNN is timed by --impl reference"}
        out["rooflines"].append({"kernel": "update operator (conv_tc_kernel x12 + layout / aggregation kernels)", "bound": "tensor", "achieved": flops / ms / 1e9, "peak": tf_sust, "unit": "TFLOP/s",
                                 "frac": flops / ms / 1e9 / tf_sust, "peak_source": src + " bf16_tflops_sustained (a 10+ ms tensor-bound kernel sequence runs under the power cap)", "ms": ms,
                                 "algorithmic_flops": flops})
        del net, inp, corr, motn, mod
    except Exception as e:
        out["update_operator"] = {"ms": None, "error": str(e)[:200]}
    # ---- correlation volume build (128 edges)
    try:
        if be.corr_volume_supported(128, HT, WD):
            n_e = 128
            fm = torch.randn(FRAMES, 128, HT, WD, generator=g, device=dev).half()
            ii = torch.arange(n_e, device=dev) % FRAMES; jj = (ii + 1) % FRAMES
            ms = _time_ms(lambda: be.corr_volume_pyramid(fm, fm, ii, jj))
            byts = n_e * (HT * WD) ** 2 * 2 * 1.328125
            out["rooflines"].append({"kernel": "corr_volume_pyramid_kernel (128 edges)", "bound": "hbm", "achieved": byts / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": byts / ms / 1e6 / hbm,
                                     "peak_source": src, "ms": ms, "algorithmic_bytes": byts, "tflops": 2.0 * n_e * (HT * WD) ** 2 * 128 / ms / 1e9})
            del fm
    except Exception as e:
        out["rooflines"].append({"kernel": "corr_volume_pyramid_kernel", "error": str(e)[:200]})
    # ---- altcorr (48 edges, 4 levels)
    try:
        n_e = 48
        fm = torch.randn(1, 16, 128, HT, WD, generator=g, device=dev).half()
        pyr = [fm]
        for _ in range(3):
            pyr.append(torch.nn.functional.avg_pool2d(pyr[-1][0], 2, stride=2)[None].contiguous())
        sc = synth.make_scene(dict(E=n_e, N=16, ht=HT, wd=WD, stereo=False, itrs=1, lm=1e-4, ep=0.1), seed=2)
        coords = sc["coords_gt"].permute(0, 3, 1, 2)[None].contiguous().to(dev)
        ii, jj = sc["ii"].to(dev), sc["jj"].to(dev)
        cl = [(coords / 2 ** l).contiguous() for l in range(4)]
        ms = _time_ms(lambda: [be.altcorr_forward(fm, pyr[l], cl[l], ii, jj, 3) for l in range(4)])
        byts = n_e * (128 * HT * WD * 2 * (1 + 1.328125) + 8 * HT * WD * 4 + 4 * 49 * HT * WD * 2)
        fl = 2.0 * 4 * HT * WD * 64 * 128 * n_e
        out["rooflines"].append({"kernel": "altcorr_forward_kernel (48 edges x 4 levels)", "bound": "hbm", "achieved": byts / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": byts / ms / 1e6 / hbm,
                                 "peak_source": src, "ms": ms, "algorithmic_bytes": byts, "tflops": fl / ms / 1e9,
                                 "note": "compulsory bytes (SURVEY 8d); the kernel is a SIMT gather + 128-channel dot product, far from this bound"})
        del fm, pyr
    except Exception as e:
        out["rooflines"].append({"kernel": "altcorr_forward_kernel", "error": str(e)[:200]})
    # ---- streaming geometry at the step's scene size
    try:
        sc = synth.make_scene(dict(E=512, N=FRAMES, ht=HT, wd=WD, stereo=False, itrs=1, lm=1e-4, ep=0.1), seed=0)
        P, D, K, ii, jj = [sc[k].to(dev) for k in ("poses", "disps", "intrinsics", "ii", "jj")]
        hw = HT * WD
        a, b = torch.meshgrid(torch.arange(FRAMES), torch.arange(FRAMES), indexing="ij")
        a, b = a.reshape(-1).to(dev), b.reshape(-1).to(dev)
        ix = torch.arange(FRAMES, device=dev); th = torch.full((FRAMES,), 0.05, device=dev)
        for name, fn, byts in (("projmap_kernel (512 edges)", lambda: be.projmap(P, D, K, ii, jj), 512 * hw * 20),
                               ("iproj_kernel (%d frames)" % FRAMES, lambda: be.iproj(P, D, K), FRAMES * hw * 16),
                               ("frame_distance_kernel (%d pairs)" % (FRAMES * FRAMES), lambda: be.frame_distance(P, D, K, a, b, 0.3), FRAMES * FRAMES * hw * 4),
                               ("depth_filter_kernel (%d frames)" % FRAMES, lambda: be.depth_filter(P, D, K, ix, th), FRAMES * hw * 8)):
            ms = _time_ms(fn, iters=10)
            out["rooflines"].append({"kernel": name, "bound": "hbm", "achieved": byts / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": byts / ms / 1e6 / hbm, "peak_source": src, "ms": ms,
                                     "algorithmic_bytes": byts, "note": "L2-resident working set at this size: launch / latency bound"})
    except Exception as e:
        out["rooflines"].append({"kernel": "geometry ops", "error": str(e)[:200]})
    # ---- fp64 damped solve at the step's system size
    try:
        n = 6 * (FRAMES - 1)
        A = torch.randn(n, n, generator=g, device=dev, dtype=torch.float64)
        H = (A @ A.t() + n * torch.eye(n, device=dev, dtype=torch.float64)).contiguous()
        bvec = torch.randn(n, generator=g, device=dev, dtype=torch.float64)
        x = torch.empty(n, device=dev); fail = torch.zeros(1, dtype=torch.int32, device=dev)
        wsb = L.dba_solve_workspace_bytes(n)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        vp = lambda t: ctypes.c_void_p(t.data_ptr())
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        ms = _time_ms(lambda: L.dba_solve_spd(vp(H), vp(bvec), n, ctypes.c_float(1e-4), ctypes.c_float(0.1), vp(x), vp(fail), vp(ws), ctypes.c_size_t(wsb), st), iters=20)
        fl = n ** 3 / 3.0
        kname = "chol_resident_kernel" if n <= 448 and os.environ.get("DBA_CHOL_RESIDENT", "1") != "0" else "chol_cluster_kernel"
        out["rooflines"].append({"kernel": "%s (n = %d, fp64)" % (kname, n), "bound": "fp64 issue rate", "achieved": fl / ms / 1e9, "peak": 34.0, "unit": "TFLOP/s", "frac": fl / ms / 1e9 / 34.0,
                                 "peak_source": "measured fp64 FMA issue rate (profiles/r1_fp64_issue_rate.txt)", "ms": ms, "algorithmic_flops": fl,
                                 "note": "latency bound: a chain of n/32 dependent column steps (potrf -> substitution -> update), the figure of merit is the time"})
    except Exception as e:
        out["rooflines"].append({"kernel": "chol_cluster_kernel", "error": str(e)[:200]})
    # ---- row F1: proximity edge selection (frontend window and a global-BA sized grid), with the reference's Python loop restated on the CPU beside it
    try:
        import time as _time
        _prox = None
        if cpu_legs:                                         # CPU baseline leg (like `cpu_baseline`): the oracle is only ever the thing timed beside / checked against
            import oracle.proximity as _prox
        for (t, t0, t1, nms, th, mf, tag) in ((30, 25, 5, 1, 16.0, -1, "frontend window 5 x 25 pairs"), (400, 0, 0, 2, 22.0, -1, "global BA 400 x 400 pairs")):
            gg = torch.Generator().manual_seed(11)
            ni, nj = t - t0, t - t1
            fi = torch.arange(t0, t, dtype=torch.float32)[:, None]; fj = torch.arange(t1, t, dtype=torch.float32)[None, :]
            dm = (6.0 * (fi - fj).abs() * (0.6 + 0.8 * torch.rand(ni, nj, generator=gg)) + torch.rand(ni, nj, generator=gg)).reshape(-1)
            dm = torch.where(torch.rand(ni * nj, generator=gg) < 0.08, 2.0 + 12.0 * torch.rand(ni * nj, generator=gg), dm)
            dd = dm.to(dev)
            known = torch.zeros(0, dtype=torch.long, device=dev)
            es = be.proximity_edges(dd, t0, t1, t, known, known, 2, nms, th, mf, False)
            ms = _time_ms(lambda: be.proximity_edges(dd, t0, t1, t, known, known, 2, nms, th, mf, False), iters=20)
            entry = {"kernel": "proximity_edges (row F1, %s)" % tag, "bound": "latency (serial greedy selection)", "ms": ms, "edges_selected": int(es.shape[0]),
                     "note": "ms includes the one host read of the edge count; cpu_restatement_ms = oracle/proximity.py (the reference's Python loop restated), one core"}
            if _prox is not None:
                c0 = _time.perf_counter()
                want, _ = _prox.proximity_edges(dm.numpy(), t0, t1, t, [], [], rad=2, nms=nms, thresh=th, max_factors=mf)
                entry["cpu_restatement_ms"] = 1e3 * (_time.perf_counter() - c0)
                entry["identical_to_cpu_restatement"] = bool(es.shape[0] == want.shape[0] and (es.cpu().numpy() == want).all())
            out["rooflines"].append(entry)
    except Exception as e:
        out["rooflines"].append({"kernel": "proximity_edges", "error": str(e)[:200]})
    return out


# ---------------------------------------------------------------------------------------------------------
def cpu_baseline(pb, corr_edges=64, ba_edges=128):
    """the CPU oracle (a port of the reference kernels, oracle/) on a BOUNDED sample of the same step, host cores"""
    import oracle
    cores = min(os.cpu_count() or 1, 32)          # torch CPU ops stop scaling (and start thrashing) far below 128 threads
    torch.set_num_threads(cores)
    h = pb["host"]
    n = min(corr_edges, pb["E"])
    vols = [v[:n].cpu() for v in pb["pyr"]]
    coords = h["coords"][:n]
    t0 = time.time()
    for l, v in enumerate(vols):
        oracle.corr_index_forward(v, coords / 2 ** l, RADIUS)
    t_corr = (time.time() - t0) * pb["E"] / n
    nb = min(ba_edges, pb["E"])
    P, D = h["poses"].clone(), h["disps"].clone()
    ii, jj = h["ii"][:nb], h["jj"][:nb]
    kx = torch.unique(torch.cat([torch.arange(pb["t0"], pb["t1"]), ii]))
    t0 = time.time()
    oracle.ba(P, D, h["intrinsics"], h["disps_sens"], h["targets"][:nb], h["weights"][:nb], h["eta_by_frame"][kx], ii, jj, pb["t0"], pb["t1"],
              BA_ITERS, LM, EP, False)
    t_ba = (time.time() - t0) * pb["E"] / nb
    return {"value": 1.0 / (t_corr + t_ba), "unit": "iters/s", "cores": cores, "kind": "port",
            "sample": "oracle corr_index_forward on %d of %d edges (4 levels) + oracle ba(itrs=2) on a %d-edge subgraph of the same %d-keyframe window; "
                      "both times scaled linearly by edge count; torch CPU threads=%d" % (n, pb["E"], nb, FRAMES, cores), "corr_s": t_corr, "ba_s": t_ba}


# ---------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world, dev):
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
    try:
        import droid_backends_ref as ref
    except Exception as e:                                   # reference build absent: the CPU oracle port is the reference arm
        return run_reference_cpu(args, dev, "oracle/_ref not importable: %s" % str(e)[:80])
    lib = ctypes.CDLL(ref.__file__)
    lib.droid_ref_solve_seconds.restype = ctypes.c_double
    pb = build_problem(args, 0, 1, dev)
    h = pb["host"]
    E = pb["E"]
    d = {k: v.to(dev) for k, v in h.items()}
    CH = 128

    def corr_all(coords):
        outs = []
        for l in range(LEVELS if WITH_CORR else 0):
            c = coords / 2 ** l
            parts = [ref.corr_index_forward(pb["pyr"][l][s:s + CH], c[s:s + CH].contiguous(), RADIUS)[0] for s in range(0, E, CH)]
            outs.append(parts)
        return outs

    def step_resident():
        P, D = d["poses"].clone(), d["disps"].clone()
        corr_all(pb["coords"])
        ref.ba(P, D, d["intrinsics"], d["disps_sens"], d["targets"], d["weights"], d["eta"], d["ii"], d["jj"], pb["t0"], pb["t1"], BA_ITERS, LM, EP, False)

    pin = {k: h[k].pin_memory() for k in ("coords", "targets", "weights", "eta", "poses", "disps", "disps_sens", "ii", "jj", "intrinsics")}
    Pn = pb["t1"] - pb["t0"]
    out_pin = dict(poses=torch.empty(FRAMES, 7).pin_memory(), disps=torch.empty(FRAMES, HT, WD).pin_memory(), dx=torch.empty(Pn, 6).pin_memory())
    h2d = sum(v.numel() * v.element_size() for v in pin.values()); d2h = sum(v.numel() * v.element_size() for v in out_pin.values())

    def step_e2e():
        g = {k: pin[k].to(dev, non_blocking=True) for k in pin}
        corr_all(g["coords"])
        dx, dz = ref.ba(g["poses"], g["disps"], g["intrinsics"], g["disps_sens"], g["targets"], g["weights"], g["eta"], g["ii"], g["jj"],
                        pb["t0"], pb["t1"], BA_ITERS, LM, EP, False)
        out_pin["poses"].copy_(g["poses"], non_blocking=True); out_pin["disps"].copy_(g["disps"], non_blocking=True); out_pin["dx"].copy_(dx, non_blocking=True)

    def timed(fn, steps, warm):
        for _ in range(warm): fn()
        torch.cuda.synchronize()
        s0 = lib.droid_ref_solve_seconds()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time(); e0.record()
        for _ in range(steps): fn()
        e1.record(); torch.cuda.synchronize()
        return max(e0.elapsed_time(e1), (time.time() - w0) * 1e3) / steps, (lib.droid_ref_solve_seconds() - s0) * 1e3 / steps

    sampler = ClockSampler(torch.cuda.current_device()); sampler.start()
    ms_step, solve_ms = timed(step_resident, args.steps, max(args.warmup, 3))
    clocks = sampler.stop()
    e2e_ms, _ = timed(step_e2e, args.steps, 2)
    if CFG_NAME == "metric":
        metric, unit = "BA-update iters/sec (512 edges, 344x64x48)", "iters/s (512-edge equivalents)"
    else:
        metric, unit = "BA-update iters/sec (BASELINE config %s)" % CFG_NAME, "iters/s (one step = %sba(itrs=%d))" % ("4-level corr_index_forward + " if WITH_CORR else "", BA_ITERS)
    upd = reference_update_operator_ms(E, dev) if (CFG_NAME == "metric" and not args.no_extras) else None
    line = {
        "metric": metric, "value": 1e3 / ms_step, "unit": unit, "n_gpus": 1,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": SCALING, "vs_baseline": None,
        "dtype": "f32 (CPU solve in f64), %s corr volumes" % args.dtype, "data": "synthetic", "impl": "reference", "update_operator": upd,
        "config": {"workload": "%s: %d edges over a %d-keyframe window at %dx%d, %s + ba(itrs=%d, lm=%g, ep=%g)" % (CFG_NAME, E, FRAMES, HT, WD, ("4-level r=3 corr_index_forward (chunks of %d edges: 32-bit accessors)" % CH) if WITH_CORR else "no lookup", BA_ITERS, LM, EP), "name": CFG_NAME,
                   "implementation": "unmodified /root/reference/src/*.cu + droid.cpp built for sm_100a (oracle/build_ref.sh); CPU solve = dense fp64 LLT stand-in for Eigen::SimplicialLLT",
                   "cpu_solve_ms_per_step": solve_ms, "ms_per_step_without_cpu_solve": ms_step - solve_ms},
        "e2e": {"value": 1e3 / e2e_ms, "unit": unit, "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "cpu_baseline": {"value": 1e3 / ms_step, "unit": "iters/s", "cores": os.cpu_count(), "kind": "reference",
                         "sample": "full workload, %d steps; the reference path is CUDA kernels + a host-side sparse-block solve (its CPU part uses 1 thread)" % args.steps},
        "clocks": clocks,
    }
    print(json.dumps(line))


def reference_update_operator_ms(E, dev, iters=3):
    """the reference's update operator formula (droid_net.py:111-143 as restated in oracle/update.py, pinned bit-exactly against the
    reference module) through torch/cuDNN under fp16 autocast like factor_graph.py:214 -- what `update_operator` of our arm replaces"""
    try:
        import oracle
        from droid_slam_b200 import synth
        w = {k: v.to(dev) for k, v in synth.make_update_weights(0).items()}
        g = torch.Generator(device=dev).manual_seed(7)
        net = torch.tanh(torch.randn(1, E, 128, HT, WD, generator=g, device=dev)).half()
        inp = torch.relu(torch.randn(1, E, 128, HT, WD, generator=g, device=dev)).half()
        corr = torch.randn(1, E, 196, HT, WD, generator=g, device=dev).half()
        motn = torch.randn(1, E, 4, HT, WD, generator=g, device=dev)
        ii = torch.arange(E, device=dev) % FRAMES
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            ms = _time_ms(lambda: oracle.update_module_forward(w, net, inp, corr, motn, ii), iters=iters)
        return {"ms": ms, "edges": E, "impl": "reference formula (oracle/update.py) through torch/cuDNN convolutions under fp16 autocast"}
    except Exception as e:
        return {"ms": None, "error": str(e)[:200]}


def run_reference_cpu(args, dev, why):
    import oracle  # noqa: F401
    pb = build_problem(args, 0, 1, dev)
    cb = cpu_baseline(pb)
    ms = 1e3 / cb["value"]
    print(json.dumps({"metric": "BA-update iters/sec (512 edges, 344x64x48)", "value": cb["value"], "unit": "iters/s (512-edge equivalents)", "n_gpus": 1,
                      "steps": 1, "warmup": 0, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                      "data": "synthetic", "impl": "reference", "config": {"workload": "metric (CPU oracle port; %s)" % why},
                      "cpu_baseline": dict(cb, kind="port"), "e2e": {"value": cb["value"], "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if args.impl == "reference":
        # the reference has no multi-GPU path: rank 0 alone measures it, the other ranks of a torchrun launch exit without work
        # (no process group is created, so nothing can wait on anything)
        if rank == 0:
            run_reference(args, 0, 1, dev)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")       # unset: NCCL prints its version banner on stdout next to the one JSON line; a caller's own setting (e.g. INFO) is kept
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        if args.impl == "reference":
            run_reference(args, rank, world, dev)
        else:
            run_ours(args, rank, world, dev)
    finally:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
