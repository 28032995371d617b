#!/usr/bin/env python
"""bench.py -- throughput of the 3D-GCN hot path (BASELINE.json metric: 3D-GCN fwd point clouds/sec @1028 pts).

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA path)
  python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/<name>.npy
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the UNMODIFIED reference modules (oracle/_ref/pyref,
                                                           # staged from /root/reference by build()) on host cores;
                                                           # the oracle port only when that staging is absent

One "step" = one full TG-Pose network forward (Face_Enc backbone on the sm_100a kernels + pose heads)
over one batch of 32 synthetic NOCS-shaped clouds x 1028 points per GPU (BASELINE.json configs[1]).
N > 1: one process per GPU (torchrun), the batch dimension is sharded, no data-path collective
(inference), weak scaling.  Rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "3D-GCN fwd point clouds/sec @1028 pts"
UNIT = "clouds/s"
N_PTS = 1028
PER_GPU_BATCH = 32
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # CUDA-core FMA peak at sm_max_mhz (SURVEY 8d): 74.4
DTYPE = "f32 (encoder + kNN contractions 3xTF32 on tcgen05, heads fp16 + 2 bf16 cross terms, everything else fp32 FMA)"
WORKLOAD = "full TG-Pose network forward (Face_Enc 3D-GCN + heads), 32 x 1028 points per GPU"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def synth_inputs(batch, seed):
    """SURVEY 8d: object-sized clouds at camera range, 6 categories."""
    import torch
    g = torch.Generator().manual_seed(seed)
    pts = torch.rand(batch, N_PTS, 3, generator=g)
    t = torch.stack([torch.rand(batch, generator=g) * 0.6 - 0.3, torch.rand(batch, generator=g) * 0.6 - 0.3,
                     torch.rand(batch, generator=g) * 0.8 + 0.6], dim=1)
    pts = (pts - 0.5) * 0.3 + t[:, None, :]
    cat = torch.randint(0, 6, (batch, 1), generator=g).float()
    return pts, cat


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def _nvml_loop(self, handle, nv):
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        mx = nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM)
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)
                rs = int(get_reasons(handle))
                self.nvml_rows.append((float(sm), float(mx), [n for n, b in bits.items() if rs & b]))
            except Exception:
                break
            time.sleep(0.004)

    def start(self):
        # in-process NVML polling every ~4 ms (a step lasts ~3 ms, a default run well under a second: nvidia-smi's
        # 100 ms loop would deliver one or two samples); nvidia-smi -lms stays as the fallback
        self._stop = threading.Event()
        self.nvml_rows = []
        try:
            import pynvml as nv
            import torch
            nv.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(self.gpu).uuid)
                handle = nv.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
            except Exception:
                handle = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)
            threading.Thread(target=self._nvml_loop, args=(handle, nv), daemon=True).start()
            self.proc = None
            self.nvml = True
            return
        except Exception:
            self.nvml = False
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if getattr(self, "nvml", False):
            self._stop.set()
            time.sleep(0.01)
            rows = list(self.nvml_rows)
            if not rows:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
            sm = sorted(r[0] for r in rows)
            reasons = sorted({n for r in rows for n in r[2]})
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[1] for r in rows), "reasons": reasons,
                    "samples": len(sm), "source": "NVML, 4 ms period, during the timed and end-to-end loops"}
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_port_run(batch, steps, warmup, seed=1234):
    """FALLBACK when oracle/_ref/pyref is absent: the oracle port (C/OpenMP kernels + numpy/BLAS heads) of the same
    full-network forward on host cores."""
    import torch
    from oracle import oracle as orc
    from tgpose_b200.posenet import PoseNet9D
    torch.manual_seed(0)
    net = PoseNet9D().eval()
    sd = {k: v.detach().numpy() for k, v in net.state_dict().items()}
    pts, cat = synth_inputs(batch, seed)
    pts, cat = pts.numpy(), cat.numpy()
    cores = os.cpu_count() or 1
    orc.set_num_threads(cores)
    orc.USE_BLAS = True      # dense contractions through BLAS sgemm, like the reference's torch CPU path
    times = []
    for i in range(warmup + steps):
        torch.manual_seed(7)
        perm1, perm2 = torch.randperm(N_PTS).numpy(), torch.randperm(N_PTS // 4).numpy()
        t0 = time.perf_counter()
        orc.posenet_forward(sd, pts, cat, perm1, perm2)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    per = sum(times) / len(times)
    return {"value": batch / per, "seconds_per_step": per, "cores": cores, "batch": batch, "kind": "port",
            "what": "C/OpenMP oracle kernels + BLAS sgemm contractions (oracle/_ref/pyref not staged)"}


def cpu_reference_run(batch, steps, warmup, seed=1234, budget_s=None):
    """The reference's OWN modules (network/fs_net_repo/PoseNet9D.py + gcn3d.py ..., staged byte for byte into
    oracle/_ref/pyref by oracle/build_ref.py) on the host cores: torch CPU, eval, no_grad, all threads.
    budget_s: shrink the batch (a bounded sample of the 32-cloud step) so that warmup + steps passes fit the budget."""
    import torch
    from oracle import build_ref
    mods = build_ref.import_pyref()
    if mods is None:
        return None
    _gcn3d, _face, pose = mods
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    net = pose.PoseNet9D().eval()

    def one(pts, cat):
        torch.manual_seed(7)
        t0 = time.perf_counter()
        with torch.no_grad():
            out = net(pts, cat)
        dt = time.perf_counter() - t0
        assert bool(torch.isfinite(out["Pred_T"]).all())
        return dt

    # the first pass at a candidate batch is the first warm-up pass; if the remaining passes would not fit the budget
    # the batch is halved (the reference's per-cloud cost GROWS with the batch: it materialises (B,N,k,S*C) tensors)
    done_warm = 0
    while True:
        pts, cat = synth_inputs(batch, seed)
        t1 = one(pts, cat)
        done_warm = 1
        if budget_s is None or batch <= 2 or t1 * (steps + max(warmup - 1, 0)) <= budget_s:
            break
        batch //= 2
    times = [one(pts, cat) for _ in range(max(warmup - done_warm, 0) + steps)][max(warmup - done_warm, 0):]
    per = sum(times) / len(times)
    return {"value": batch / per, "seconds_per_step": per, "cores": cores, "batch": batch, "kind": "reference",
            "what": "unmodified reference PoseNet9D (oracle/_ref/pyref: network/fs_net_repo/*.py), torch CPU eval/no_grad, "
                    f"torch.set_num_threads({cores})"}


def cpu_arm(batch, steps, warmup, budget_s):
    r = None
    try:
        r = cpu_reference_run(batch, steps, warmup, budget_s=budget_s)
    except Exception as e:          # a broken staging must not take the bench line down: say so and use the port
        sys.stderr.write(f"bench.py: reference CPU arm failed ({type(e).__name__}: {e}); using the oracle port\n")
    if r is None:
        r = cpu_port_run(min(batch, 2), steps, warmup)
    return r


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # BASELINE.json configs[1] on the host: the same 32-cloud step when warmup + steps passes fit ~4 minutes, else the
    # largest power-of-two sample of it that does (configs[0] is the 2-cloud case)
    r = cpu_arm(PER_GPU_BATCH, args.steps, args.warmup, budget_s=240.0)
    sample = (f"{r['batch']} of the 32 clouds per step (same generator and seeds as the CUDA arm)" if r["batch"] < PER_GPU_BATCH
              else "the full 32-cloud step")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["seconds_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "points": N_PTS, "per_gpu_batch": PER_GPU_BATCH, "cpu_batch": r["batch"]},
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                         "sample": f"{sample}; {r['what']}"},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from tgpose_b200 import _lib, ops
    from tgpose_b200.posenet import PoseNet9D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False

    B = args.batch
    torch.manual_seed(0)
    net = PoseNet9D().to(dev).eval()
    # several distinct input batches so no iteration re-reads the previous one's data
    n_sets = 4
    host_sets = []
    for s in range(n_sets):
        pts, cat = synth_inputs(B, 1234 + 17 * rank + s)
        host_sets.append((pts.pin_memory(), cat.pin_memory()))
    dev_sets = [(p.to(dev), c.to(dev)) for p, c in host_sets]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2

    def eager_step(pts, cat):
        torch.manual_seed(7)          # Pool_layer draws its permutation from the CPU generator (gcn3d.py:242)
        with torch.no_grad():
            return net(pts, cat)

    graphed = None
    if not args.no_graph:
        from tgpose_b200.graph import GraphedPoseNet
        graphed = GraphedPoseNet(net, B, N_PTS)

    def step(pts, cat):
        if graphed is None:
            return eager_step(pts, cat)
        torch.manual_seed(7)
        return graphed(pts, cat)      # copies the inputs into the graph's static buffers, draws the perms, replays

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(*dev_sets[i % n_sets])
    barrier()

    # ---- device-resident timing: K steps, CUDA events per step, L2 flushed between steps
    # ---- per-kernel table: an EAGER pass of the same steps with CUDA events around every C-ABI call (a graph replay
    # cannot be instrumented per call); the launches counted here are the ones each graph replay re-issues
    event_log = None
    kt_steps = min(args.steps, 5)
    l0 = _lib.launch_count()
    if rank == 0:
        ops.EVENT_LOG = {}
    # (the forked streams of the forward -- pose tails beside the decoder chain, coordinate-only work beside conv_0 / conv_1 --
    # are folded into the main stream for this pass: two kernels sharing the GPU would each be charged the other's time)
    enc_ = net.face_all.encoder
    forks = (net.overlap_heads, enc_.xyz_ahead)
    net.overlap_heads, enc_.xyz_ahead = False, False
    # An eager launch costs the host more (python, ctypes, tensor-map encodes: 20-40 us) than most of these kernels run, so
    # with an idle GPU the interval between a call's two events is host time, not kernel time.  Each pass therefore starts
    # behind a ~6 ms device-side spin: the host queues the whole forward while the GPU waits, the launches then run back to
    # back, and an event pair brackets the kernel alone.
    spin = getattr(torch.cuda, "_sleep", None)
    for i in range(kt_steps):
        flush.zero_()
        if spin is not None:
            spin(int(6e-3 * 1.9e9))
        eager_step(*dev_sets[i % n_sets])
    barrier()
    net.overlap_heads, enc_.xyz_ahead = forks
    event_log, ops.EVENT_LOG = ops.EVENT_LOG, None
    l0 = _lib.launch_count()
    eager_step(*dev_sets[0])             # the launches of one forward as the graph replays them (forks on)
    barrier()
    launches_per_step = _lib.launch_count() - l0

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.zero_()
        ev[i][0].record()
        out = step(*dev_sets[i % n_sets])
        ev[i][1].record()
    barrier()
    wall = time.perf_counter() - wall0
    launches = launches_per_step * args.steps
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    if args.dump_outputs and rank == 0:
        # the graph's static outputs are overwritten by the later loops: copy the last timed step's now
        dump_outputs(args.dump_outputs, out)

    # ---- encoder only (SURVEY 8d: "report encoder-only clouds/s -- the optimisation target -- and full-network clouds/s
    # separately"): Face_Enc.forward alone, same clouds (centred like PoseNet9D.py:48), same replay/flush/event protocol
    enc_ms = None
    if graphed is not None:
        from tgpose_b200.graph import GraphedPoseNet as _G
        genc = _G(net, B, N_PTS, encoder_only=True)
        cen_sets = [(p_ - p_.mean(dim=1, keepdim=True), c_) for p_, c_ in dev_sets]
        for i in range(3):
            torch.manual_seed(7)
            genc(*cen_sets[i % n_sets])
        evs_e = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()
        for i in range(args.steps):
            flush.zero_()
            evs_e[i][0].record()
            torch.manual_seed(7)
            genc(*cen_sets[i % n_sets])
            evs_e[i][1].record()
        barrier()
        enc_ms = sum(a.elapsed_time(b) for a, b in evs_e) / args.steps
        del genc

    # ---- end to end: pinned host inputs -> H2D -> forward -> D2H of the pose outputs, every step
    barrier()
    out_keys = ("p_green_R", "p_red_R", "f_green_R", "f_red_R", "Pred_T", "Pred_s")
    h2d = d2h = 0
    # every step's pose outputs are read back into pinned host memory (one buffer per step); each step is bracketed by its
    # own CUDA-event pair on the launching stream: H2D of the clouds, the forward, D2H of the poses; the 256 MB L2 flush sits
    # between the pairs like in the device-resident loop; the host waits once, after the last step
    res_host = [torch.empty((B, 14), dtype=torch.float32).pin_memory() for _ in range(args.steps)]   # 3+3+1+1+3+3 pose values
    barrier()
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for i in range(args.steps):
        hp, hc = host_sets[i % n_sets]
        flush.zero_()                 # same L2 protocol as the device-resident loop; outside the step's event pair
        ev2[i][0].record()
        if graphed is None:
            out = step(hp.to(dev, non_blocking=True), hc.to(dev, non_blocking=True))
        else:
            out = step(hp, hc)        # pinned host -> the graph's static input buffers (H2D inside the timed region)
        res = torch.cat([out[k].reshape(B, -1) for k in out_keys], dim=1)
        res_host[i].copy_(res, non_blocking=True)
        ev2[i][1].record()
        if i == 0:
            h2d = hp.numel() * 4 + hc.numel() * 4
            d2h = res.numel() * 4
    ev2[-1][1].synchronize()
    assert all(bool(torch.isfinite(r).all()) for r in res_host)
    barrier()
    e2e_ms = sum(a.elapsed_time(b) for a, b in ev2)
    clocks = sampler.stop() if rank == 0 else None

    t = torch.tensor([dev_ms, e2e_ms, enc_ms or 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, enc_ms = float(t[0]), float(t[1]), (float(t[2]) if enc_ms else None)

    # ---- configs[2] beside the headline, in the same run: the RL_TDA training step at a global batch of 256 (256 / N per
    # GPU, strong scaling) with the NCCL gradient all-reduce -- so the scaling curve shows the path's one collective
    train_rec = None
    graph_used = graphed is not None
    if not args.no_train:
        graphed = None
        torch.cuda.empty_cache()
        try:
            train_rec = train_record(args, dev, rank, world, steps=args.train_steps, warmup=2)
        except Exception as e:      # the headline line must survive a failure of the secondary record; say what happened
            train_rec = {"error": f"{type(e).__name__}: {e}"[:300]}
    chamfer_rec = chamfer_record(dev, flush) if rank == 0 else None

    if rank == 0:
        peaks = measured_peaks()
        ms_per_step = dev_ms / args.steps
        total = B * world
        line = {
            "metric": METRIC, "value": total / (ms_per_step / 1e3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "points": N_PTS, "per_gpu_batch": B, "global_batch": total, "parallelism": f"dp{world}",
                       "weights": "random-init (seed 0)", "l2": "256 MB flush write between timed steps",
                       "launch": "CUDA graph replay of the whole forward" if graph_used else "eager launches"},
            "e2e": {"value": total / (e2e_ms / args.steps / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "wall_s": wall,
        }
        if enc_ms:
            line["encoder_only"] = {"value": total / (enc_ms / 1e3), "unit": UNIT, "ms_per_step": enc_ms,
                                    "what": "Face_Enc.forward alone (FaceRecon.py:39-86: 5 graph convs, 2 pools, upsampling, concat), "
                                            "CUDA graph replay, same clouds / flush / events as `value`"}
        line.update(kernel_report(event_log, kt_steps, B, peaks))
        if chamfer_rec:
            line.setdefault("kernel_rooflines", {})["chamfer_fwd"] = chamfer_rec
        if train_rec is not None:
            line["train"] = train_rec
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_arm(8, 2, 1, budget_s=30.0)
            line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                                    "sample": f"{r['batch']} of the 32 clouds per step, 2 timed passes after 1 warm-up; {r['what']}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(directory, out):
    """Write the outputs of one forward (the dict a caller of PoseNet9D receives) as DIR/<name>.npy, float32.
    The inputs and weights are seeded, so two builds run with the same arguments can be compared file for file.
    All files together stay within DUMP_CAP_BYTES: an array larger than its share keeps a fixed, seeded sample of its
    rows (the same rows in every run)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    share = DUMP_CAP_BYTES // max(len(out), 1)
    for name, t in out.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            a = a.reshape(a.shape[0], -1) if a.ndim > 1 and a[0].nbytes <= share else a.reshape(-1, 1)
            keep = share // a[0].nbytes
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(directory, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------ secondary records
def chamfer_record(dev, flush):
    """chamfer3D forward at BASELINE configs[2] size (256 x 1028 vs 1024 points) against the FP32 roof, and -- when
    oracle/_ref/chamfer3D was built -- the reference's own kernel on the same inputs (the kernel to beat, SURVEY 2b)."""
    import torch
    from tgpose_b200 import ops
    B, n, m = 256, N_PTS, 1024
    g = torch.Generator().manual_seed(77)
    a, b = torch.rand(B, n, 3, generator=g).to(dev), torch.rand(B, m, 3, generator=g).to(dev)
    o = (torch.zeros(B, n, device=dev), torch.zeros(B, m, device=dev),
         torch.zeros(B, n, dtype=torch.int32, device=dev), torch.zeros(B, m, dtype=torch.int32, device=dev))

    def timed(fn, iters=10):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2]

    ms = timed(lambda: ops.chamfer_forward(a, b, *o))
    flops = 2.0 * B * n * m * 9          # SURVEY 8d: 2*n*m*8 + 2*n*m per cloud pair
    rec = {"bound": "fp32", "shape": f"{B} x {n} x {m}", "ms": round(ms, 4), "achieved_tflops": round(flops / ms / 1e9, 3),
           "frac_fp32": round(flops / ms / 1e9 / FP32_PEAK_TFLOPS, 4)}
    try:
        from oracle import build_ref
        ref = build_ref.load_chamfer()
        if ref is not None:
            r = tuple(torch.zeros_like(t) for t in o)
            rms = timed(lambda: ref.forward(a, b, *r))
            rec["reference_kernel_ms"] = round(rms, 4)
            rec["reference_kernel"] = "losses/chamfer3D/chamfer3D.cu compiled for sm_100a (oracle/_ref), same inputs, same box"
            rec["bit_equal_to_reference"] = bool(all(torch.equal(x, y) for x, y in zip(o, r)))
    except Exception as e:
        rec["reference_kernel_error"] = f"{type(e).__name__}: {e}"[:200]
    return rec


def train_record(args, dev, rank, world, steps, warmup):
    """RL_TDA training step (BASELINE configs[2]) at global batch 256: ms/step (max over ranks), the all-reduce's share."""
    import torch
    import torch.distributed as dist
    from tgpose_b200.posenet import PoseNet9D
    from tgpose_b200.train_step import TrainStep, augment, synthetic_targets
    gb = args.train_batch
    Bt = gb // world
    torch.manual_seed(0)
    net = PoseNet9D(train_outputs=True).to(dev)
    net2 = PoseNet9D(only_encoder=True).to(dev)         # frozen encoder on the augmented cloud (RL_TDA.py:20,117-118)
    step = TrainStep(net, optimizer="ranger", net2=net2)
    sets = []
    for s_ in range(2):
        pts, cat = synth_inputs(Bt, 4321 + 17 * rank + s_)
        sets.append((pts.pin_memory(), cat.pin_memory(), synthetic_targets(Bt, 99 + rank + s_, dev),
                     augment(pts, 55 + rank + s_).pin_memory()))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(warmup):
        hp, hc, tgt, ha = sets[i % 2]
        step(hp.to(dev, non_blocking=True), hc.to(dev, non_blocking=True), tgt, ha.to(dev, non_blocking=True))
    barrier()
    step.ar_events = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss_host = None
    for i in range(steps):
        hp, hc, tgt, ha = sets[i % 2]
        loss = step(hp.to(dev, non_blocking=True), hc.to(dev, non_blocking=True), tgt,
                    ha.to(dev, non_blocking=True))                                        # H2D inside the timed region
        loss_host = float(loss)                                                           # D2H of the step's loss
    e1.record()
    barrier()
    early = getattr(step.overlap, "launched_early", None) if step.overlap is not None else None
    ar_ms = sum(a.elapsed_time(b) for a, b in step.ar_events) / max(steps, 1)
    t = torch.tensor([e0.elapsed_time(e1) / steps, ar_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    nbytes = int(step.opt.flat_grads.numel()) * 4
    del step, net
    torch.cuda.empty_cache()
    return {"metric": "RL_TDA train step clouds/sec @1028 pts", "value": gb / (ms / 1e3), "unit": UNIT, "ms_per_step": ms,
            "global_batch": gb, "per_gpu_batch": Bt, "scaling": "strong", "steps": steps, "warmup": warmup,
            "optimizer": "Ranger (fused kernels) + flat_and_anneal schedule", "loss": loss_host,
            "step": "net1 fwd+bwd, net2 fwd (no grad) on the augmented cloud, feature-consistency + symmetry-aware recon losses, "
                    "chamfer3D / DCD recon loss, pose terms, clip 5, Ranger, scheduler (trainer/RL_TDA.py:110-226)",
            "allreduce": {"collective": "NCCL all-reduce (sum, / world) of the flat fp32 gradient arena in ~32 MB slices, each "
                                        "launched from an autograd hook when its last gradient has landed (overlaps backward)"
                                        if world > 1 else "none (world 1)",
                          "bytes_per_step": nbytes if world > 1 else 0, "slices": step_buckets(world, nbytes),
                          "slices_launched_during_backward": early,
                          "exposed_ms_per_step": float(t[1]),
                          "timing": "CUDA events from the end of backward to the last slice's completion (the part of the "
                                    "collective NOT hidden behind backward), max over ranks"},
            "e2e": "pinned-host H2D of the step's clouds and the D2H read of its loss are inside the timed region"}


def step_buckets(world, nbytes, bucket=32 << 20):
    return 0 if world == 1 else (nbytes + bucket - 1) // bucket


# ------------------------------------------------------------------------------------------------ training step
def run_train(args):
    """BASELINE.json configs[2]: RL_TDA training step (fwd + bwd + chamfer/DCD loss + gradient all-reduce + optimizer)
    at a GLOBAL batch of 256 x 1028 points, sharded over the ranks (strong scaling).  Secondary bench line."""
    import torch
    import torch.distributed as dist
    from tgpose_b200 import _lib, ops
    from tgpose_b200.posenet import PoseNet9D
    from tgpose_b200.train_step import TrainStep, augment, synthetic_targets

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    gb = args.train_batch
    B = gb // world
    torch.manual_seed(0)
    net = PoseNet9D(train_outputs=True).to(dev)
    net2 = PoseNet9D(only_encoder=True).to(dev)
    step = TrainStep(net, optimizer=args.optimizer, net2=net2)
    sets = []
    for s_ in range(2):
        pts, cat = synth_inputs(B, 4321 + 17 * rank + s_)
        sets.append((pts.pin_memory(), cat.pin_memory(), synthetic_targets(B, 99 + rank + s_, dev),
                     augment(pts, 55 + rank + s_).pin_memory()))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        hp, hc, tgt, ha = sets[i % 2]
        step(hp.to(dev, non_blocking=True), hc.to(dev, non_blocking=True), tgt, ha.to(dev, non_blocking=True))
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.EVENT_LOG = {} if rank == 0 else None
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    loss = None
    for i in range(args.steps):
        hp, hc, tgt, ha = sets[i % 2]
        loss = step(hp.to(dev, non_blocking=True), hc.to(dev, non_blocking=True), tgt,
                    ha.to(dev, non_blocking=True))                                        # H2D inside the timed region
        loss_host = float(loss)                                                           # D2H of the step's loss
    e1.record()
    barrier()
    launches = _lib.launch_count() - l0
    event_log, ops.EVENT_LOG = ops.EVENT_LOG, None
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0]) / args.steps
    if rank == 0:
        kern = {}
        tot = 0.0
        for name, evs in (event_log or {}).items():
            if name.startswith("__"):
                continue
            v = sum(a.elapsed_time(b) for a, b in evs) / args.steps
            kern[name] = round(v, 4)
            tot += v
        val = gb / (ms / 1e3)
        line = {"metric": "RL_TDA train step clouds/sec @1028 pts", "value": val, "unit": UNIT, "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "RL_TDA training step: PoseNet9D fwd+bwd, chamfer3D/DCD recon loss, gradient "
                                       f"all-reduce, clip, {args.optimizer} step; global batch 256 x 1028 points",
                           "points": N_PTS, "global_batch": gb, "per_gpu_batch": B, "parallelism": f"dp{world}",
                           "l2": "per-step working set (> 1 GB of activations) exceeds the 126 MB L2"},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": B * (2 * N_PTS * 3 + 1) * 4, "d2h_bytes_per_step": 4},
                "gpu_launches": int(launches), "allreduce_buckets": step.buckets, "loss": loss_host, "clocks": clocks,
                "tgpose_kernel_ms_per_step": round(tot, 3), "kernels_ms_per_step": dict(sorted(kern.items()))}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ microbench sweep
def run_micro(args):
    """BASELINE.json configs[3]: kNN + Conv_surface / Conv_layer sweep, N = 1028..16384, k = 10..50, S = 7, C = 128,
    D in {3, 128}; CUDA events, L2 flushed between iterations; per-kernel roofline fractions (SURVEY 8d work counts)."""
    import torch
    from tgpose_b200 import _lib, ops
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    _lib.load()
    dev = torch.device("cuda", 0)
    peaks = measured_peaks()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    S, C, D = 7, 128, 128
    rows = []

    def timed(fn, iters):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2] / 1e3

    g = torch.Generator().manual_seed(1234)
    for N in (1028, 2048, 4096, 8192, 16384):
        B = max(1, (32 * 1028) // N)
        xyz = torch.rand(B, N, 3, generator=g).to(dev)
        feat = (torch.randn(B, N, D, generator=g) * 0.3).to(dev)
        dirs = ((torch.rand(3, S * C, generator=g) - 0.5) * 0.07).to(dev)
        M = B * N
        slab = torch.randn(C // 4, M, S * 4, generator=g).to(dev)
        centre = torch.randn(M, C, generator=g).to(dev)
        for k in (10, 20, 30, 40, 50):
            it = 5 if N >= 8192 else 10
            t_xyz = timed(lambda: ops.knn_xyz(xyz, k, want64=False, want32=True), it)
            t_feat = timed(lambda: ops.knn_feat(feat, k, want64=False, want32=True), it)
            idx = ops.knn_xyz(xyz, k, want64=False, want32=True)[1]
            t_surf = timed(lambda: ops.surface_conv(xyz, idx, dirs, S, C), it)
            rec = ops.edge_records(xyz, idx)
            t_lay = timed(lambda: ops.layer_conv(rec, dirs, centre, slab, B, N, S, C), it)
            f_xyz = B * (N * N * (2 * 3 + 3) + N * N)
            f_feat = B * (N * N * (2 * D + 3) + N * N)
            f_surf = B * (N * k * S * C * 8 + N * S * C)
            f_lay = B * (N * k * S * C * 9 + N * S * C)
            b_lay = B * (4 * (3 * N + S * C * N + C * N + C * N + 3 * S * C) + 4 * N * k)
            rows.append({"N": N, "B": B, "k": k,
                         "knn_xyz": {"ms": t_xyz * 1e3, "gpairs_s": B * N * N / t_xyz / 1e9, "fp32_frac": f_xyz / t_xyz / 1e12 / FP32_PEAK_TFLOPS},
                         "knn_feat_D128": {"ms": t_feat * 1e3, "gpairs_s": B * N * N / t_feat / 1e9, "tflops": f_feat / t_feat / 1e12,
                                           "fp32_frac": f_feat / t_feat / 1e12 / FP32_PEAK_TFLOPS,
                                           "path": "tcgen05 3xTF32 + threshold select (64 group minima)" if k <= 31 else "tcgen05 3xTF32 + threshold select (128 group minima)"},
                         "surface_conv": {"ms": t_surf * 1e3, "tflops": f_surf / t_surf / 1e12, "fp32_frac": f_surf / t_surf / 1e12 / FP32_PEAK_TFLOPS},
                         "layer_conv": {"ms": t_lay * 1e3, "tflops": f_lay / t_lay / 1e12, "fp32_frac": f_lay / t_lay / 1e12 / FP32_PEAK_TFLOPS,
                                        "hbm_gbs": b_lay / t_lay / 1e9, "hbm_frac": b_lay / t_lay / 1e9 / peaks["hbm_gbs"],
                                        "table": "smem" if N * S * 16 + 4 * 2 * k * 64 <= 227 * 1024 else "L2 gather"}})
    print(json.dumps({"metric": "kNN + Conv_surface/Conv_layer microbench sweep", "S": S, "C": C, "D": D,
                      "fp32_peak_tflops": FP32_PEAK_TFLOPS, "hbm_peak_gbs": peaks["hbm_gbs"], "peak_source": peaks["source"],
                      "timing": "median of CUDA-event times, 256 MB L2 flush before each iteration", "rows": rows}), flush=True)


def profile_traffic(kernel_substr):
    """DRAM bytes per forward of the kernels whose name contains `kernel_substr`, from the newest committed
    profiles/*_kernels.json that captured such a kernel (written by scripts/make_profile_summary.py from an ncu capture of one
    inference forward; the training-step captures do not contain the forward kernels); None if absent."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_kernels.json")), reverse=True):
        try:
            per = json.load(open(path))["per_kernel"]
            tot = sum(v["dram_bytes"] for k, v in per.items() if kernel_substr in k)
            if tot > 0:
                return tot
        except Exception:
            continue
    return None


def kernel_report(event_log, steps, B, peaks):
    """Per-kernel device time inside the timed steps (CUDA events around each C-ABI call on the launching
    stream) -> share of the step and roofline of the dominant kernel (algorithmic work: DESIGN.md / SURVEY 8d)."""
    if not event_log:
        return {}
    agg = {}
    for name, evs in event_log.items():
        if name.startswith("__"):
            continue
        ms = [a.elapsed_time(b) for a, b in evs]
        agg[name] = {"launches_per_step": len(ms) / steps, "ms_per_step": sum(ms) / steps}
    total = sum(v["ms_per_step"] for v in agg.values())
    for v in agg.values():
        v["share"] = v["ms_per_step"] / total if total else 0.0
    top = max(agg, key=lambda n: agg[n]["ms_per_step"])
    out = {"kernels": {k: {kk: round(vv, 5) for kk, vv in v.items()} for k, v in sorted(agg.items())},
           "dominant_kernel": top}
    N0, k, S = N_PTS, 20, 7
    if top == "layer_conv":
        # conv_1..conv_4 launches: flops = N*k*S*C*9 + N*S*C ; compulsory bytes per SURVEY 8d
        shapes = [(N0, 20, 128), (N0 // 4, 20, 256), (N0 // 4, 20, 256), (N0 // 16, 8, 512)]
        flops = sum(n * kk * S * c * 9 + n * S * c for n, kk, c in shapes) * B
        byts = sum(4 * (3 * n + S * c * n + c * n + c * n + 3 * S * c) + 4 * n * kk for n, kk, c in shapes) * B
        t = agg[top]["ms_per_step"] / 1e3
        out["roofline"] = {"bound": "fp32", "kernel": "layer_conv_kernel (4 launches/step)",
                           "achieved": flops / t / 1e12, "peak": FP32_PEAK_TFLOPS, "unit": "TFLOP/s",
                           "frac": flops / t / 1e12 / FP32_PEAK_TFLOPS, "traffic": None,
                           "peak_source": "148 SM x 128 lanes x 2 flop x 1.965 GHz (SURVEY 8d); no measured fp32 peak",
                           "hbm": {"achieved": byts / t / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                   "frac": byts / t / 1e9 / peaks["hbm_gbs"], "peak_source": peaks["source"]}}
    elif top == "gemm_tc":
        # SURVEY 8d: achieved = algorithmic flops (the plain 2*M*K*N of every launch in the step) / summed launch time;
        # frac = achieved / TF32 peak, TF32 peak = measured dense bf16 / 2.  The tensor cores have no fp32 mode, so a
        # contraction held to fp32-level accuracy executes more than one tensor pass per algorithmic flop (3 TF32 passes for
        # the encoder's 3xTF32 operands, 1.5 TF32-pass equivalents for the heads' fp16 + 2 bf16 operands): that overhead is
        # the kernel's own and is reported beside the fraction (`executed_tf32_equiv_*`), not folded into the roof.
        shapes = [x for x in event_log.get("__gemm_shapes__", []) if x[0] == "gemm_tc"]
        # algorithmic flops = those of the REFERENCE's contraction: a launch that is a factored piece of one (the heads' first
        # layers with the upsampled channels contracted per coarse point, posenet.py) logs the reference figure it stands for
        def algo(m, kdim, n, rest):
            return float(rest[1]) if len(rest) > 1 and rest[1] is not None else 2.0 * m * kdim * n
        flops = sum(algo(m, kdim, n, rest) for _, m, kdim, n, *rest in shapes) / steps
        launched = sum(2.0 * m * kdim * n for _, m, kdim, n, *_ in shapes) / steps
        # the step runs at full SM clocks (1965 MHz sampled, no power capping even over 1000 steps), so the BURST bf16
        # figure is the applicable denominator, not the power-capped sustained one
        tf32_peak = peaks["bf16_tflops"] / 2.0
        exec_flops = sum(2.0 * m * kdim * n * (1.5 if (rest and rest[0]) else 3.0) for _, m, kdim, n, *rest in shapes) / steps
        t = agg[top]["ms_per_step"] / 1e3
        out["roofline"] = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05; all launches in the step)",
                           "achieved": flops / t / 1e12, "peak": tf32_peak, "unit": "TFLOP/s",
                           "frac": flops / t / 1e12 / tf32_peak, "traffic": profile_traffic("gemm_tc_kernel"),
                           "launched_2mnk_tflops": launched / t / 1e12,
                           "executed_tf32_equiv_tflops": exec_flops / t / 1e12,
                           "executed_tf32_equiv_frac": exec_flops / t / 1e12 / tf32_peak,
                           "peak_source": f"{peaks['source']} burst dense bf16 / 2 = TF32 rate (SM clocks stay at max during the step); "
                                          "achieved = algorithmic 2MNK flops of the reference's contractions that the gemm_tc launches "
                                          "compute / their summed CUDA-event time; launched_2mnk = 2MNK of the launches as issued (the "
                                          "heads' first layers contract their 1024 upsampled input channels per coarse point: 3x fewer)",
                           "traffic_source": "sum of dram__bytes_read+write over the gemm_tc launches of one forward, "
                                             "profiles/*_kernels.json (ncu); bytes per step"}
    # the other kernels of the step against their roofs (algorithmic work per SURVEY 8d at this step's shapes; times are
    # the per-call CUDA-event sums of the eager pass, which include a few us of event overhead per launch)
    N1, N2 = N0 // 4, N0 // 16
    k2 = min(k, N2 // 8)
    def ms(name):
        return agg[name]["ms_per_step"] / 1e3 if name in agg else None
    kr = {}
    if ms("knn_feat"):
        fl = B * sum(n * n * (2 * d + 3) + n * n for n, d in ((N0, 128), (N1, 128), (N1, 256), (N2, 256)))
        kr["knn_feat"] = {"bound": "fp32 roof (inner products run on the tensor pipe)", "achieved_tflops": fl / ms("knn_feat") / 1e12,
                          "frac_fp32": fl / ms("knn_feat") / 1e12 / FP32_PEAK_TFLOPS}
    if ms("knn_xyz"):
        fl = B * sum(n * n * 9 + n * n for n in (N0, N1, N2))
        kr["knn_xyz"] = {"bound": "fp32 / selection", "achieved_tflops": fl / ms("knn_xyz") / 1e12,
                         "frac_fp32": fl / ms("knn_xyz") / 1e12 / FP32_PEAK_TFLOPS,
                         "gpairs_s": B * (N0 * N0 + N1 * N1 + N2 * N2) / ms("knn_xyz") / 1e9}
    if ms("layer_conv_fwd"):
        shp = [(N0, k, 128), (N1, k, 256), (N1, k, 256), (N2, k2, 512)]
        fl = B * sum(n * kk * S * c * 9 + n * S * c for n, kk, c in shp)
        by = B * sum(4 * (3 * n + S * c * n + c * n + c * n + 3 * S * c) + 4 * n * kk for n, kk, c in shp)
        kr["layer_conv_fwd"] = {"bound": "fp32 roof in algorithmic flops; the kernel sits on the shared-memory pipe (ncu: LSU 81 %)", "achieved_tflops": fl / ms("layer_conv_fwd") / 1e12,
                                "frac_fp32": fl / ms("layer_conv_fwd") / 1e12 / FP32_PEAK_TFLOPS,
                                "compulsory_gbs": by / ms("layer_conv_fwd") / 1e9,
                                "frac_hbm": by / ms("layer_conv_fwd") / 1e9 / peaks["hbm_gbs"]}
    if ms("surface_conv_fwd"):
        fl = B * (N0 * k * S * 128 * 8 + N0 * S * 128)
        kr["surface_conv_fwd"] = {"bound": "fp32", "achieved_tflops": fl / ms("surface_conv_fwd") / 1e12,
                                  "frac_fp32": fl / ms("surface_conv_fwd") / 1e12 / FP32_PEAK_TFLOPS}
    if ms("orl_global"):
        by = B * sum(4 * n * c + 4 * n * kk + 4 * c for n, c, kk in ((N0, 128, k), (N0, 128, k), (N1, 256, k), (N1, 256, k), (N2, 512, k2)))
        kr["orl_global"] = {"bound": "hbm", "achieved_gbs": by / ms("orl_global") / 1e9,
                            "frac_hbm": by / ms("orl_global") / 1e9 / peaks["hbm_gbs"]}
    if ms("concat_rows"):
        # bytes moved by the two operand-assembly launches of the factored heads (posenet.py): per level-0 point the
        # [fm_0 | fm_1 | one-hot | xyz] row (265 floats read, 3 x 320 16-bit slots written), per level-1 point [fm_2 | fm_3]
        # (512 floats read, 3 x 512 slots written); the level-2 operand goes through split_mixed
        by = B * (N0 * (4 * 265 + 6 * 320) + N1 * (4 * 512 + 6 * 512))
        kr["concat_rows"] = {"bound": "hbm", "achieved_gbs": by / ms("concat_rows") / 1e9,
                             "frac_hbm": by / ms("concat_rows") / 1e9 / peaks["hbm_gbs"]}
    out["kernel_rooflines"] = {kk_: {a: (round(b, 4) if isinstance(b, float) else b) for a, b in v.items()} for kk_, v in kr.items()}
    if os.environ.get("TGP_BENCH_GEMM_TABLE"):
        shapes = event_log.get("__gemm_shapes__", [])
        evs = {"gemm": list(event_log.get("gemm", [])), "gemm_tc": list(event_log.get("gemm_tc", []))}
        pos = {"gemm": 0, "gemm_tc": 0}
        rows = {}
        for nm, m, kdim, n, *rest in shapes:
            a, b = evs[nm][pos[nm]]
            pos[nm] += 1
            rows.setdefault((nm, m, kdim, n) + tuple(rest), []).append(a.elapsed_time(b))
        for key, v in sorted(rows.items(), key=lambda kv: -sum(kv[1])):
            sys.stderr.write(f"GEMM {key}: {len(v) / steps:.1f}/step, {sum(v) / steps:.4f} ms/step\n")
    out["kernels"].pop("__gemm_shapes__", None)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="clouds per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the secondary `train` record (configs[2]) of the default run")
    ap.add_argument("--train-steps", type=int, default=5, help="timed steps of the secondary `train` record")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--mode", default="infer", choices=["infer", "train", "micro"],
                    help="infer: BASELINE.json configs[1] (the headline); train: configs[2], a secondary line")
    ap.add_argument("--train-batch", type=int, default=256, help="global batch of the training step")
    ap.add_argument("--optimizer", default="ranger", choices=["ranger", "adam"],
                    help="--mode train: the reference's Ranger (fused kernels) or torch's fused Adam")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (inference arm, rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.mode != "infer"):
        ap.error("--dump-outputs applies to the inference arm (--impl ours --mode infer)")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.mode == "train":
        run_train(args)
    elif args.mode == "micro":
        run_micro(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
