#!/usr/bin/env python
"""bench.py -- forward throughput (M points/s) of the hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload randlanet|pointpillars|kpconv]
    python bench.py --impl reference ...        # the CPU arm (torch port of the reference forward)
    python bench.py ... --dump-outputs DIR      # also write the outputs of the last timed step as DIR/<name>.npy

Launched by the driver either directly (N = 1) or through torch.distributed.run (one rank
per GPU, NCCL).  One JSON line on rank 0.  A "step" is one forward pass of the workload's
model over one synthetic batch:

  randlanet    (default; BASELINE.json configs[2]) RandLA-Net, SemanticKITTI shape: ONE batch of
               8 clouds x 45 056 pts sharded 8/N clouds per rank (strong scaling, the configuration
               BASELINE.json specifies), per-frame logits all-gathered over NCCL in the e2e region;
               `--units U` switches to weak scaling (U clouds per GPU)
  pointpillars (configs[1]) PointPillars, KITTI shape: frames of ~20 000 pts (`--shape waymo --total-units 32`
               = configs[4]: 32 Waymo-shaped frames of ~180 000 pts sharded over the ranks)
  kpconv       (configs[3]) KPFCNN, S3DIS shape: 4 clouds of 65 536 pts (rooms pre-gridded at 4 cm)

`value` : inputs resident in HBM, K steps between two barrier+synchronize brackets, CUDA
          events, max over ranks.
`e2e`   : the same K steps through the public API with PINNED HOST inputs: H2D of every input tensor,
          the forward, the post-batch all_gather of per-frame results (N > 1) and D2H of the result
          inside the timed region.  RandLA-Net is measured through both public entries -- the
          reference's input dict (int64 index pyramid from the host, 90 MB/step) and forward_points
          (points only; the k-NN pyramid of RandLANet.transform runs on the device) -- and the faster
          one is the headline; the other is reported beside it.
`roofline`: the dominant kernel class, timed with CUDA events inside the timed steps.
`cpu_baseline`: oracle/models_torch.py (the pinned port of the reference forward) on the
          host cores, bounded sample (rank 0, N = 1 only).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

L2_BYTES = 126e6


# ----------------------------------------------------------------------------- utilities
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], src="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (rank 0)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index
        self.t_begin = self.t_end = None

    def start(self):
        """Launches the sampler and waits for its first row (nvidia-smi needs ~0.1-1 s to come up;
        the timed region of a fast workload is shorter than that)."""
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "10"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t0 = time.perf_counter()
            while not self.rows and time.perf_counter() - t0 < 5.0:
                time.sleep(0.01)
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def begin(self):
        self.t_begin = time.perf_counter()

    def stop(self):
        self.t_end = time.perf_counter()
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.05)
        self.proc.terminate()
        lo = (self.t_begin or 0.0) - 0.005
        rows = [r for t, r in self.rows if lo <= t <= self.t_end + 0.015 and len(r) == 6]
        window = "timed region"
        if not rows:   # region shorter than the sampling period: take the rows around it
            rows = [r for t, r in self.rows if t >= lo - 0.25 and len(r) == 6]
            window = "timed region +-0.25 s"
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[2:]) if v.lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(sm), window=window)


def pin(t):
    return t.contiguous().pin_memory()


def nbytes(x):
    if isinstance(x, torch.Tensor):
        return x.numel() * x.element_size()
    if isinstance(x, dict):
        return sum(nbytes(v) for v in x.values())
    if isinstance(x, (list, tuple)):
        return sum(nbytes(v) for v in x)
    return 0


def to_dev(x, dev):
    if isinstance(x, torch.Tensor):
        return x.to(dev, non_blocking=True)
    if isinstance(x, dict):
        return {k: to_dev(v, dev) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [to_dev(v, dev) for v in x]
    return x


DUMP_BYTES = 60 * 10 ** 6      # what --dump-outputs writes in all stays under 64 MB, .npy headers included


def take_outputs(names, out):
    """The step's output tensors as host float32 arrays to be written as <name>.npy.  Larger than DUMP_BYTES together,
    every output is cut to the same fixed, seeded sample of its flattened elements, and <name>.index.npy (float64)
    holds the flat indices that were kept."""
    outs = out if isinstance(out, (tuple, list)) else (out,)
    assert len(outs) == len(names), (len(outs), names)
    total = 4 * sum(o.numel() for o in outs)
    arrays = {}
    for name, o in zip(names, outs):
        o = o.detach()
        if total > DUMP_BYTES:
            k = o.numel() * DUMP_BYTES // (3 * total)      # 4 bytes of value + 8 of index per kept element
            idx = np.unique(np.random.default_rng(0).integers(0, o.numel(), k))
            arrays[name + ".index"] = idx.astype(np.float64)
            o = o.reshape(-1)[torch.from_numpy(idx).to(o.device)]
        arrays[name] = o.float().cpu().numpy()
    return arrays


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ----------------------------------------------------------------------------- workloads
class RandLAWorkload:
    name = "RandLA-Net forward, SemanticKITTI-shaped batch (clouds of 45 056 pts; total_units below), BASELINE configs[2]"
    short = "randlanet_semantickitti_8x45056"
    manifest = "randlanet_semantickitti.manifest.json"
    output_names = ("logits",)

    default_total = 8

    def __init__(self, clouds=8, n=45056):
        self.B, self.N = clouds, n

    def points_per_step(self):
        return self.B * self.N

    def build_inputs_gpu(self, unit_ids):
        """KNN pyramid on the GPU (o3dml_knn_search), returned as HOST pinned tensors."""
        import open3d_ml_b200 as M
        from open3d_ml_b200 import synth
        per = []
        for u in unit_ids:
            pc = torch.from_numpy(synth.semantickitti_cloud(self.N, 1000 + u)).cuda()
            lv = dict(coords=[], neighbor_indices=[], sub_idx=[], interp_idx=[])
            for i in range(4):
                n = pc.shape[0]
                nb = M.knn_search(pc, pc, 16, index_dtype=torch.int64).neighbors_index.view(n, 16)
                sub = pc[:n // 4]
                up = M.knn_search(sub, pc, 1, index_dtype=torch.int64).neighbors_index.view(n, 1)
                lv["coords"].append(pc)
                lv["neighbor_indices"].append(nb)
                lv["sub_idx"].append(nb[:n // 4])
                lv["interp_idx"].append(up)
                pc = sub
            per.append(lv)
        inp = {k: [pin(torch.stack([p[k][i] for p in per]).cpu()) for i in range(4)]
               for k in ("coords", "neighbor_indices", "sub_idx", "interp_idx")}
        inp["features"] = pin(inp["coords"][0].clone())
        return inp

    def build_inputs_cpu(self, clouds):
        from oracle import models_torch as MT
        from open3d_ml_b200 import synth
        per = [MT.randlanet_build_inputs(synth.semantickitti_cloud(self.N, b)) for b in range(clouds)]
        inp = {k: [torch.from_numpy(np.stack([p[k][i] for p in per])) for i in range(4)]
               for k in ("coords", "neighbor_indices", "sub_idx", "interp_idx")}
        inp["features"] = inp["coords"][0].clone()
        return inp

    def make_model(self, sd):
        import open3d_ml_b200 as M
        return M.RandLANetB200(sd)

    def cpu_forward(self, sd, inp):
        from oracle import models_torch as MT
        return MT.randlanet_forward(sd, inp)

    def frames_out(self, out):
        return out                      # [B, N, classes]: one row block per frame

    # algorithmic bytes of one lfa_pool launch (DESIGN.md): per point 12 (xyz) + 8*16 (idx)
    # + 4*d/2 (gathered features, each input row once) + 4*d (pooled output)
    def roofline_bytes(self, d, points):
        return points * (12 + 128 + 2 * d + 4 * d)

    def roofline_flops(self, d, stage, points):
        h = d // 2
        per_nk = 2 * d * d + 2 * 10 * h + (2 * h * h if stage == 2 else 0) + 3 * d
        return points * 16 * per_nk


class PointPillarsWorkload:
    name = "PointPillars forward, synthetic KITTI frames (~20 000 pts), BASELINE configs[1]"
    short = "pointpillars_kitti"
    manifest = "pointpillars_kitti.manifest.json"
    output_names = ("cls", "reg", "dir")
    dense_gflop_per_frame = 68.3   # SECOND + SECONDFPN + head at 496 x 432 (SURVEY.md 8d)
    default_total = 1

    def __init__(self, frames=1, n=20000, shape="kitti"):
        self.B, self.N, self.shape = frames, n, shape
        if shape == "waymo":          # BASELINE configs[4]: ~180 000 pts in [-74.88, 74.88]^2 x [-2, 4], 468 x 468 BEV
            self.N = 180000 if n == 20000 else n
            self.name = "PointPillars forward, synthetic Waymo-shaped frames (~180 000 pts), BASELINE configs[4]"
            self.short = "pointpillars_waymo"
            self.manifest = "pointpillars_waymo.manifest.json"
            self.dense_gflop_per_frame = 279.5
            self.default_total = 32

    def points_per_step(self):
        return self.B * self.N

    def _frame(self, seed):
        from open3d_ml_b200 import synth
        if self.shape == "waymo":
            return synth.lidar_frame(self.N, seed, (-74.88, -74.88, -2, 74.88, 74.88, 4))
        return synth.lidar_frame(self.N, seed)

    def build_inputs_gpu(self, unit_ids):
        return [pin(torch.from_numpy(self._frame(1000 + u))) for u in unit_ids]

    def build_inputs_cpu(self, frames):
        return [torch.from_numpy(self._frame(b)) for b in range(frames)]

    def frames_out(self, out):
        return torch.cat([o.flatten(1) for o in out], 1)      # [B, (cls + reg + dir) * H * W]

    def make_model(self, sd):
        import open3d_ml_b200 as M
        return M.PointPillarsB200(sd, self.cfg)

    def cpu_forward(self, sd, inp):
        from oracle import models_torch as MT
        return MT.pointpillars_forward(sd, inp, self.cfg)


def pick_cpu_threads(wl, sd):
    """torch's CPU kernels do not scale to every core of a large host (oversubscription makes the
    128-thread run ~100x slower than 16 threads on the GPU box): time one small forward per
    candidate and keep the fastest, so that the CPU arm is the reference at its best."""
    n_all = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, n_all) if c <= n_all})
    small = type(wl)(1, 4096 if wl.N > 4096 else wl.N)
    small.cfg = getattr(wl, "cfg", None)
    inp = small.build_inputs_cpu(1)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        with torch.no_grad():
            small.cpu_forward(sd, inp)
            t0 = time.perf_counter()
            small.cpu_forward(sd, inp)
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


class KPConvWorkload:
    name = "KPConv (KPFCNN) forward, S3DIS-shaped clouds (65 536 pts, rooms pre-gridded at 4 cm), BASELINE configs[3]"
    short = "kpconv_s3dis"
    manifest = "kpconv_s3dis.manifest.json"
    output_names = ("logits",)
    gflop_per_cloud = 90.3   # SURVEY.md 8d (encoder 54.8 + decoder/head 35.5)
    default_total = 4

    def __init__(self, clouds=4, n=65536):
        self.B, self.N = clouds, n

    def points_per_step(self):
        return self.B * self.N

    def _clouds(self, count, seed0):
        from open3d_ml_b200 import synth
        return [synth.room_cloud(self.N, seed0 + b) for b in range(count)]

    def frames_out(self, out):
        return out.view(self.B, self.N, -1)

    def build_inputs_gpu(self, unit_ids):
        from open3d_ml_b200 import synth
        from open3d_ml_b200.kpconv import build_batch
        self.raw_clouds = [synth.room_cloud(self.N, 1000 + u) for u in unit_ids]
        b = build_batch(self.raw_clouds, self.cfg)
        return {k: ([pin(t.cpu()) for t in v] if isinstance(v, list) and v and isinstance(v[0], torch.Tensor)
                    else (pin(v.cpu()) if isinstance(v, torch.Tensor) else v)) for k, v in b.items()}

    def build_inputs_cpu(self, count):
        from open3d_ml_b200.kpconv import build_batch
        if torch.cuda.is_available():
            b = build_batch(self._clouds(count, 0), self.cfg)
            return {k: ([t.cpu() for t in v] if isinstance(v, list) and v and isinstance(v[0], torch.Tensor)
                        else (v.cpu() if isinstance(v, torch.Tensor) else v)) for k, v in b.items()}
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import helpers as H
        return H.kp_batch_tensors(H.kp_batch(self._clouds(count, 0), self.cfg))

    def make_model(self, sd):
        import open3d_ml_b200 as M
        return M.KPFCNNB200(sd, self.cfg)

    def cpu_forward(self, sd, inp):
        from oracle import models_torch as MT
        return MT.kpfcnn_forward(sd, inp, self.cfg)


def load_weights(wl, seed=1):
    from oracle import weights
    man, extra = weights.load_manifest(os.path.join(ROOT, "tests", "golden", wl.manifest))
    wl.cfg = extra.get("cfg")
    return weights.seeded_state_dict(man, seed)


# ----------------------------------------------------------------------------- reference arm
def run_reference(args, wl):
    """The reference's own forward on the host cores: the torch port of oracle/models_torch.py
    (pinned to the unmodified reference classes by tests/test_oracle_models.py).  The reference
    tree itself cannot be installed on the GPU box (its ops live in the absent `open3d` package,
    SURVEY.md section 0), hence kind = "port"."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sd = load_weights(wl)
    pick_cpu_threads(wl, sd)
    sample = 1
    inp = wl.build_inputs_cpu(sample)
    pts = sample * wl.N
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 2))):
            wl.cpu_forward(sd, inp)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = wl.cpu_forward(sd, inp)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, take_outputs(wl.output_names, out))
    v = pts * args.steps / dt / 1e6
    line = dict(metric="M points/s forward", value=round(v, 5), unit="Mpoints/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=round(1e3 * dt / args.steps, 3),
                higher_is_better=True, scaling=("weak" if args.units else "strong"), vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload=wl.name, sample="%d unit(s) of %d pts per step" % (sample, wl.N)),
                cpu_baseline=dict(value=round(v, 5), unit="Mpoints/s", cores=torch.get_num_threads(),
                                  kind="port", sample="%d x %d pts, %d steps" % (sample, wl.N, args.steps)),
                e2e=dict(value=round(v, 5), unit="Mpoints/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    emit(line)


# ----------------------------------------------------------------------------- B200 arm
def timed_region(fn, steps, dist_on, dev):
    import torch.distributed as dist
    torch.cuda.synchronize(dev)
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    if dist_on:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if dist_on:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def pin_to_gpu_numa_node(local):
    """Binds this rank's host threads to the cores of the NUMA node its GPU hangs off (the pinned-host -> device copies
    of the e2e region cross the inter-socket link otherwise: round-1 e2e scaling 0.90 at 8 GPUs).  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bdf = bus.lower()[-12:]                    # 0000:1b:00.0
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:  # noqa: BLE001
        return None


def ev_time_ms(fn, reps=5, warm=2):
    """Mean device time of fn() over reps, CUDA events on the current stream."""
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def measured_traffic(kind):
    """DRAM bytes per step of the dominant kernel class from the committed ncu --set full capture of THIS
    round's build (profiles/r02_traffic.json, written by tools/ncu_traffic.py); None when absent."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(path):
        return None, None
    d = json.load(open(path)).get(kind)
    if not d:
        return None, None
    return d.get("dram_bytes_per_step"), "profiles/r02_traffic.json (%s)" % d.get("source", "ncu --set full")


def run_b200(args, wl):
    import torch.distributed as dist
    from open3d_ml_b200 import _lib as L
    from open3d_ml_b200 import shard as SH
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist_on = world > 1
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa_node(local) if dist_on else None
    if dist_on:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    # ---- which units does this rank own?
    total = args.total_units or (0 if args.units else wl.default_total)
    if total and total >= world:
        scaling = "strong"                       # one fixed batch sharded over the ranks (BASELINE configs[2]/[4])
        lo, hi = SH.shard_bounds(total, rank, world)
        unit_ids = list(range(lo, hi))
    else:
        scaling = "weak"
        per = args.units or 1
        total = per * world
        unit_ids = list(range(rank * per, (rank + 1) * per))
    wl.B = len(unit_ids)
    sd = load_weights(wl)
    model = wl.make_model(sd)
    host_inp = wl.build_inputs_gpu(unit_ids)
    dev_inp = to_dev(host_inp, dev)
    is_rl = hasattr(model, "forward_points")
    graphed = is_rl and hasattr(model, "forward_graphed")

    last_out = [None]

    def step_resident():
        last_out[0] = model.forward_graphed(dev_inp) if graphed else model(dev_inp)
        return last_out[0]

    def with_gather(out):
        """Post-batch exchange (object_detection.py:222-233 / SURVEY 8e): all_gather of the per-frame results over NCCL so
        that every rank holds the whole batch on the device; each rank hands its OWN frames' results to its host, rank 0
        additionally the whole-batch summary the metrics need (semseg: the label map of every frame, uint8; detection:
        the per-frame maximum) -- reading all logits back through rank 0's PCIe link would serialise the job on it
        (219 MB per step at 8 GPUs x 8 clouds)."""
        if not dist_on:
            return out
        fr = wl.frames_out(out).contiguous()
        allf = SH.gather_frame_results(fr, total)
        if rank != 0:
            return fr
        summary = allf.argmax(-1).to(torch.uint8) if allf.dim() == 3 else allf.amax(dim=1)
        return fr, summary

    for _ in range(args.warmup):
        step_resident()
    # --- roofline instrumentation: CUDA events around every launch of the dominant kernel class (eager steps
    # after the timed region: a graph replay has no per-kernel events)
    timers = []
    dense_timers = []
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(2):           # the GPU idled while the sampler came up: re-warm the clocks
        step_resident()
    if hasattr(model, "backbone_neck_head"):
        orig_bnh = model.backbone_neck_head

        def timed_bnh(canvas):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            r = orig_bnh(canvas)
            b.record()
            dense_timers.append((a, b, canvas.shape[0]))
            return r
        model.backbone_neck_head = timed_bnh
    if rank == 0:
        clocks.begin()
    launches0 = L.lib().o3dml_launch_count()
    torch.cuda.cudart().cudaProfilerStart()      # ncu --profile-from-start off sees only the timed steps
    ms = timed_region(step_resident, args.steps, dist_on, dev)
    torch.cuda.cudart().cudaProfilerStop()
    launches = L.lib().o3dml_launch_count() - launches0
    clk = clocks.stop() if rank == 0 else None
    # copied before any later call can overwrite them (graph replays reuse their output buffers)
    dumped = take_outputs(wl.output_names, last_out[0]) if args.dump_outputs and rank == 0 else None
    if hasattr(model, "backbone_neck_head"):
        model.backbone_neck_head = orig_bnh      # timers cover the resident region only
    lfa_ms_in_step = None
    if hasattr(model, "_lfa_pool"):
        orig = model._lfa_pool

        def timed_lfa(stage, d, coords, nidx, feat, B, N, p, agg):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            orig(stage, d, coords, nidx, feat, B, N, p, agg)
            b.record()
            timers.append((stage, d, B * N, a, b))
        model._lfa_pool = timed_lfa
        for _ in range(3):
            model(dev_inp)                       # eager, same stream, back to back with warm clocks
        timers.clear()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            model(dev_inp)
        e1.record()
        torch.cuda.synchronize()
        model._lfa_pool = orig
        lfa_ms_in_step = e0.elapsed_time(e1)
    # --- e2e A: the reference-facing call (host input pytree as the reference's dataloader delivers it)
    from open3d_ml_b200 import PipelinedRunner
    gather_on = [False]
    base = model.forward_graphed if graphed else model
    fwd = lambda d: with_gather(base(d)) if gather_on[0] else base(d)   # noqa: E731
    runner = PipelinedRunner(fwd, dev)

    def e2e_stream(run, inp, n):
        acc = 0.0
        for res in run.run(inp for _ in range(n)):
            r0 = res[0] if isinstance(res, tuple) else res
            acc += float(r0.view(-1)[0])          # the caller touches every result on the host
        return acc

    # first pass without the collective: the CUDA graphs of both input slots are captured while no NCCL work is in
    # flight (capturing with a collective of the previous batch still running faulted on 2 of 4 ranks at N = 4)
    e2e_stream(runner, host_inp, 2)
    torch.cuda.synchronize(dev)
    if dist_on:
        dist.barrier()
    gather_on[0] = True
    e2e_stream(runner, host_inp, max(3, args.warmup // 2))
    # the e2e region is host-paced (pinned copies, Python between batches): one scheduling hiccup of the box triples a
    # 20-step region, so it is timed twice (K steps each, max over ranks each) and the faster one is reported
    ms_e2e = min(timed_region(lambda: e2e_stream(runner, host_inp, args.steps), 1, dist_on, dev) for _ in range(2))
    out_host = None

    def step_e2e_sync():
        nonlocal out_host
        out = with_gather(model(host_inp))       # eager (no graph): plain synchronous call   # H2D of every input inside the model call (randlanet.py:254-264)
        outs = out if isinstance(out, (tuple, list)) else (out,)
        if out_host is None:
            out_host = [torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs]
        for h, o in zip(out_host, outs):
            h.copy_(o, non_blocking=True)
        torch.cuda.current_stream().synchronize()   # the caller consumes the result every step

    for _ in range(2):
        step_e2e_sync()
    ms_e2e_sync = timed_region(step_e2e_sync, args.steps, dist_on, dev)
    pts_step = wl.N * total
    e2e_modes = {"reference_inputs": dict(
        value=round(pts_step * args.steps / (ms_e2e * 1e-3) / 1e6, 3), ms_per_step=round(ms_e2e / args.steps, 4),
        h2d_bytes_per_step=nbytes(host_inp),
        mode="PipelinedRunner over the reference's input pytree (2 slots: copies of neighbouring batches overlap the forward); "
             "faster of two K-step regions",
        sync_value=round(pts_step * args.steps / (ms_e2e_sync * 1e-3) / 1e6, 3))}
    # --- e2e B (RandLA-Net): points only; RandLANet.transform's k-NN pyramid runs on the device
    extra = {}
    if is_rl:
        pts_host = dict(points=pin(host_inp["coords"][0].clone()))
        gather_on[0] = False
        fwd_pts = lambda d: (with_gather(model.forward_points_graphed(d["points"])) if gather_on[0]   # noqa: E731
                             else model.forward_points_graphed(d["points"]))
        runner_p = PipelinedRunner(fwd_pts, dev)
        e2e_stream(runner_p, pts_host, 2)
        torch.cuda.synchronize(dev)
        if dist_on:
            dist.barrier()
        gather_on[0] = True
        e2e_stream(runner_p, pts_host, max(3, args.warmup // 2))
        ms_p = min(timed_region(lambda: e2e_stream(runner_p, pts_host, args.steps), 1, dist_on, dev) for _ in range(2))
        e2e_modes["points_only"] = dict(
            value=round(pts_step * args.steps / (ms_p * 1e-3) / 1e6, 3), ms_per_step=round(ms_p / args.steps, 4),
            h2d_bytes_per_step=nbytes(pts_host),
            mode="PipelinedRunner over forward_points: only xyz crosses PCIe, the k-NN pyramid (randlanet.py:218-229) "
                 "is built on the device inside the timed region, pyramid + forward replayed from one CUDA graph")
        dpts = dev_inp["coords"][0]
        extra["knn_pyramid_ms"] = round(ev_time_ms(lambda: model.build_pyramid(dpts)), 4)
        extra["forward_points_ms"] = round(ev_time_ms(lambda: model.forward_points_graphed(dpts)), 4)
    if hasattr(wl, "raw_clouds"):
        from open3d_ml_b200.kpconv import build_batch
        t0 = time.perf_counter()
        for _ in range(3):
            build_batch(wl.raw_clouds, wl.cfg)
        torch.cuda.synchronize()
        extra["kpconv_batch_build_ms"] = round((time.perf_counter() - t0) / 3 * 1e3, 3)
        extra["kpconv_batch_build_note"] = ("KPConvBatch.segmentation_inputs on the device: 13 radius searches + 4 grid "
                                            "subsamplings, wall clock incl. the size read-backs (concat_batcher.py:186-305)")
    value = pts_step * args.steps / (ms * 1e-3) / 1e6
    outs = with_gather(step_resident())
    outs = outs if isinstance(outs, (tuple, list)) else (outs,)
    chk = torch.stack([o.float().abs().mean() for o in outs]).sum().reshape(1)
    assert bool(torch.isfinite(chk).all())

    if rank != 0:
        if dist_on:
            dist.destroy_process_group()
        return
    pk = peaks()
    roof = None
    if timers:
        tot_ms = sum(a.elapsed_time(b) for _, _, _, a, b in timers)
        tot_bytes = sum(wl.roofline_bytes(d, n) for _, d, n, _, _ in timers)
        tot_flops = sum(wl.roofline_flops(d, s, n) for s, d, n, _, _ in timers)
        per = {}
        for s, d, n, a, b in timers:
            k = "lfa_pool<d=%d,stage=%d>" % (d, s)
            e = per.setdefault(k, [0.0, 0, 0.0, 0])
            e[0] += a.elapsed_time(b)
            e[1] += 1
            e[2] += wl.roofline_bytes(d, n)
            e[3] += wl.roofline_flops(d, s, n)
        ach = tot_bytes / (tot_ms * 1e-3) / 1e9
        traffic, tsrc = measured_traffic("lfa_pool") if (wl.B, wl.N) == (8, 45056) else (None, None)
        roof = dict(bound="hbm", kernel="lfa_pool: tcgen05 lfa_pool_tc_kernel (d>=64) + lfa16c_kernel (d=16), all 8 launches per step",
                    achieved=round(ach, 2), peak=pk["hbm_gbs"], unit="GB/s", frac=round(ach / pk["hbm_gbs"], 5),
                    algorithmic_bytes=int(tot_bytes / max(1, args.steps)), traffic=traffic, traffic_source=tsrc,
                    peak_source=pk["src"], timed="CUDA events around each launch in %d eager steps run right after the "
                    "timed (graph-replayed) region" % args.steps,
                    share_of_step=round(tot_ms / lfa_ms_in_step, 4),
                    fp32_tflops=round(tot_flops / (tot_ms * 1e-3) / 1e12, 3),
                    per_kernel={k: dict(avg_us=round(1e3 * e[0] / e[1], 2),
                                        gbs=round(e[2] / (e[0] * 1e-3) / 1e9, 1),
                                        tflops=round(e[3] / (e[0] * 1e-3) / 1e12, 2))
                                for k, e in sorted(per.items())})
    pkj = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    peak_tf = float(pkj.get("bf16_tflops", 1590.0))
    peak_src = "measured bf16 cuBLAS burst (MEASURED_PEAKS.json)" if pkj else "fallback (B200_PROFILING.md)"
    if dense_timers:
        # PointPillars: the dense BEV backbone + neck + head (SECOND/FPN/Anchor3DHead, 20 implicit-GEMM
        # launches of gemm_tc_kernel) is the dominant kernel class: tensor-core bound
        tot_ms = sum(a.elapsed_time(b) for a, b, _ in dense_timers)
        frames = sum(n for _, _, n in dense_timers)
        gflop = wl.dense_gflop_per_frame * frames
        ach = gflop / tot_ms            # GFLOP / ms = TFLOP/s
        traffic, tsrc = measured_traffic("pp_dense")
        roof = dict(bound="tensor", kernel="gemm_tc_kernel (tcgen05 kind::tf32, 3xTF32 split, TMA-fed): SECOND + SECONDFPN + head, 20 launches/frame",
                    achieved=round(ach, 2), peak=peak_tf, unit="TFLOP/s", frac=round(ach / peak_tf, 5), traffic=traffic,
                    traffic_source=tsrc, peak_source=peak_src,
                    share_of_step=round(tot_ms / ms, 4), algorithmic_gflop_per_frame=wl.dense_gflop_per_frame,
                    note="algorithmic FLOPs (SURVEY 8d); the 3xTF32 split issues 3x that at the TF32 rate (half the bf16 "
                         "rate the peak was measured at): the kernel's own ceiling is peak / 6")
    if roof is None and hasattr(wl, "gflop_per_cloud"):
        ach = wl.gflop_per_cloud * wl.B * args.steps / ms
        roof = dict(bound="tensor", kernel="whole KPFCNN forward (kpconv_gather + gemm_tc_kernel)", achieved=round(ach, 2),
                    peak=peak_tf, unit="TFLOP/s", frac=round(ach / peak_tf, 5), traffic=None, peak_source=peak_src,
                    algorithmic_gflop_per_cloud=wl.gflop_per_cloud)
    # --- cpu baseline (bounded sample, N = 1 only) + the same port run eagerly on the GPU (informational)
    cpu = None
    if world == 1 and not args.no_cpu:
        pick_cpu_threads(wl, sd)
        cin = wl.build_inputs_cpu(1)
        with torch.no_grad():
            wl.cpu_forward(sd, cin)
            t0 = time.perf_counter()
            reps = 3
            for _ in range(reps):
                wl.cpu_forward(sd, cin)
            dt = (time.perf_counter() - t0) / reps
        cpu = dict(value=round(wl.N / dt / 1e6, 5), unit="Mpoints/s", cores=torch.get_num_threads(),
                   kind="port", sample="1 unit of %d pts, %d forwards, oracle/models_torch.py" % (wl.N, reps))
        try:
            sd_g = {k: v.to(dev) for k, v in sd.items()}
            gin = to_dev(cin, dev)
            with torch.no_grad():
                t_g = ev_time_ms(lambda: wl.cpu_forward(sd_g, gin), reps=5, warm=2)
            extra["gpu_eager_baseline"] = dict(value=round(wl.N / (t_g * 1e-3) / 1e6, 4), unit="Mpoints/s",
                                               what="the same torch port (oracle/models_torch.py) run eagerly on this GPU with "
                                                    "library kernels, 1 unit; informational: what the reference's own torch code "
                                                    "gets from a B200 without this library")
        except Exception as e:  # noqa: BLE001
            msg = str(e)[:200]
            if "numpy" in msg:
                msg = "the torch port of this workload voxelizes on the host with numpy: no GPU-eager arm"
            extra["gpu_eager_baseline"] = dict(unavailable=msg)
    best = max(e2e_modes, key=lambda k: e2e_modes[k]["value"])
    e2e = dict(e2e_modes[best], unit="Mpoints/s", entry=best,
               d2h_bytes_per_step=sum(nbytes(o) for o in outs),
               collective=("all_gather of per-frame results over NCCL every step (shard.gather_frame_results)"
                           if dist_on else "none (1 rank)"),
               other_entries={k: v for k, v in e2e_modes.items() if k != best})
    bi = nbytes(host_inp)
    line = dict(metric="M points/s forward", value=round(value, 3), unit="Mpoints/s", n_gpus=world,
                steps=args.steps, warmup=args.warmup, ms_per_step=round(ms / args.steps, 4),
                higher_is_better=True, scaling=scaling, vs_baseline=None, dtype="f32", data="synthetic",
                config=dict(workload=wl.name, total_units=total, units_on_rank0=wl.B, points_per_unit=wl.N,
                            parallelism="frame-shard x%d (%s scaling), no data-path collective in the forward; "
                                        "post-batch all_gather of per-frame results in the e2e region" % (world, scaling),
                            l2="inputs + activations per step (%.0f MB inputs) exceed the 126 MB L2; no flush"
                               % (bi / 1e6),
                            launch="forward replayed from a CUDA graph" if graphed or dense_timers else "eager launches",
                            numa_node_rank0=numa),
                clocks=clk, e2e=e2e, gpu_launches=int(launches), roofline=roof, cpu_baseline=cpu, **extra)
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    emit(line)
    if dist_on:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the process's original stdout."""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # libraries (NCCL's version banner, torchrun notices) write to fd 1: keep the original stdout
    # for the JSON line only and send everything else to stderr
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="randlanet", choices=["randlanet", "pointpillars", "kpconv"])
    ap.add_argument("--units", type=int, default=0, help="clouds / frames PER GPU: weak scaling (0 = strong scaling)")
    ap.add_argument("--total-units", type=int, default=0,
                    help="clouds / frames in the whole batch, sharded over the ranks: strong scaling (0 = config default)")
    ap.add_argument("--shape", default="kitti", choices=["kitti", "waymo"], help="pointpillars frame shape")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32; rank 0's frames; a fixed "
                         "seeded sample of each output when they exceed 60 MB together, see take_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    wl = (RandLAWorkload(args.units or 8) if args.workload == "randlanet" else
          PointPillarsWorkload(args.units or 1, shape=args.shape) if args.workload == "pointpillars" else
          KPConvWorkload(args.units or 4))
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_b200(args, wl)


if __name__ == "__main__":
    main()
