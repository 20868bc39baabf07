#!/usr/bin/env python
"""SPG step benchmark (BASELINE.json: "SPG train-step edges+points/sec ...; ECC scatter HBM %peak").

    python bench.py --gpus N --steps K --warmup W                 # this repo's sm_100a path, configs[1]
    python bench.py --impl reference --steps K --warmup W         # the reference's own CPU modules
    python bench.py --workload room_fwd|sema3d_eval|vkitti_train|sweep_vv|sweep_mat [--nodes N]

Default workload (the headline line): one full training step of configs[1] ("S3DIS Area-5 fold
training, gru_10_1_1_1_0, fp32") on one synthetic S3DIS-shaped batch per GPU: PointNet embedding of
every superpoint that has a cloud, filter network, 10 x {ECC, GRUCellEx}, classifier, weighted CE,
full backward, element-wise gradient clamp, Adam (learning/main.py:199-213).  value = (edges +
points) per second summed over ranks (weak scaling: one batch of scenes per rank, one all-reduce of
the flat gradient per step).  The other BASELINE configs are `--workload` lines (superpoint_graph_
b200/workloads.py); inference workloads time main.py:229-264's forward.

The line also carries `parity_rel_err`: the first step from the initial state, checked against one
step of the CPU arm on the same batch (the bench measures, the tests assert).

Timing: every step is bracketed by CUDA events on the launching stream; an L2 flush (a 256 MiB
memset) runs between steps outside the brackets; the reported time is the max over ranks of the
summed step times, after a barrier + synchronize on both sides of the K steps.

Reference arm: build() compiles the reference's learning/{pointnet,graphnet,modules}.py and
learning/ecc/* to bytecode under oracle/_ref/ where a reference checkout exists (oracle/build_ref.py).
`--impl reference` drives those modules through their own API on the host CPU (baseline/ref_arm.py);
`cpu_baseline.kind` is "reference" then, "port" (oracle/nets_ref) without them.

`--dump-outputs DIR` writes what the timed path returned in its last timed step (rank 0): logits.npy
(float32 [superpoints, classes]) and, for training workloads, loss.npy (float32 [1]).  Inputs and
initial weights are seeded, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "spg_train_step_edges_plus_points_per_sec"
METRIC_EVAL = "spg_forward_edges_plus_points_per_sec"
UNIT = "edges+points/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="s3dis_train",
                    help="s3dis_train (configs[1], default) | room_fwd (configs[0]) | sema3d_eval (configs[2]) | "
                         "vkitti_train (configs[3]) | sweep_vv | sweep_mat (configs[4])")
    ap.add_argument("--nodes", type=int, default=None, help="superpoints per batch (default: the workload's)")
    ap.add_argument("--no-parity", action="store_true", help="skip the one-step check against the reference/oracle")
    ap.add_argument("--ecc-nodes", type=int, default=100000, help="ECC roofline microbench size")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer pass (profiling runs)")
    ap.add_argument("--trace-gemm", action="store_true", help="per-shape timing of the SIMT GEMM calls (stderr)")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches only (no CUDA-graph replay)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), bf16=float(d["bf16_tflops"]),
                    bf16_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def workload_counts(batch):
    from superpoint_graph_b200.synthetic import batch_counts
    N, nv, pts, E = batch_counts(batch)
    return dict(superpoints=N, embedded_superpoints=nv, points=pts, edges=E)


class ClockSampler(object):
    """SM clock + throttle reasons sampled DURING the timed region: NVML from a background thread
    (every ~5 ms); `nvidia-smi -lms` as a fallback when NVML cannot be loaded."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, "/tmp/spg_clocks_%d.csv" % os.getpid()
        self.thread, self.stop_flag, self.samples, self.reasons, self.max_mhz = None, False, [], set(), None

    def _nvml_loop(self, nv, handle):
        masks = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                for name, m in masks.items():
                    if r & m:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import threading

            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES if it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except Exception:
                    idx = self.index
            handle = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            if self.samples:
                sm = sorted(self.samples)
                out = {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz,
                       "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml"}
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, mx = [], set(), None
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                sm.append(float(f[1]))
                mx = float(f[2])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        except Exception:
            pass
        if sm:
            sm.sort()
            out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                   "source": "nvidia-smi"}
        return out


# ------------------------------------------------------------------------------ reference arm
def host_info():
    model = None
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"nproc": os.cpu_count() or 1, "cpu_model": model}


class CpuArm(object):
    """The reference's CPU path for one workload: the reference's OWN modules when oracle/_ref holds
    them (kind "reference": baseline/ref_arm.py), else the oracle port (kind "port")."""

    def __init__(self, w, sd_ecc=None, sd_ptn=None):
        from baseline import ref_arm
        self.w, self.margs = w, w["margs"]
        self.kind = "reference" if ref_arm.available() else "port"
        self.sd = (sd_ecc, sd_ptn)
        self._make()

    def _make(self):
        sd_ecc, sd_ptn = self.sd
        if self.kind == "reference":
            from baseline import ref_arm
            self.impl = ref_arm.ReferenceStep(self.margs, seed=1)
            if sd_ecc is not None:
                self.impl.load(sd_ecc, sd_ptn)
        else:
            from oracle import nets_ref
            from superpoint_graph_b200 import workloads
            from superpoint_graph_b200.trainer import create_model
            if sd_ecc is None:
                torch.manual_seed(1)
                model = create_model(self.margs)
                sd_ecc, sd_ptn = model.ecc.state_dict(), model.ptn.state_dict()
            self.pcfg, self.mcfg = workloads.oracle_cfg(self.margs)
            self.impl = nets_ref.RefTrainer(sd_ptn, sd_ecc, self.pcfg, self.mcfg, lr=self.margs.lr,
                                            grad_clip=self.margs.grad_clip, ecc_mode="loop")

    def step(self, batch):
        """-> (loss | None, logits)"""
        if self.w["train"]:
            if self.kind == "reference":
                try:
                    return self.impl.train_step(batch)
                except RuntimeError as ex:
                    # the reference's matrix-filter backward does not run on torch >= 2 (index_add_ shape
                    # check at learning/ecc/GraphConvModule.py:146, SURVEY.md 8(c)): time the oracle port
                    if "source tensor shape must match" not in str(ex):
                        raise
                    self.kind, self.note = "port", ("the reference's matrix-filter backward fails on torch>=2 "
                                                    "(ecc/GraphConvModule.py:146): oracle port timed instead")
                    self._make()
            return self.impl.step(batch)
        if self.kind == "reference":
            return None, self.impl.eval_step(batch)
        from oracle import nets_ref
        with torch.no_grad():
            return None, nets_ref.spg_forward(batch, self.impl.sd_ptn, self.impl.sd_ecc, self.pcfg, self.mcfg,
                                              False, ecc_mode="loop")

    def describe(self):
        if getattr(self, "note", None):
            return "oracle port of the reference CPU path (oracle/nets_ref, ecc_mode=loop); " + self.note
        if self.kind == "reference":
            return ("the reference's own modules (oracle/_ref: learning/pointnet.py, graphnet.py, modules.py, "
                    "ecc/*; use_pyg=0, cuda=False) through CloudEmbedder.run / GraphNetwork / cross_entropy / "
                    "clamp / Adam")
        return "oracle port of the reference CPU path (oracle/nets_ref, ecc_mode=loop)"

    def pick_threads(self, batch, budget_s=20.0):
        """torch's CPU kernels on these tensors get slower with very many threads; use the fastest of
        a few thread counts up to all cores (one probe step each, bounded)."""
        ncpu = os.cpu_count() or 1
        best, best_t = ncpu, float("inf")
        t_begin = time.perf_counter()
        for th in sorted({min(8, ncpu), min(16, ncpu), min(32, ncpu), ncpu}):
            torch.set_num_threads(th)
            self.step(batch)
            t0 = time.perf_counter()
            self.step(batch)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = th, dt
            if time.perf_counter() - t_begin > budget_s:
                break
        torch.set_num_threads(best)
        self._make()  # probing advanced the optimizer: start again from the initial state
        return best


def config_of(w, counts, world):
    """The `config` object — identical in both arms for the same launch."""
    return dict(workload=w["title"],
                parallelism="scene-parallel dp%d, one all-reduce of the flat gradient per step" % world
                if w["train"] else "scene-parallel dp%d (inference: no collective)" % world,
                l2="256 MiB memset between timed steps (outside the event brackets); 4 rotating batches",
                **counts)


def cpu_sample_nodes(w):
    """Bounded CPU sample: the per-node Python loops of the reference make a CPU step ~1 ms per
    superpoint-iteration; cap the sample so a K-step run ends within minutes."""
    return min(w["nodes"], 2048)


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the workload's step on this box's
    host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from superpoint_graph_b200 import workloads
    w = workloads.get(args.workload, args.nodes)
    counts_full = workload_counts(workloads.batch(w, 1)) if w["nodes"] <= 32768 else None
    ws = workloads.get(args.workload, cpu_sample_nodes(w))
    batch = workloads.batch(ws, 1)
    counts = workload_counts(batch)
    arm = CpuArm(ws)
    threads = arm.pick_threads(batch)
    for _ in range(args.warmup):
        arm.step(batch)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arm.step(batch)
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    value = (counts["edges"] + counts["points"]) / dt
    world = int(os.environ.get("WORLD_SIZE", "1"))
    sample = "%d full %s steps on a batch of %d superpoints (%s)" % (
        args.steps, "training" if w["train"] else "inference", counts["superpoints"], arm.describe())
    if ws["nodes"] != w["nodes"]:
        sample += "; bounded sample of the %d-superpoint workload, throughput is size-normalised" % w["nodes"]
    line = {
        "impl": "reference", "metric": METRIC if w["train"] else METRIC_EVAL, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
        "config": config_of(w, counts_full or workload_counts_nominal(w, counts), world),
        "rates": rates(counts, 1, dt * 1e3),
        "cpu_baseline": dict(value=value, unit=UNIT, cores=threads, kind=arm.kind, sample=sample, **host_info()),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_counts_nominal(w, sample_counts):
    """Counts of the full workload when only a bounded sample was generated on the CPU arm (scaled)."""
    k = w["nodes"] / float(sample_counts["superpoints"])
    return {key: int(round(v * k)) for key, v in sample_counts.items()}


def rates(counts, world, ms_per_step):
    """SURVEY 8(d): the metric's components, whole job."""
    k = world / (ms_per_step * 1e-3)
    return {"superpoints_per_s": counts["superpoints"] * k, "points_per_s": counts["points"] * k,
            "edges_per_s": counts["edges"] * k, "edge_iterations_per_s": counts["edges"] * 10 * k}


# ------------------------------------------------------------------------------------ our arm
def cpu_baseline(w, sd_ecc, sd_ptn, budget_s=25.0):
    """`cpu_baseline` of the b200 line: the same CPU arm, bounded sample, timed on this box."""
    from superpoint_graph_b200 import workloads
    ws = workloads.get(w["name"], cpu_sample_nodes(w))
    batch = workloads.batch(ws, 1)
    counts = workload_counts(batch)
    arm = CpuArm(ws, sd_ecc, sd_ptn)
    threads = arm.pick_threads(batch, budget_s=budget_s / 2)
    arm.step(batch)  # warm-up
    times = []
    t_start = time.perf_counter()
    while len(times) < 5 and (time.perf_counter() - t_start) < budget_s / 2:
        t0 = time.perf_counter()
        arm.step(batch)
        times.append(time.perf_counter() - t0)
    times.sort()
    dt = times[len(times) // 2]
    return dict(value=(counts["edges"] + counts["points"]) / dt, unit=UNIT, cores=threads, kind=arm.kind,
                sample="median of %d full steps on a batch of %d superpoints on the host (%s)" % (
                    len(times), counts["superpoints"], arm.describe()),
                ms_per_step=dt * 1e3, **host_info())


def parity_check(w, batch, sd_ecc, sd_ptn, loss, logits):
    """One step of the CPU arm from the same initial state on the same batch: relative errors of the
    GPU step's loss and logits (the bench asserts nothing; the line carries the numbers)."""
    arm = CpuArm(w, sd_ecc, sd_ptn)
    ref_loss, ref_logits = arm.step(batch)
    lg = logits.detach().float().cpu()
    out = {"logits": float((lg - ref_logits).abs().max() / ref_logits.abs().max()), "checker": arm.kind,
           "superpoints": int(lg.shape[0])}
    if ref_loss is not None:
        out["loss"] = abs(float(loss) - ref_loss) / abs(ref_loss)
    return out


def ncu_traffic():
    """Per-launch DRAM traffic of the dominant kernels from the committed ncu captures
    (profiles/ncu_traffic.json); {} if the file is missing."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            return json.load(f)
    except (OSError, ValueError):
        return {}


def ecc_roofline(dev, n_nodes, pk, flush, sweep=True):
    """ECC gather-product-scatter kernels at sweep size (configs[4]), measured honestly: the L2 is
    flushed (256 MiB memset) before EVERY timed launch, so nothing is served from a warm L2; sizes
    10 k / 100 k / 300 k superpoints with ~10 and ~20 in-edges per node.  Algorithmic bytes per
    SURVEY.md 8(d): filters once, node rows once (gathers counted as compulsory), output once, int32
    indices.  The matrix-filter kernels ([E,32,32], 4 KB per edge) run at the headline size only."""
    from superpoint_graph_b200 import ops
    from superpoint_graph_b200.synthetic import make_batch
    H = 32

    def timed(fn, reps=7):
        for _ in range(2):
            fn()
        ts = []
        for _ in range(reps):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            e.synchronize()
            ts.append(s.elapsed_time(e))
        ts.sort()
        return ts[len(ts) // 2]

    def one(n, k, modes):
        b = make_batch(n_nodes=n, k=k, seed=5, npts=1, minpts=1)
        N, E = b["degs"].numel(), b["idxn"].numel()
        graph = ops.EccGraph(b["idxn"], None, b["degs"], n_in=N)
        x = torch.randn(N, H, device=dev)
        g = torch.randn(N, H, device=dev)
        res = {}
        for mode in modes:
            w = torch.randn((E, H, H) if mode == "mat" else (E, H), device=dev)
            wbytes = 4 * H * H * E if mode == "mat" else 4 * H * E
            gw = torch.empty_like(w)
            cases = {
                "fwd": (lambda: ops.ecc_fwd(x, w, graph, H), wbytes + 8 * H * N + 4 * E + 4 * (N + 1)),
                "bwd_x": (lambda: ops.ecc_bwd_x(w, g, graph, H), wbytes + 8 * H * N + 8 * E + 8 * (N + 1)),
                "bwd_w": (lambda: ops.ecc_bwd_w(x, g, graph, tuple(w.shape), out=gw),
                          wbytes + 8 * H * N + 4 * E + 4 * (N + 1)),
            }
            for name, (fn, nbytes) in cases.items():
                ms = timed(fn)
                gbs = nbytes / (ms * 1e-3) / 1e9
                res["%s_%s" % (mode, name)] = {"ms": ms, "bytes": nbytes, "gbs": gbs, "frac": gbs / pk["hbm"]}
            del w, gw
        return dict(nodes=N, edges=E, kernels=res)

    head = one(n_nodes, 8, ("vv", "mat"))
    head["l2"] = "256 MiB memset before every timed launch"
    if sweep:
        head["sweep_vv"] = [dict(nodes=r["nodes"], edges=r["edges"],
                                 **{k: round(v["frac"], 4) for k, v in r["kernels"].items()})
                            for r in (one(n, k, ("vv",)) for n in (10000, 100000, 300000) for k in (8, 18))]
    return head


def loader_roofline(dev, pk, with_cpu):
    """Per-superpoint batch loader (SURVEY.md 8(f) rank 1): `spg_cloud_build` on 32768 resident
    superpoints of 40..600 points (S3DIS attributes, L=128) against the HBM roofline, and the
    reference's numpy `load_superpoint` (oracle port) on a bounded sample of the same superpoints.
    Algorithmic bytes per output point: F*4 read + 4 (sample index) + F*4 written."""
    from types import SimpleNamespace

    from superpoint_graph_b200 import ops
    from superpoint_graph_b200.spg_loader import attrib_columns
    rng = np.random.default_rng(2)
    nv, L, C = 32768, 128, 15
    counts = rng.integers(40, 601, size=nv)
    starts = np.concatenate([[0], np.cumsum(counts)[:-1]])
    host_pts = rng.standard_normal((int(counts.sum()), C), dtype=np.float32)
    padded = np.zeros((host_pts.shape[0], 16), np.float32)  # SuperpointStore's device layout
    padded[:, :C] = host_pts
    pts = torch.from_numpy(padded).to(dev)
    del padded
    idx = (rng.random((nv, L)) * counts[:, None]).astype(np.int32)
    cols = attrib_columns("xyzrgbelpsvXYZ", C)
    F = len(cols)
    t_idx = torch.from_numpy(idx).to(dev)
    t_start = torch.from_numpy(starts.astype(np.int64)).to(dev)
    t_count = torch.from_numpy(counts.astype(np.int32)).to(dev)
    t_cols = torch.tensor(cols, dtype=torch.int32, device=dev)
    clouds = torch.empty((nv, F, L), dtype=torch.float32, device=dev)
    diam = torch.empty(nv, dtype=torch.float32, device=dev)

    def fn():
        ops.cloud_build(pts, t_start, t_count, t_idx, t_cols, L, True, None, None, 0.0, 0.05, 0, clouds, diam)

    for _ in range(3):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
    for s_, e_ in ev:
        s_.record()
        fn()
        e_.record()
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)[len(ev) // 2]
    nbytes = nv * L * (2 * F * 4 + 4)
    gbs = nbytes / (ms * 1e-3) / 1e9
    out = {"kernel": "cloud_build", "bound": "hbm", "superpoints": nv, "points_resident": int(counts.sum()),
           "ms": ms, "bytes": nbytes, "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s",
           "frac": gbs / pk["hbm"], "traffic": None, "gpu_superpoints_per_s": nv / (ms * 1e-3)}
    tr = ncu_traffic().get("cloud_build")
    if tr:
        out["traffic"] = tr["bytes_per_launch"]
        out["traffic_note"] = "ncu --set full, %s (%s)" % (tr["launch"], tr["source"])
    if with_cpu:
        from oracle import loader_ref  # CPU baseline leg only
        n_cpu = 2000
        t0 = time.perf_counter()
        for i in range(n_cpu):
            P = host_pts[starts[i]:starts[i] + counts[i]]
            loader_ref.load_superpoint(P, idx[i], "xyzrgbelpsvXYZ", 1)
        dt = time.perf_counter() - t0
        out["cpu_superpoints_per_s"] = n_cpu / dt
        out["cpu_sample"] = "%d of the same superpoints, oracle port of load_superpoint, 1 thread (numpy)" % n_cpu
    return out


DUMP_BYTES = 64 * 10 ** 6


def host_outputs(loss, logits):
    """A step's (loss, logits) as float32 host arrays, copied now: a replayed graph reuses its output buffers."""
    out = {"logits": logits.detach().float().cpu().numpy()}
    if loss is not None:
        out["loss"] = loss.detach().float().reshape(-1).cpu().numpy()
    return out


def dump_outputs(path, arrays, budget=DUMP_BYTES):
    """Writes every array as path/<name>.npy.  Past `budget` bytes in all, logits keeps a fixed seeded
    sample of its rows, whose indices go to logits_rows.npy (float64)."""
    arrays = dict(arrays)
    lg = arrays["logits"]
    rest = sum(a.nbytes + 128 for k, a in arrays.items() if k != "logits") + 2 * 128  # + .npy headers
    if rest + lg.nbytes > budget:
        keep = (budget - rest) // (lg.shape[1] * lg.itemsize + 8)
        rows = np.sort(np.random.default_rng(0).choice(lg.shape[0], keep, replace=False))
        arrays["logits"], arrays["logits_rows"] = lg[rows], rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_b200(args):
    import torch.distributed as dist

    from superpoint_graph_b200 import _lib, ops, workloads
    from superpoint_graph_b200.spg_pointnet import CloudEmbedder
    from superpoint_graph_b200.trainer import HostBatch, Trainer, create_model

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback")
    _lib.lib()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    pk = peaks()

    w = workloads.get(args.workload, args.nodes)
    margs, train = w["margs"], w["train"]
    torch.manual_seed(1)  # --seed 1 (main.py:77); Trainer also broadcasts rank 0's parameters once
    model = create_model(margs)
    sd_ecc = {k: v.clone() for k, v in model.ecc.state_dict().items()}
    sd_ptn = {k: v.clone() for k, v in model.ptn.state_dict().items()}
    model.to(dev)
    trainer = Trainer(model, margs, process_group=pg, world_size=world, dtype=w["dtype"])

    # 4 distinct batches per rank, rotated; rank-offset seeds (scene-parallel)
    nb = 4 if w["nodes"] <= 20000 else (2 if w["nodes"] <= 50000 else 1)  # a 100k-superpoint step keeps ~45 GB of activations
    batches = [workloads.batch(w, 1 + 1000 * rank + i) for i in range(nb)]
    hbs = [HostBatch(b) for b in batches]
    counts = workload_counts(batches[0])
    units = [workload_counts(b)["edges"] + workload_counts(b)["points"] for b in batches]
    dbs = [hb.to_device(dev) for hb in hbs]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def step(db):
        if train:
            return trainer.train_step(db)
        return None, trainer.eval_step(db)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- self-check: the very first step from the initial state against the CPU arm (rank 0)
    parity = None
    loss0, logits0 = step(dbs[0])
    torch.cuda.synchronize()
    if rank == 0 and not args.no_parity:
        if w["nodes"] <= 4096:
            parity = parity_check(w, batches[0], sd_ecc, sd_ptn, None if loss0 is None else float(loss0[0]), logits0)
        else:
            parity = {"skipped": "CPU step at %d superpoints exceeds the bench's time bound; this shape is "
                                 "covered by tests/test_gpu_shapes.py" % w["nodes"]}

    # ---- device-resident timing (value)
    for i in range(args.warmup):
        step(dbs[i % nb])
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = ops.total_launches()
    evs = []
    done_units = 0
    t_wall = time.perf_counter()
    for i in range(args.steps):
        flush.zero_()  # L2 flush, outside the event bracket
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = step(dbs[i % nb])
        e.record()
        evs.append((s, e))
        done_units += units[i % nb]
    barrier()
    wall = time.perf_counter() - t_wall
    clocks = sampler.stop()
    last = host_outputs(*out) if args.dump_outputs else None
    launches = ops.total_launches() - launches0
    total_ms = sum(s.elapsed_time(e) for s, e in evs)
    tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    uu = torch.tensor([float(done_units)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(uu, op=dist.ReduceOp.SUM)
    total_ms, all_units = float(tt), float(uu)
    value = all_units / (total_ms * 1e-3)

    eager_ms, eager_value = total_ms / args.steps, value
    # ---- same K steps replayed from CUDA graphs (one per distinct batch shape): identical kernels,
    # one graph launch per step instead of ~100 kernel launches
    graph_keys, graph_err = None, None
    if not args.no_graph and train and w["nodes"] <= 50000:  # (a captured graph pins its activations)
        try:
            per_step0 = ops.total_launches()
            graph_keys = [trainer.capture(dbs[i], key=i, warmup=1) for i in range(nb)]
            launches_per_step = (ops.total_launches() - per_step0) // (2 * nb) + 1  # (1 warm-up + 1 capture) x nb
            for i in range(args.warmup):
                trainer.replay(graph_keys[i % nb])
            barrier()
            sampler = ClockSampler(local)
            sampler.start()
            evs, done_units = [], 0
            t_wall = time.perf_counter()
            for i in range(args.steps):
                flush.zero_()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                out = trainer.replay(graph_keys[i % nb])
                e.record()
                evs.append((s, e))
                done_units += units[i % nb]
            barrier()
            wall = time.perf_counter() - t_wall
            clocks = sampler.stop()
            launches = launches_per_step * args.steps
            total_ms = sum(s.elapsed_time(e) for s, e in evs)
            tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
            uu = torch.tensor([float(done_units)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dist.all_reduce(uu, op=dist.ReduceOp.SUM)
            total_ms, all_units = float(tt), float(uu)
            value = all_units / (total_ms * 1e-3)
            if args.dump_outputs:
                last = host_outputs(*out)
        except Exception as ex:  # keep the eager numbers
            graph_keys, graph_err = None, repr(ex)
    eval_keys = None
    if not args.no_graph and not train and w["nodes"] <= 50000:
        # inference: the same forward replayed from a CUDA graph (the eager forward is issue-bound on the host
        # at these sizes)
        try:
            per_step0 = ops.total_launches()
            eval_keys = [trainer.capture_eval(dbs[i], key=i, warmup=1) for i in range(nb)]
            launches_per_step = (ops.total_launches() - per_step0) // (2 * nb)
            for i in range(args.warmup):
                trainer.replay_eval(eval_keys[i % nb])
            barrier()
            sampler = ClockSampler(local)
            sampler.start()
            evs, done_units = [], 0
            t_wall = time.perf_counter()
            for i in range(args.steps):
                flush.zero_()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                out = None, trainer.replay_eval(eval_keys[i % nb])
                e.record()
                evs.append((s, e))
                done_units += units[i % nb]
            barrier()
            wall = time.perf_counter() - t_wall
            clocks = sampler.stop()
            launches = launches_per_step * args.steps
            total_ms = sum(s.elapsed_time(e) for s, e in evs)
            tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
            uu = torch.tensor([float(done_units)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dist.all_reduce(uu, op=dist.ReduceOp.SUM)
            total_ms, all_units = float(tt), float(uu)
            value = all_units / (total_ms * 1e-3)
            if args.dump_outputs:
                last = host_outputs(*out)
        except Exception as ex:  # keep the eager numbers
            eval_keys, graph_err = None, repr(ex)

    # ---- end-to-end through the public API with host buffers (H2D + step + D2H of loss/logits)
    h2d = hbs[0].h2d_bytes()
    out_host = torch.empty((w["nodes"], margs.classes), dtype=torch.float32).pin_memory()
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()

    def e2e_step(i):
        if graph_keys is not None:  # refresh the graph's static input buffers, then replay
            hbs[i % nb].copy_into(dbs[i % nb])
            return trainer.replay(graph_keys[i % nb])
        if not train:
            hb = hbs[i % nb]
            if eval_keys is not None and hb.clouds.numel() * 4 < CloudEmbedder.PIPELINE_MIN_BYTES:
                hb.copy_into(dbs[i % nb])  # small batch: refresh the graph's static inputs, replay
                return None, trainer.replay_eval(eval_keys[i % nb])
            return None, trainer.eval_step_host(hb)  # large: chunked upload overlapped with the forward
        return step(hbs[i % nb].to_device(dev))

    for i in range(0 if args.no_e2e else max(3, args.warmup // 2)):
        e2e_step(i)
    barrier()
    e2e_ms, e2e_units = 1e-9, 0
    for i in range(0 if args.no_e2e else args.steps):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        loss, logits = e2e_step(i)
        out_host[:logits.shape[0]].copy_(logits, non_blocking=True)
        if loss is not None:
            loss_host.copy_(loss, non_blocking=True)
        e.record()
        e.synchronize()  # the trainer reads loss/logits on the host every step (main.py:216-221)
        e2e_ms += s.elapsed_time(e)
        e2e_units += units[i % nb]
    barrier()
    t2 = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    u2 = torch.tensor([float(e2e_units)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        dist.all_reduce(u2, op=dist.ReduceOp.SUM)
    e2e_value = float(u2) / (float(t2) * 1e-3)
    d2h = int(w["nodes"] * margs.classes * 4 + (4 if train else 0))

    line = {
        "metric": METRIC if train else METRIC_EVAL, "value": value, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
        "config": config_of(w, counts, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": float(t2) / args.steps},
        "rates": rates(counts, world, total_ms / args.steps),
        "gpu_launches": int(launches),
        "cuda_graph": graph_keys is not None or eval_keys is not None,
        "eager": {"ms_per_step": eager_ms, "value": eager_value},
        "wall_ms_per_step_incl_flush": wall * 1e3 / args.steps,
        "clocks": clocks,
        "peaks": pk["source"],
    }
    if parity is not None:
        line["parity_rel_err"] = parity

    if graph_err:
        line["cuda_graph_error"] = graph_err
    if rank == 0 and not args.no_roofline:
        # per-kernel shares of the step (events around every launch; separate, untimed pass)
        ops.prof_reset()
        ops.prof_enable(1)
        flops0 = {"gemm_f32": ops.GEMM_FLOPS[0] - ops.TC_FLOPS[0] - ops.DW_FLOPS[0],
                  "tc_gemm_3xtf32": ops.TC_FLOPS[0], "tc_dw_3xtf32": ops.DW_FLOPS[0],
                  "pointnet_fused_eval": ops.FUSED_FLOPS[0]}
        nprof = 3
        for i in range(nprof):
            step(dbs[i % nb]) if world == 1 else None
        torch.cuda.synchronize()
        ops.prof_enable(0)
        if world == 1:
            ks = ops.prof_collect()
            tot = sum(v[1] for v in ks.values())
            top = sorted(ks.items(), key=lambda kv: -kv[1][1])
            line["kernel_shares"] = {k: {"launches_per_step": v[0] / nprof, "ms_per_step": v[1] / nprof,
                                         "share": v[1] / tot} for k, v in top[:12]}
            flops1 = {"gemm_f32": ops.GEMM_FLOPS[0] - ops.TC_FLOPS[0] - ops.DW_FLOPS[0],
                      "tc_gemm_3xtf32": ops.TC_FLOPS[0], "tc_dw_3xtf32": ops.DW_FLOPS[0],
                      "pointnet_fused_eval": ops.FUSED_FLOPS[0]}
            notes = {"gemm_f32": "exact-fp32 FMA GEMM (small/odd shapes), measured against the bf16 tensor peak",
                     "tc_gemm_3xtf32": "tcgen05 kind::tf32, 3 MMAs per product (error-compensated split, fp32-"
                                       "equivalent): algorithmic FLOPs counted once; ceiling = bf16 peak / 6",
                     "tc_dw_3xtf32": "tcgen05 kind::tf32 MN-major operands, 3 MMAs per product; ceiling = bf16 peak / 6",
                     "pointnet_fused_eval": ("fused eval trunk, tcgen05 kind::f16 on bf16 operands: ceiling = bf16 peak"
                                             if w["dtype"] == "bf16" else
                                             "fused eval trunk, tcgen05 kind::tf32, 3 MMAs per product (fp32-equivalent): "
                                             "algorithmic FLOPs counted once; ceiling = bf16 peak / 6")}
            dense = {}
            for name in ("tc_gemm_3xtf32", "tc_dw_3xtf32", "gemm_f32", "pointnet_fused_eval"):
                if name in ks and ks[name][1] > 0:
                    ach = (flops1[name] - flops0[name]) / (ks[name][1] * 1e-3) / 1e12
                    dense[name] = {"kernel": name, "bound": "tensor", "achieved": ach, "peak": pk["bf16_sustained"],
                                   "unit": "TFLOP/s", "frac": ach / pk["bf16_sustained"], "traffic": None,
                                   "share_of_step": ks[name][1] / tot, "note": notes[name]}
            for name, obj in dense.items():
                tr = ncu_traffic().get(name)
                if name == "pointnet_fused_eval" and w["dtype"] == "bf16":
                    tr = None  # the committed ncu capture is of the fp32 (3xTF32) variant
                if tr:
                    obj["traffic"] = tr["bytes_per_launch"]
                    obj["traffic_note"] = "ncu --set full, %s (%s); algorithmic %.4g B" % (
                        tr["launch"], tr["source"], tr["algorithmic_bytes"])
            gname = top[0][0]
            if gname in dense:
                line["roofline"] = dense[gname]
            line["roofline_dense_kernels"] = dense
        extras = args.workload == "s3dis_train"  # the component rooflines ride on the headline line only
        try:
            if not extras:
                raise StopIteration
            er = ecc_roofline(dev, args.ecc_nodes, pk, flush)
            line["roofline_ecc"] = er
            k = er["kernels"]["mat_fwd"]
            ecc_obj = {"kernel": "ecc_mat_fwd", "bound": "hbm", "achieved": k["gbs"], "peak": pk["hbm"],
                       "unit": "GB/s", "frac": k["frac"], "traffic": None,
                       "workload": "configs[4]-scale: %d superpoints, %d edges, [E,32,32] filters" % (er["nodes"], er["edges"])}
            tr = ncu_traffic().get("ecc_mat_fwd")
            if tr and tr.get("nodes") == er["nodes"]:
                ecc_obj["traffic"] = tr["bytes_per_launch"]
                ecc_obj["traffic_note"] = "ncu --set full, %s (%s); algorithmic %.4g B" % (
                    tr["launch"], tr["source"], tr["algorithmic_bytes"])
            if "roofline" not in line:
                line["roofline"] = ecc_obj
            else:
                line["roofline_ecc_scatter"] = ecc_obj
            kv = er["kernels"]["vv_fwd"]
            line["roofline_ecc_scatter_vv"] = {
                "kernel": "ecc_vv_fwd", "bound": "hbm", "achieved": kv["gbs"], "peak": pk["hbm"],
                "unit": "GB/s", "frac": kv["frac"], "traffic": (ncu_traffic().get("ecc_vv_fwd") or {}).get("bytes_per_launch"),
                "workload": "configs[1]/[4] filter mode (vector filters [E,32]): %d superpoints, %d edges, L2 flushed "
                            "before every launch" % (er["nodes"], er["edges"])}
        except StopIteration:
            pass
        except Exception as ex:  # keep the bench line even if the microbench cannot run
            line["roofline_ecc_error"] = repr(ex)
        try:
            if not extras:
                raise StopIteration
            line["roofline_loader"] = loader_roofline(dev, pk, not args.no_cpu_baseline)
        except StopIteration:
            pass
        except Exception as ex:
            line["roofline_loader_error"] = repr(ex)

    if rank == 0 and world == 1 and args.trace_gemm:
        ops.GEMM_TRACE = []
        step(dbs[0])
        torch.cuda.synchronize()
        agg = {}
        for desc, e0, e1 in ops.GEMM_TRACE:
            a = agg.setdefault(desc, [0, 0.0])
            a[0] += 1
            a[1] += e0.elapsed_time(e1)
        ops.GEMM_TRACE = None
        for desc, (n, ms) in sorted(agg.items(), key=lambda kv: -kv[1][1])[:25]:
            print("[gemm_f32] %-40s x%d  %.3f ms" % (desc, n, ms), file=sys.stderr)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(w, sd_ecc, sd_ptn)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
