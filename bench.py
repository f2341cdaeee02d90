#!/usr/bin/env python
"""bench.py — keyframe-BA-updates/s (+ rendered Mrays/s) on synthetic GO-SLAM workloads.

Workload (BASELINE.json configs[1]): Replica room0 RGB-D shapes — 8-keyframe local window,
1/8-resolution 40x80, 36 edges (|i-j| <= 3).  One STEP = one keyframe-BA-update:
    all-pairs correlation build + 4-level pyramid for the window's 36 edges (tcgen05)
  + reprojection of every edge
  + fused 4-level radius-3 lookup
  + dense bundle adjustment, 3 Gauss-Newton iterations (RGB-D prior on)
`value` is measured with inputs resident in HBM; `e2e` runs the same step through the public
Python API from pinned HOST buffers (H2D of the step's inputs and D2H of the updated state
inside the timed region).  The renderer (2^18-ray batches x 72 samples through the fused
marcher) is reported in the same line under "render".

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
N > 1: one rank per GPU under torchrun; every rank owns an independent keyframe window and
ray batch (weak scaling, no data-path collective — SURVEY §8e), time = max over ranks.
--dump-outputs DIR writes the updated poses / inverse depths and the lookup features of the last
timed step as DIR/<name>.npy (float32); inputs are seeded, so two builds can be compared on them.
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

NUM_KF, HT, WD, BA_ITERS = 8, 40, 80, 3
RAYS, SAMPLES = 1 << 18, 72
METRIC = "keyframe-BA-updates/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML (nvidia_ml_py) in a thread at
    ~1 kHz (the timed region of the default run is ~10 ms), falling back to nvidia-smi polling."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.stop, self.max_mhz = index, [], False, None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        if self.nvml is not None:
            nv = self.nvml
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                    "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self.stop:
                try:
                    mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    r = int(get_reasons(self.h))
                    self.samples.append([mhz, self.max_mhz] + [("Active" if (r & m) else "Not Active") for m in bits.values()])
                except Exception:
                    pass
                time.sleep(0.001)
            return
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.05)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(str(s[2 + i]).lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------ workload
def make_window(seed, ht=None, wd=None, num_kf=None):
    from goslam_b200 import synthetic
    ht, wd, num_kf = ht or HT, wd or WD, num_kf or NUM_KF
    sc, g = synthetic.make_scene(num_kf=num_kf, ht=ht, wd=wd, seed=seed, rgbd=True)
    coords = synthetic.true_reprojection(sc)          # plain-torch setup helper (targets = reprojection + noise)
    targets, weights, eta = synthetic.make_update(sc, coords[0], g, noise=0.5)
    sc.update(targets=targets, weights=weights, eta=eta)
    return sc


class Window:
    """device-resident state of one 8-keyframe window + the public-API step."""

    def __init__(self, sc, dev):
        self.dev = dev
        self.num_kf, self.ht, self.wd = int(sc["num_kf"]), int(sc["ht"]), int(sc["wd"])
        self.host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in sc.items()}
        self.d = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in sc.items()}
        self.poses0 = self.d["poses"].clone()
        self.disps0 = self.d["disps"].clone()
        # the factor graph's correlation slot pool, allocated once (FactorGraph.max_factors slots)
        from goslam_b200.modules.corr import CorrPool
        self.pool = CorrPool(int(sc["ii"].numel()), self.ht, self.wd, device=dev, layout="tiled")
        self.corr = None

    def build(self, km):
        from goslam_b200.modules import CorrBlock
        if self.corr is not None:
            self.corr.free()                    # rm_factors: the slots go back to the pool
        self.corr = CorrBlock.from_video(km, self.d["ii"], self.d["jj"], self.ht, self.wd, pool=self.pool)
        return self.corr

    def step(self, reset=True):
        from goslam_b200 import droid_backends
        from goslam_b200.modules import CorrBlock
        from goslam_b200.modules.corr import fmaps_to_kmajor
        d = self.d
        if reset:                               # device-resident loop: restart from the same state every step
            d["poses"].copy_(self.poses0)       # (the end-to-end loop gets fresh inputs from the host instead)
            d["disps"].copy_(self.disps0)
        ii, jj = d["ii"], d["jj"]
        # FactorGraph.add_factors' volume, video-level: K-major re-layout of the window's feature
        # maps (per keyframe, redone every step here) + on-device edge -> frame indexing
        km = fmaps_to_kmajor(d["fmaps"][:self.num_kf])
        corr = self.build(km)
        coords, _ = droid_backends.reproject(d["poses"], d["disps"], d["intrinsics"], ii, jj, want_valid=False)
        feat = corr(coords)
        droid_backends.ba(d["poses"], d["disps"], d["intrinsics"][0], d["disps_sens"], d["targets"],
                          d["weights"], d["eta"], ii, jj, 1, self.num_kf, BA_ITERS, 1e-4, 0.1, False)
        d["disps"].clamp_(min=0.001)            # src/depth_video.py:269
        return feat

    E2E_KEYS = ("fmaps", "poses", "disps", "disps_sens", "intrinsics", "targets", "weights", "eta", "ii", "jj")

    def step_e2e(self, out_pinned):
        """one update through the public API from pinned HOST buffers: H2D of every input of the
        step, the step, D2H of the updated state.  Copies run on a side stream into the other half
        of a double buffer, so the transfer of update i+1 overlaps the kernels of update i (each
        step still waits for ITS inputs and its result is read back)."""
        if not hasattr(self, "_e2e"):
            # all inputs of a step live in ONE pinned host block and one device block per buffer half:
            # one H2D copy per step instead of ten (the end-to-end loop is otherwise host-bound)
            offs, total = {}, 0
            for k in self.E2E_KEYS:
                offs[k] = total
                total += (self.host[k].numel() * self.host[k].element_size() + 255) // 256 * 256
            packed = torch.empty(total, dtype=torch.uint8).pin_memory()

            def views(block):
                return {k: block[offs[k]:offs[k] + self.host[k].numel() * self.host[k].element_size()]
                        .view(self.host[k].dtype).view(self.host[k].shape) for k in self.E2E_KEYS}
            hv = views(packed)
            for k in self.E2E_KEYS:
                hv[k].copy_(self.host[k])
            self._e2e = dict(copy=torch.cuda.Stream(self.dev), bufs=[None, None], blocks=[None, None], packed=packed,
                             ready=[None, None], done=[None, None], parity=0, graphs=[None, None], graph_failed=False)
            for b in range(2):
                self._e2e["blocks"][b] = torch.empty(total, dtype=torch.uint8, device=self.dev)
                self._e2e["bufs"][b] = views(self._e2e["blocks"][b])
        st = self._e2e
        cur = st["parity"]
        main = torch.cuda.current_stream(self.dev)
        if st["ready"][cur] is None:                      # first call: nothing prefetched yet
            self._prefetch(cur)
        main.wait_event(st["ready"][cur])
        for k in self.E2E_KEYS:
            self.d[k] = st["bufs"][cur][k]
        self._prefetch(cur ^ 1)                           # next update's inputs, overlapped
        if st["graphs"][cur] is None and not st["graph_failed"]:
            st["graphs"][cur] = self._capture()           # the six launches of the step become one graph launch
            if st["graphs"][cur] is None:
                st["graph_failed"] = True
        if st["graphs"][cur] is not None:
            st["graphs"][cur].replay()
        else:
            self.step(reset=False)
        out_pinned[0].copy_(self.d["poses"], non_blocking=True)
        out_pinned[1].copy_(self.d["disps"], non_blocking=True)
        st["done"][cur] = torch.cuda.Event()
        st["done"][cur].record(main)
        st["parity"] = cur ^ 1

    @property
    def graphed(self):
        st = getattr(self, "_e2e", None)
        return bool(st and st["graphs"][0] is not None and st["graphs"][1] is not None)

    def _capture(self):
        """CUDA graph of one step on the CURRENT input buffers (self.d): kmajor, correlation build, reproject,
        lookup, BA table kernel, cooperative BA kernel — launched as one graph afterwards, which takes the host
        (Python + ctypes + driver) out of the critical path of the end-to-end loop."""
        try:
            side = torch.cuda.Stream(self.dev)
            side.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(side):
                self.step(reset=False)                    # warm-up off the capture: module load, workspaces, attributes
            torch.cuda.current_stream(self.dev).wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.step(reset=False)
            return g
        except Exception as e:   # noqa: BLE001 — e.g. a driver that cannot capture cooperative launches
            self.graph_error = "%s: %s" % (type(e).__name__, e)
            return None

    def _prefetch(self, b):
        st = self._e2e
        with torch.cuda.stream(st["copy"]):
            if st["done"][b] is not None:                 # buffer b must not be in use by an older step
                st["copy"].wait_event(st["done"][b])
            st["blocks"][b].copy_(st["packed"], non_blocking=True)
            st["ready"][b] = torch.cuda.Event()
            st["ready"][b].record(st["copy"])

    def h2d_bytes(self):
        return sum(self.host[k].numel() * self.host[k].element_size() for k in
                   ("fmaps", "poses", "disps", "disps_sens", "intrinsics", "targets", "weights", "eta", "ii", "jj"))

    def d2h_bytes(self):
        return self.d["poses"].numel() * 4 + self.d["disps"].numel() * 4


def make_renderer(dev, seed):
    from goslam_b200 import neus, synthetic
    offs, ress, _, total = neus.hashgrid_layout()
    w = synthetic.make_neus_weights(seed=seed, total_grid_params=total, layout=(offs, ress))
    net = neus.InstantNeuS(synthetic.NEUS_CFG, [[-2.0, 2.0]] * 3)
    with torch.no_grad():
        net.sdf_network.encoding.encoding.params.copy_(w["grid"])
        net.sdf_network.sdf_layer.weight.copy_(w["sdf_w"])
        net.sdf_network.sdf_layer.bias.copy_(w["sdf_b"])
        net.color_network._B.copy_(w["color_B"])
        net.color_network.network.params.copy_(w["mlp"])
    net = net.to(dev)
    rays = synthetic.make_rays(RAYS, S=SAMPLES, seed=seed)
    return net, rays, w


def time_gpu(fn, steps, warmup, dist_barrier):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    dist_barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    dist_barrier()
    return e0.elapsed_time(e1) / steps          # ms per step


def max_over_ranks(x, world):
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ------------------------------------------------------------------------------------ CPU arm
def cpu_reference_step(sc, n_corr_edges=4, ba_iters=1):
    """Reference algorithm on the host cores (oracle port): correlation build + pyramid + lookup
    on `n_corr_edges` of the 36 edges and `ba_iters` BA iteration(s) on the full graph; returns
    the time extrapolated to the full step (36 edges, 3 iterations)."""
    from oracle import ba_oracle, corr_oracle, geom_oracle
    ii, jj = sc["ii"], sc["jj"]
    N = ii.numel()
    t0 = time.perf_counter()
    pyr = corr_oracle.corr_build(sc["fmaps"][ii[:n_corr_edges], 0].float(), sc["fmaps"][jj[:n_corr_edges], 0].float(), 4)
    coords, _ = geom_oracle.reproject(sc["poses"].numpy(), sc["disps"].numpy(), sc["intrinsics"].numpy(),
                                      ii[:n_corr_edges].numpy(), jj[:n_corr_edges].numpy())
    corr_oracle.corr_pyramid_lookup([p.numpy() for p in pyr], coords[0], 3)
    t1 = time.perf_counter()
    ba_oracle.ba(sc["poses"].numpy(), sc["disps"].numpy(), sc["intrinsics"][0].numpy(), sc["disps_sens"].numpy(),
                 sc["targets"].numpy(), sc["weights"].numpy(), sc["eta"].numpy(), ii.numpy(), jj.numpy(),
                 1, NUM_KF, ba_iters, 1e-4, 0.1, False)
    t2 = time.perf_counter()
    full = (t1 - t0) * N / n_corr_edges + (t2 - t1) * BA_ITERS / ba_iters
    return full, (t2 - t0)


def cpu_sample_plan(sc, budget_s):
    """(edges, BA iterations) of the CPU sample: the whole step when it fits `budget_s` seconds on this
    host, otherwise as many of the 36 edges (+ 1 of the 3 iterations) as fit; probed warm."""
    cpu_reference_step(sc, 2, 1)                     # thread pools, allocator
    est_full, _ = cpu_reference_step(sc, 2, 1)
    if est_full <= budget_s:
        return 36, BA_ITERS
    return max(2, int(36 * budget_s / est_full)), 1


def run_reference(args, rank, world):
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    sc = make_window(43)
    n_e, n_it = cpu_sample_plan(sc, 150.0 / max(1, args.steps + args.warmup))
    for _ in range(max(args.warmup, 0)):
        cpu_reference_step(sc, n_e, n_it)
    ts = []
    for _ in range(args.steps):
        full, _ = cpu_reference_step(sc, n_e, n_it)
        ts.append(full)
    ms = 1e3 * float(np.mean(ts))
    val = 1e3 / ms                # the host's cores are the same whatever N is: its N windows run one after another
    sample = ("per step: corr build+pyramid+lookup on %d/36 edges and %d/3 BA iterations (numpy/torch CPU port of the "
              "reference kernels)%s" % (n_e, n_it, "" if n_e == 36 else ", extrapolated linearly to the full step"))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "updates/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "cpu_baseline": {"value": val, "unit": "updates/s", "cores": os.cpu_count(), "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(world):
    return {"workload": "configs[1]: Replica room0 RGB-D shapes, 8-keyframe window, 40x80 @1/8, 36 edges, "
                        "corr build + 4-level r=3 lookup + 3 BA iters per update",
            "keyframes": NUM_KF, "grid": [HT, WD], "edges": 36, "ba_iters": BA_ITERS,
            "windows_per_gpu": 1,
            "parallelism": "value / e2e / headline_640x480 / render: one window + one ray batch per GPU x%d, no collective "
                           "(weak scaling); sharded_graph: ONE graph over all ranks, NCCL all-reduce + all-gather per BA "
                           "iteration (strong scaling)" % world,
            "l2": "each step writes a 0.98 GB correlation pyramid (> 126 MB L2) before it is read back, no explicit flush needed",
            "corr_layout": "tiled slot pool (CorrPool)",
            "render": {"rays": RAYS, "samples_per_ray": SAMPLES}}


# ------------------------------------------------------------------------------------ legs
def build_roofline(win, pk, steps, warm, ms_step):
    """the dominant kernel (tcgen05 correlation build) timed alone on this stream, against the measured HBM peak"""
    from goslam_b200.modules.corr import fmaps_to_kmajor
    d = win.d
    km = fmaps_to_kmajor(d["fmaps"][:win.num_kf])
    ms_build = time_gpu(lambda: win.build(km), max(steps, 10), warm, lambda: None)
    N, hw = int(d["ii"].numel()), win.ht * win.wd
    lvl = sum((win.ht >> i) * (win.wd >> i) for i in range(4))
    build_bytes = N * (2 * 128 * hw * 2 + hw * lvl * 2)
    build_flops = N * 2.0 * 128 * hw * hw
    ach = build_bytes / (ms_build * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tp):      # dram__bytes_read+write of the `ncu --set full` capture of this kernel on this workload
        traffic = json.load(open(tp)).get("corr_build_tc_staged_kernel@%dx%d" % (win.ht, win.wd), {}).get("dram_bytes_per_launch")
    return {"kernel": "corr_build_tc_staged_kernel", "bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s",
            "frac": ach / pk["hbm"], "traffic": traffic, "algorithmic_bytes": build_bytes,
            "peak_source": pk["src"] + " (burst copy bandwidth)", "ms_per_launch": ms_build,
            "share_of_step": ms_build / ms_step, "tensor_tflops": build_flops / (ms_build * 1e-3) / 1e12,
            "tensor_frac_of_measured_burst": build_flops / (ms_build * 1e-3) / 1e12 / pk["tf_burst"]}


def stereo_build_leg(dev, rank, steps, warm, pk):
    """configs[4] shapes (EuRoC stereo, 40x60 @1/8, rig = 2): the correlation build + 4-level lookup of a 36-edge graph that
    includes the 8 left-right self-edges (ii == jj reads the second camera's features, src/factor_graph.py:108-112)"""
    from goslam_b200.modules import CorrBlock
    from goslam_b200.modules.corr import CorrPool, fmaps_to_kmajor
    ht, wd, nkf = 40, 60, 8
    g = torch.Generator().manual_seed(77 + rank)
    fm = torch.randn(nkf, 2, 128, ht, wd, generator=g).half().to(dev)
    km = fmaps_to_kmajor(fm)
    ii = torch.cat([torch.arange(nkf), torch.arange(28) % nkf]).to(dev)
    jj = torch.cat([torch.arange(nkf), (torch.arange(28) % nkf + 1 + torch.arange(28) // nkf) % nkf]).to(dev)
    N = int(ii.numel())
    pool = CorrPool(N, ht, wd, device=dev)
    coords = (torch.stack(torch.meshgrid(torch.arange(wd), torch.arange(ht), indexing="xy"), dim=-1).float()[None, None]
              .expand(1, N, ht, wd, 2).contiguous().to(dev) + 1.7)
    blk = [None]

    def build():
        if blk[0] is not None:
            blk[0].free()
        blk[0] = CorrBlock.from_video(km, ii, jj, ht, wd, rig=2, pool=pool)

    build()
    ms_l = time_gpu(lambda: blk[0](coords), max(steps, 10), warm, lambda: None)
    ms_b = time_gpu(build, max(steps, 10), warm, lambda: None)
    hw = ht * wd
    lvl = sum((ht >> i) * (wd >> i) for i in range(4))
    bb = N * (2 * 128 * hw * 2 + hw * lvl * 2)
    lb = N * hw * 912
    return {"workload": "EuRoC stereo shapes 40x60 @1/8, rig 2, 36 edges incl. 8 self-edges (left-right)", "build_ms": ms_b,
            "build_roofline": {"kernel": "corr_build_tc_staged_kernel", "bound": "hbm", "achieved": bb / (ms_b * 1e-3) / 1e9,
                               "peak": pk["hbm"], "unit": "GB/s", "frac": bb / (ms_b * 1e-3) / 1e9 / pk["hbm"], "algorithmic_bytes": bb},
            "lookup_ms": ms_l,
            "lookup_roofline": {"kernel": "corr_lookup_kernel", "bound": "hbm", "achieved": lb / (ms_l * 1e-3) / 1e9, "peak": pk["hbm"],
                                "unit": "GB/s", "frac": lb / (ms_l * 1e-3) / 1e9 / pk["hbm"], "algorithmic_bytes": lb}}


DUMP_SAMPLE = 1 << 22          # elements kept of a dumped output larger than this (16 MB in float32)


def dump_outputs(out_dir, outputs):
    """out_dir/<name>.npy in float32 for each output; of one with more than DUMP_SAMPLE elements, the elements at a
    fixed seeded sample of flat indices (ascending), the same for every run with the same arguments"""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        a = t.detach().float().cpu().numpy().reshape(-1)
        if a.size > DUMP_SAMPLE:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a.reshape(t.shape) if a.size == t.numel() else a)


def window_leg(sc, dev, steps, warm, barrier, world, pk, clock_index=None, dump_dir=None):
    """device-resident + end-to-end timing of the keyframe-BA-update on one window shape; with dump_dir, what the
    last timed step computed (BA poses and inverse depths, lookup features) is written there"""
    win = Window(sc, dev)
    last = {}

    def step():
        last["corr"] = win.step()

    if clock_index is not None:
        with ClockSampler(clock_index) as clk:
            ms_step = time_gpu(step, steps, warm, barrier)
        clocks = clk.summary()
    else:
        ms_step, clocks = time_gpu(step, steps, warm, barrier), None
    if dump_dir is not None:
        dump_outputs(dump_dir, {"poses": win.d["poses"], "disps": win.d["disps"], "corr": last["corr"]})
    ms_step = max_over_ranks(ms_step, world)
    outp = (torch.empty_like(sc["poses"]).pin_memory(), torch.empty_like(sc["disps"]).pin_memory())
    ms_e2e = max_over_ranks(time_gpu(lambda: win.step_e2e(outp), steps, warm, barrier), world)
    graphed = win.graphed
    roof = build_roofline(win, pk, steps, warm, ms_step)
    rec = {"value": world * 1e3 / ms_step, "unit": "updates/s", "ms_per_step": ms_step,
           "e2e": {"value": world * 1e3 / ms_e2e, "unit": "updates/s", "ms_per_step": ms_e2e,
                   "h2d_bytes_per_step": win.h2d_bytes(), "d2h_bytes_per_step": win.d2h_bytes(),
                   "cuda_graph": graphed},
           "roofline": roof}
    return rec, clocks


def sharded_graph_leg(dev, steps, warm, barrier, world, rank):
    """configs[3]: ONE 64-keyframe global-BA graph (ScanNet shapes, 30x40) sharded over the ranks by source
    frame — per update: reproject + motion features + 4-level windowed correlation of the local edges, then 2
    BA iterations with one all-reduce of the reduced camera system and one all-gather of the owned inverse-
    depth rows each.  Strong scaling: the graph is the same whatever N is."""
    import torch.distributed as dist
    from goslam_b200 import droid_backends, graph, parallel, synthetic
    num_kf, ht, wd, iters = 64, 30, 40, 2
    sc, g = synthetic.make_scene(num_kf=num_kf, ht=ht, wd=wd, seed=43, rgbd=True, buffer=num_kf + 2)
    D = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in sc.items()}
    # Backend.ba's edge rule (src/backend.py:25-99, radius 1, nms 5, thresh 25, max_factors 6*64), on the device
    ix = torch.arange(0, num_kf)
    gi, gj = torch.meshgrid(ix, ix, indexing="ij")
    dmat = droid_backends.frame_distance_bidirectional(D["poses"], D["disps"], D["intrinsics"][0].contiguous(),
                                                       gi.reshape(-1).to(dev), gj.reshape(-1).to(dev), 0.3)
    ii, jj = graph.backend_edges(dmat, 0, num_kf, 1, 5, 25.0, 384, False)
    sc["ii"], sc["jj"] = ii.cpu(), jj.cpu()
    sc["t0"], sc["t1"] = 1, num_kf
    coords = synthetic.true_reprojection(sc)
    tg, wg, eta = synthetic.make_update(sc, coords[0], g, noise=0.5)
    kx = torch.unique(torch.cat([torch.arange(1, num_kf), sc["ii"]]))
    eta_f = torch.zeros(num_kf + 2, ht, wd)
    eta_f[kx] = eta
    eta_f = eta_f.to(dev)
    group = None
    if world == 1 and not dist.is_initialized():
        # single process: a one-rank gloo group keeps the code path identical (no collective is issued)
        dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)
        own_group = True
    else:
        own_group = False
    p0, d0 = D["poses"].clone(), D["disps"].clone()
    res = {}
    errors = {}
    for exchange in (("nccl", "peer") if world > 1 else ("nccl",)):
        D["poses"].copy_(p0)
        try:
            sg = parallel.ShardedGraph(D["poses"], d0.clone(), D["intrinsics"], D["disps_sens"], D["fmaps"], ii, jj, 1, num_kf,
                                       group=group, exchange=exchange)
            ok_here = torch.ones(1, device=dev)
        except Exception as exc:          # e.g. no peer access between two GPUs of the box: keep the NCCL number
            errors[exchange] = repr(exc)[:200]
            ok_here = torch.zeros(1, device=dev)
        if world > 1:                     # all ranks take the same branch
            dist.all_reduce(ok_here, op=dist.ReduceOp.MIN)
        if ok_here.item() == 0:
            errors.setdefault(exchange, "setup failed on another rank")
            continue
        tg_l, wg_l = sg.local(tg.to(dev)), sg.local(wg.to(dev))                      # planar [n,2,h,w]
        tgt_flow = sg.local(tg.permute(0, 2, 3, 1).contiguous().to(dev))            # [n,h,w,2] for the motion features

        def update():
            if sg.link is not None:
                sg.link.wait_idle()              # the peers' last rows have landed before the replica is reset
            sg.poses.copy_(p0)
            sg.disps.copy_(d0)
            sg.features(tgt_flow)
            sg.bundle_adjust(tg_l, wg_l, eta_f, iters, 1e-5, 1e-2)

        ms_x = max_over_ranks(time_gpu(update, steps, warm, barrier), world)
        if sg.link is not None:
            sg.link.wait_idle()
        torch.cuda.synchronize()
        # replicas must agree bit for bit after the update (every rank solved the same summed system)
        agree_x = True
        if world > 1:
            for t in (sg.poses, sg.disps):
                ref = t.clone()
                dist.broadcast(ref, src=0)
                flag = torch.tensor([float(torch.equal(ref, t))], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                agree_x = agree_x and bool(flag.item() == 1.0)
        res[exchange] = {"ms_per_update": ms_x, "replicas_bit_identical": agree_x, "poses": sg.poses.clone(),
                         "timeout": bool(sg.link.timeout.item()) if sg.link is not None else False}
        if sg.link is not None:
            sg.link.close()
    best = min(res, key=lambda k: res[k]["ms_per_update"])
    ms, agree = res[best]["ms_per_update"], all(r["replicas_bit_identical"] for r in res.values())
    exchanges = {k: {"ms_per_update": r["ms_per_update"], "replicas_bit_identical": r["replicas_bit_identical"]} for k, r in res.items()}
    for k, v in errors.items():
        exchanges[k] = {"error": v}
    if "peer" in res:
        exchanges["peer"]["max_abs_pose_diff_vs_nccl"] = float((res["peer"]["poses"] - res["nccl"]["poses"]).abs().max())
        exchanges["peer"]["wait_timed_out"] = res["peer"]["timeout"]
    if own_group:
        dist.destroy_process_group()
    P = num_kf - 1
    return {"metric": "keyframe-BA-updates/s (one sharded graph)", "value": 1e3 / ms, "unit": "updates/s",
            "ms_per_update": ms, "scaling": "strong", "n_gpus": world,
            "workload": "configs[3]: 64-keyframe global BA graph, ScanNet 30x40 @1/8, %d edges (Backend.ba rule), "
                        "reproject + 4-level windowed correlation + 2 BA iters (lm 1e-5, ep 1e-2), P = %d poses" % (int(ii.numel()), P),
            "parallelism": "edges sharded by source frame over %d rank(s); per BA iteration 1 all-reduce of %d B "
                           "(reduced camera system, f64) + 1 all-gather of the owned inverse-depth rows" % (world, 8 * (36 * P * P + 6 * P)),
            "local_edges_rank0": int(sg.ii.numel()), "replicas_bit_identical": agree, "exchange": best,
            "exchanges": exchanges,
            "exchange_note": "nccl: all-reduce + all-gather per iteration; peer: the solve kernel sums the ranks' partial systems "
                             "out of peer memory while it loads the matrix, the back-substitution writes the owned rows into every "
                             "replica (goslam_ba_phase1_peers / goslam_ba_phase2_peers, CUDA IPC over NVLink, no collective)"}


def full_update_leg(dev, steps, warm, barrier, world, rank):
    """configs[2]-style front-end update THROUGH THE REFERENCE-FACING API: goslam_b200.FactorGraph.update on a
    goslam_b200.DepthVideo (Replica shapes: 8 keyframes, 40x80, 36 edges) with the update operator in the loop —
    reproject + motion features, 4-level lookup, UpdateModule (one library call: tcgen05 implicit-GEMM encoders, ConvGRU,
    heads, GraphAgg), 2 BA iterations, clamp.  Random-init weights of the reference architecture (no checkpoint travels to the box);
    graph state is restored before every update so that all steps see the same inputs."""
    import types
    from goslam_b200 import synthetic
    from goslam_b200.depth_video import DepthVideo
    from goslam_b200.droid_net import UpdateModule
    from goslam_b200.factor_graph import FactorGraph
    sc, g = synthetic.make_scene(num_kf=NUM_KF, ht=HT, wd=WD, seed=243 + rank, rgbd=True, buffer=NUM_KF + 2)
    cfg = {"cam": {"H_out": 8 * HT, "W_out": 8 * WD}, "mode": "rgbd", "tracking": {"buffer": NUM_KF + 2}}
    video = DepthVideo(cfg, types.SimpleNamespace(device=str(dev)))
    for k in ("poses", "disps", "disps_sens", "intrinsics", "fmaps"):
        getattr(video, k)[:] = sc[k].to(dev)
    video.nets[:] = (0.5 * torch.randn(NUM_KF + 2, 128, HT, WD, generator=g)).half().to(dev)
    video.inps[:] = (0.5 * torch.randn(NUM_KF + 2, 128, HT, WD, generator=g)).abs().half().to(dev)
    video.counter.value = NUM_KF
    torch.manual_seed(11)
    op = UpdateModule().to(dev).eval()
    with torch.no_grad():                                    # keep the random operator's flow corrections small
        for head in (op.delta[2], op.weight[2]):
            head.weight.mul_(0.05)
    graph = FactorGraph(video, op, device=str(dev), max_factors=48, upsample=False)
    graph.add_neighborhood_factors(0, NUM_KF, r=3)
    saved = dict(poses=video.poses.clone(), disps=video.disps.clone(), net=graph.net.clone(), target=graph.target.clone(),
                 weight=graph.weight.clone(), damping=graph.damping.clone())

    def update():
        video.poses.copy_(saved["poses"]); video.disps.copy_(saved["disps"]); graph.damping.copy_(saved["damping"])
        graph.net, graph.target, graph.weight = saved["net"].clone(), saved["target"].clone(), saved["weight"].clone()
        graph.update(1, NUM_KF, iters=2, use_inactive=False)

    ms = max_over_ranks(time_gpu(update, steps, warm, barrier), world)
    # the operator alone, and its ConvGRU against the same module evaluated by torch / cuDNN under autocast
    coords1, motion = graph._features(graph.ii, graph.jj, graph.target)
    corr = graph.corr(coords1)
    ms_op = time_gpu(lambda: op(graph.net, graph.inp, corr, motion, graph.ii, graph.jj), max(5, steps // 2), 3, lambda: None)
    gru = op.gru
    B = int(graph.ii.numel())

    def torch_update_op():
        """the reference UpdateModule.forward op for op (src/droid_net.py:107-140) in torch / cuDNN under autocast, on the
        same parameters: what `update_operator_ms` replaces"""
        with torch.no_grad(), torch.autocast("cuda", enabled=True):
            n_, i_, c_, f_ = [x.reshape(B, -1, HT, WD) for x in (graph.net, graph.inp, corr, motion)]
            c_, f_ = op.corr_encoder(c_), op.flow_encoder(f_)
            x = torch.cat([i_, c_, f_], dim=1)
            net_inp = torch.cat([n_, x], dim=1)
            glo = (torch.sigmoid(gru.w(n_)) * n_).view(B, 128, HT * WD).mean(dim=-1, keepdim=True).view(B, 128, 1, 1)
            z = torch.sigmoid(gru.convz(net_inp) + gru.convz_glo(glo))
            r = torch.sigmoid(gru.convr(net_inp) + gru.convr_glo(glo))
            q = torch.tanh(gru.convq(torch.cat([r * n_, x], dim=1)) + gru.convq_glo(glo))
            n2 = (1 - z) * n_ + z * q
            delta = op.delta(n2).view(1, B, -1, HT, WD).permute(0, 1, 3, 4, 2)[..., :2].contiguous()
            weight = op.weight(n2).view(1, B, -1, HT, WD).permute(0, 1, 3, 4, 2)[..., :2].contiguous()
            eta, upmask = op.agg(n2.view(1, B, 128, HT, WD), graph.ii)
            return n2, delta, weight, eta, upmask
    ms_op_torch = time_gpu(torch_update_op, max(5, steps // 2), 3, lambda: None)
    gi = [torch.randn(B, c, HT, WD, device=dev).half() for c in (128, 128, 128, 64)]

    def cudnn_gru():
        with torch.no_grad(), torch.autocast("cuda", enabled=True):
            net, x = gi[0], torch.cat(gi[1:], dim=1)
            net_inp = torch.cat([net, x], dim=1)
            glo = (torch.sigmoid(gru.w(net)) * net).view(B, 128, HT * WD).mean(dim=-1, keepdim=True).view(B, 128, 1, 1)
            z = torch.sigmoid(gru.convz(net_inp) + gru.convz_glo(glo))
            r = torch.sigmoid(gru.convr(net_inp) + gru.convr_glo(glo))
            q = torch.tanh(gru.convq(torch.cat([r * net, x], dim=1)) + gru.convq_glo(glo))
            return (1 - z) * net + z * q
    nh = [t.permute(0, 2, 3, 1).contiguous() for t in gi]
    ms_gru = time_gpu(lambda: gru.forward_nhwc(*nh), max(5, steps // 2), 3, lambda: None)
    ms_cudnn = time_gpu(cudnn_gru, max(5, steps // 2), 3, lambda: None)
    flops = 2.0 * B * HT * WD * (3 * 9 * 448 * 128 + 128 * 128)
    pk = peaks()
    return {"metric": "keyframe-BA-updates/s incl. the update operator", "value": world * 1e3 / ms, "unit": "updates/s",
            "ms_per_update": ms, "call": "goslam_b200.FactorGraph.update(t0=1, t1=8, iters=2) on goslam_b200.DepthVideo",
            "workload": "configs[2]-style front-end update: 8 keyframes, 40x80 @1/8, 36 edges, update operator (random-init "
                        "weights of the reference architecture) + lookup + 2 BA iterations",
            "update_operator_ms": ms_op, "update_operator_torch_cudnn_autocast_ms": ms_op_torch,
            "update_operator_speedup_vs_cudnn": ms_op_torch / ms_op,
            "conv_gru": {"kernel": "conv_tc_kernel x3 (tcgen05 implicit GEMM, fused gates)", "ms": ms_gru,
                         "tflops": flops / (ms_gru * 1e-3) / 1e12, "frac_of_measured_bf16_burst": flops / (ms_gru * 1e-3) / 1e12 / pk["tf_burst"],
                         "torch_cudnn_autocast_ms": ms_cudnn, "speedup_vs_cudnn": ms_cudnn / ms_gru, "bound": "tensor"}}


def render_leg(dev, rank, world, steps, barrier, pk, n_samples, n_surface, with_device_leg=True):
    """2^18-ray batches through the fused marcher; e2e = Renderer.render_batch_ray from pinned host rays"""
    import types
    from goslam_b200 import render as render_mod
    net, rays, _ = make_renderer(dev, 43 + rank)
    out = {}
    if with_device_leg:
        rd = [r.to(dev) for r in rays]
        with torch.no_grad():
            ms_r = max_over_ranks(time_gpu(lambda: net(*rd), max(5, steps // 2), 3, barrier), world)
        rbytes = RAYS * (512.0 * SAMPLES + 1216.0)
        out.update({"metric": "rendered Mrays/s", "value": world * RAYS / ms_r / 1e3, "unit": "Mrays/s", "ms_per_batch": ms_r,
                    "roofline": {"kernel": "neus_forward_kernel", "bound": "hbm", "achieved": rbytes / (ms_r * 1e-3) / 1e9,
                                 "peak": pk["hbm"], "unit": "GB/s", "frac": rbytes / (ms_r * 1e-3) / 1e9 / pk["hbm"],
                                 "traffic": None,
                                 "note": "algorithmic bytes (38,080 B/ray); the 25 MB table is L2-resident"}})
    rcfg = {"rendering": {"lindisp": False, "perturb": 1.0, "N_samples": n_samples, "N_surface": n_surface}}
    renderer = render_mod.Renderer(rcfg, None, types.SimpleNamespace(H=512, W=512, fx=460.8, fy=460.8, cx=256.0, cy=256.0))
    gt_depth = 0.5 + 2.5 * torch.rand(RAYS, generator=torch.Generator().manual_seed(43 + rank))
    hp = [rays[0].pin_memory(), rays[1].pin_memory(), gt_depth.pin_memory()]
    keep = {"color": torch.empty(RAYS, 3).pin_memory(), "depth": torch.empty(RAYS, 1).pin_memory()}

    def render_e2e():
        ro, rdir, gd = [x.to(dev, non_blocking=True) for x in hp]
        o = renderer.render_batch_ray(ro, rdir, net, None, device=dev, gt_depth=gd)
        for k in ("color", "depth"):
            keep[k].copy_(o[k].reshape(keep[k].shape), non_blocking=True)
    with torch.no_grad():
        ms_re = max_over_ranks(time_gpu(render_e2e, max(5, steps // 2), 3, barrier), world)
    out["e2e"] = {"value": world * RAYS / ms_re / 1e3, "unit": "Mrays/s", "ms_per_batch": ms_re,
                  "call": "Renderer.render_batch_ray (z-sampling %d+%d + marcher), host rays in, colour+depth out" % (n_samples, n_surface),
                  "h2d_bytes_per_batch": RAYS * 7 * 4, "d2h_bytes_per_batch": RAYS * 4 * 4}
    return out


def mapping_leg(dev, rank, world, steps, barrier):
    """SURVEY 8f-3: one iteration of Mapper.optimize_map's loop body (src/mapping.py:84-131) — differentiable forward
    through the fused marcher, the mapping losses, loss.backward() through the renderer backward kernels, clip, AdamW —
    on 2^16 rays x 72 samples PER RANK (the reference samples ~4.4 k pixels per iteration; the batch here is sized to fill the
    GPU).  Also the reference-sized batch.  N > 1: data parallel (parallel.mapping_loss_local / allreduce_gradients)."""
    from goslam_b200 import parallel, synthetic
    net, _, _ = make_renderer(dev, 43)
    parallel.broadcast_parameters(list(net.parameters()))          # data parallel: every replica starts from rank 0's weights
    out = {}
    for tag, R in (("rays_65536", 1 << 16), ("rays_4096", 1 << 12)):
        ro, rd, zv, ds = [t.to(dev) for t in synthetic.make_rays(R, S=SAMPLES, seed=47 + rank)]
        g = torch.Generator().manual_seed(5 + rank)
        rc = torch.rand(R, 3, generator=g).to(dev)
        depth = (0.5 + 2.5 * torch.rand(R, 1, generator=g)).to(dev)
        opt = torch.optim.AdamW([{"params": net.get_training_parameters(), "lr": 1e-4},
                                 {"params": net.get_volume_parameters(), "lr": 1e-3}], betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
        params = net.get_training_parameters() + net.get_volume_parameters()
        parts = {}

        def fwd_bwd():
            opt.zero_grad()
            with torch.enable_grad():
                o = net(ro, rd, zv, ds)
                # the reference's loss (src/mapping.py:97-128, weights of configs/go_slam.yaml) on this rank's slice of a
                # global batch of world x R rays, in the SUM form whose gradients add up over the ranks
                total = parallel.mapping_loss_local(net, o, rc, depth, world * R, 2.0, 2.0, 0.1)
            total.backward()

        def step():
            fwd_bwd()
            parallel.allreduce_gradients(params)          # no-op on one rank; N > 1: the replicas stay identical
            torch.nn.utils.clip_grad_norm_(params, max_norm=35.0)
            opt.step()

        n = max(5, steps // 2)
        ms = max_over_ranks(time_gpu(step, n, 3, barrier), world)
        ms_fb = time_gpu(fwd_bwd, n, 3, lambda: None)
        with torch.no_grad():
            ms_f = time_gpu(lambda: net(ro, rd, zv, ds), n, 3, lambda: None)
        out[tag] = {"value": world * R / ms / 1e3, "unit": "Mrays/s (forward + backward + AdamW)", "ms_per_iteration": ms,
                    "ms_forward_backward": ms_fb, "ms_inference_forward": ms_f, "rays": R, "samples_per_ray": SAMPLES}
    if world > 1:                                    # data parallel: the replicas must still hold identical parameters
        import torch.distributed as dist
        same = torch.ones(1, device=dev)
        for prm in params:
            ref = prm.detach().clone()
            dist.broadcast(ref, src=0)
            same = torch.minimum(same, torch.tensor([float(torch.equal(ref, prm.detach()))], device=dev))
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        out["replicas_bit_identical"] = bool(same.item() == 1.0)
    out["parallelism"] = ("data parallel over %d rank(s): each rank renders and back-propagates its %s-ray slice, gradients of all "
                          "parameters (12.6 M-entry hash grid + 10 k others) are summed with NCCL all-reduce, every rank takes the "
                          "same AdamW step (weak scaling)" % (world, "R"))
    out["call"] = ("goslam_b200.InstantNeuS.forward under grad -> mapping losses -> loss.backward() (goslam_neus_composite_backward, "
                   "cuBLAS fp16 GEMMs of the colour network with a loss scale, goslam_neus_grid_backward) -> clip_grad_norm_ -> torch.optim.AdamW.step")
    return out


# ------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-render", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only", default="", help="comma list of legs to run besides the main one: headline,sharded,full,render,mapping")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the main leg computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback in the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        barrier = lambda: dist.barrier()   # noqa: E731
    else:
        barrier = lambda: None             # noqa: E731
    legs = set(x for x in args.only.split(",") if x) or {"headline", "sharded", "full", "render", "mapping"}
    if args.no_render:
        legs.discard("render")

    from goslam_b200 import _lib
    _lib.load()
    pk = peaks()
    warm = max(args.warmup, 3)

    # ---- configs[1]: the metric's own configuration (value / e2e / roofline of the line)
    sc = make_window(43 + rank)
    main_rec, clocks = window_leg(sc, dev, args.steps, warm, barrier, world, pk, clock_index=local,
                                  dump_dir=args.dump_outputs if rank == 0 else None)
    line = {"metric": METRIC, "value": main_rec["value"], "unit": "updates/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": main_rec["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16 corr (f32 accumulate) / f32 BA (f64 solve)",
            "data": "synthetic", "config": workload_config(world), "clocks": clocks,
            "e2e": main_rec["e2e"],
            "gpu_launches": 6 * args.steps,   # kmajor, corr build, reproject, lookup, ba_prep, ba (all iterations in one cooperative kernel)
            "roofline": main_rec["roofline"]}

    # ---- north_star headline shape: 640x480 input -> 60x80 @1/8, same 8-keyframe / 36-edge window
    if "headline" in legs:
        sc60 = make_window(143 + rank, ht=60, wd=80)
        rec60, _ = window_leg(sc60, dev, max(10, args.steps // 2), warm, barrier, world, pk)
        rec60["workload"] = ("synthetic 640x480 RGB-D -> 60x80 @1/8, 8-keyframe window, 36 edges, corr build + 4-level "
                             "r=3 lookup + 3 BA iters per update; one window per GPU (weak scaling)")
        line["headline_640x480"] = rec60
        line["stereo_40x60"] = stereo_build_leg(dev, rank, max(10, args.steps // 2), warm, pk)

    # ---- configs[3]: one global-BA graph sharded over the ranks (strong scaling, NCCL exchange per BA iteration)
    if "sharded" in legs:
        line["sharded_graph"] = sharded_graph_leg(dev, max(10, args.steps // 2), warm, barrier, world, rank)

    # ---- configs[2]-style update with the update operator in the loop, through FactorGraph.update
    if "full" in legs:
        line["full_update"] = full_update_leg(dev, max(10, args.steps // 2), warm, barrier, world, rank)

    if "render" in legs:
        line["render"] = render_leg(dev, rank, world, args.steps, barrier, pk, 24, SAMPLES - 24)
        # configs[2] (Replica mono): 48 stratified + 24 surface samples (configs/Replica/replica_mono.yaml:54-55);
        # the marcher's work is the same 72 samples per ray, only the z-sampling split differs
        line["render"]["mono_48_24"] = render_leg(dev, rank, world, args.steps, barrier, pk, 48, SAMPLES - 48,
                                                  with_device_leg=False)["e2e"]

    if "mapping" in legs:
        line["mapping_step"] = mapping_leg(dev, rank, world, args.steps, barrier)

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        # the whole step (36 edges, 3 iterations, nothing extrapolated) when the host does it in <= 40 s,
        # else a proportional sample
        n_e, n_it = cpu_sample_plan(sc, 40.0)
        full, spent = cpu_reference_step(sc, n_e, n_it)
        line["cpu_baseline"] = {"value": 1.0 / full, "unit": "updates/s", "cores": os.cpu_count(), "kind": "port",
                                "extrapolated": n_e != 36,
                                "sample": "corr build+pyramid+lookup on %d/36 edges + %d/3 BA iterations "
                                          "(%.1f s of CPU work)%s" % (n_e, n_it, spent, "" if n_e == 36 else
                                                                      ", extrapolated linearly to the full step")}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
