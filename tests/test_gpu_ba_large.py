"""GPU parity of the GLOBAL-BA-sized solve paths (VERDICT r01 weak #1): every case here has 6P > 96, so
`goslam_ba` runs the multi-kernel driver — `ba_solve_cluster_kernel` (one 8-CTA cluster, matrix in
distributed shared memory, P <= ~100) or `ba_solve_kernel` out of global scratch beyond — and the split form `goslam_ba_phase1/2` that the
multi-GPU driver uses.  Checked against the fp64 CPU oracle (1e-4, north_star) and against the
reference's own CUDA kernels + restated Eigen host code (recorded in tests/golden/ref_kernels.npz).

config 4 (SURVEY §8d): 64 keyframes at 30x40, edges from Backend.ba's rule (src/backend.py:25-99 with
radius=1, nms=5, thresh=25, max_factors=384), t0=1, t1=64 (P=63, 6P=378), lm=1e-5, ep=1e-2, iters=2
(src/factor_graph.py:317-318)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import ba_oracle, geom_oracle  # noqa: E402


def dev():
    return torch.device("cuda:0")


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-12)


def _scene(num_kf, ht, wd, rgbd=True, seed=43, edges="neighborhood", radius=3):
    from goslam_b200 import droid_backends, graph, synthetic
    sc, g = synthetic.make_scene(num_kf=num_kf, ht=ht, wd=wd, rgbd=rgbd, seed=seed, with_fmaps=False,
                                 buffer=num_kf + 2, radius=radius)
    if edges == "backend":
        # Backend.ba's edge selection on the device (bit-exact vs the reference method: test_gpu_parity)
        t = num_kf
        ix = torch.arange(0, t)
        ii, jj = torch.meshgrid(ix, ix, indexing="ij")
        d = droid_backends.frame_distance_bidirectional(
            sc["poses"].to(dev()), sc["disps"].to(dev()), sc["intrinsics"][0].to(dev()).contiguous(),
            ii.reshape(-1).to(dev()), jj.reshape(-1).to(dev()), 0.3)
        es = graph.backend_edges(d, 0, t, 1, 5, 25.0, 384, False)
        assert es is not None
        sc["ii"], sc["jj"] = es[0].cpu(), es[1].cpu()
    sc["t0"], sc["t1"] = 1, num_kf
    coords, _ = geom_oracle.reproject(sc["poses"].numpy(), sc["disps"].numpy(), sc["intrinsics"].numpy(),
                                      sc["ii"].numpy(), sc["jj"].numpy())
    targets, weights, eta = synthetic.make_update(sc, torch.from_numpy(coords[0]), g, noise=0.7)
    sc["poses"][1:num_kf, :3] += 0.01 * torch.randn(num_kf - 1, 3, generator=g)
    sc["disps"][:num_kf] *= 1 + 0.03 * torch.randn(num_kf, ht, wd, generator=g)
    return sc, targets, weights, eta


CASES = {
    "P20": dict(num_kf=21, ht=12, wd=16, lm=1e-4, ep=0.1, iters=3),                         # 6P = 120
    "P31": dict(num_kf=32, ht=12, wd=16, lm=1e-4, ep=0.1, iters=3),                       # 6P = 186
    "P31_mono": dict(num_kf=32, ht=9, wd=13, rgbd=False, lm=1e-4, ep=0.1, iters=2),
    "cfg4": dict(num_kf=64, ht=30, wd=40, edges="backend", lm=1e-5, ep=1e-2, iters=2),           # 6P = 378
    "cfg4_dense": dict(num_kf=64, ht=30, wd=40, radius=3, lm=1e-5, ep=1e-2, iters=2),            # 372 edges
    "P99": dict(num_kf=100, ht=9, wd=13, radius=2, lm=1e-4, ep=0.1, iters=2),                    # 6P = 594: largest cluster solve
    "P120_global": dict(num_kf=121, ht=6, wd=8, radius=2, lm=1e-4, ep=0.1, iters=1),             # beyond the cluster: global scratch
}


def _make(name):
    c = dict(CASES[name])
    lm, ep, iters = c.pop("lm"), c.pop("ep"), c.pop("iters")
    sc, tg, wg, eta = _scene(**c)
    return sc, tg, wg, eta, lm, ep, iters


_cache = {}


def _case(name):
    if name not in _cache:
        _cache[name] = _make(name)
    return _cache[name]


def _oracle(name, motion_only):
    key = (name, motion_only, "oracle")
    if key not in _cache:
        sc, tg, wg, eta, lm, ep, iters = _case(name)
        _cache[key] = ba_oracle.ba(
            sc["poses"].numpy(), sc["disps"].numpy(), sc["intrinsics"][0].numpy(), sc["disps_sens"].numpy(),
            tg.numpy(), wg.numpy(), eta.numpy(), sc["ii"].numpy(), sc["jj"].numpy(),
            sc["t0"], sc["t1"], iters, lm, ep, motion_only, dtype=np.float64)
    return _cache[key]


@pytest.mark.parametrize("motion_only", [False, True])
@pytest.mark.parametrize("name", list(CASES))
def test_ba_large_vs_oracle(name, motion_only):
    from goslam_b200 import droid_backends
    sc, tg, wg, eta, lm, ep, iters = _case(name)
    t0, t1 = sc["t0"], sc["t1"]
    assert 6 * (t1 - t0) > 96                       # really the multi-kernel driver
    if name == "cfg4":                              # local window (2 * 63) + NMS-thinned long-range pairs
        assert 150 <= sc["ii"].numel() <= 386 and int((sc["ii"] - sc["jj"]).abs().max()) > 10
    poses, disps = sc["poses"].clone().to(dev()), sc["disps"].clone().to(dev())
    dx, dz, status = droid_backends.ba(
        poses, disps, sc["intrinsics"][0].to(dev()).contiguous(), sc["disps_sens"].to(dev()),
        tg.to(dev()), wg.to(dev()), eta.to(dev()), sc["ii"].to(dev()), sc["jj"].to(dev()),
        t0, t1, iters, lm, ep, motion_only, return_status=True)
    rp, rd, rdx, rdz, rst = _oracle(name, motion_only)
    assert status.cpu().numpy().tolist() == rst.tolist() == [0] * iters
    assert _rel(poses.cpu().numpy(), rp) < 1e-4                  # north_star: 1e-4 relative
    assert _rel(dx.cpu().numpy(), rdx) < 5e-3                    # the last step itself (small vs the state)
    if not motion_only:
        assert _rel(disps.cpu().numpy(), rd) < 1e-4
        assert np.abs(dz.cpu().numpy() - rdz).max() < 1e-4 * max(np.abs(rd).max(), 1.0)
    else:
        assert torch.equal(disps.cpu(), sc["disps"]) and dz is None
    assert torch.equal(poses[:t0].cpu(), sc["poses"][:t0]) and torch.equal(poses[t1:].cpu(), sc["poses"][t1:])


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("motion_only", [False, True])
@pytest.mark.parametrize("name", ["P20", "cfg4"])
def test_ba_split_form_vs_oracle(name, motion_only, world):
    """goslam_ba_phase1 / goslam_ba_phase2 with `world` emulated ranks on ONE GPU: edges sharded by source
    frame, local systems summed (what the all-reduce does), every rank solves + retracts its replica and
    back-substitutes only the frames it owns [owner_lo, owner_hi), owned rows merged (the all-gather)."""
    from goslam_b200 import parallel
    sc, tg, wg, eta, lm, ep, iters = _case(name)
    t0, t1 = sc["t0"], sc["t1"]
    num, ht, wd = sc["disps"].shape
    kx = torch.unique(torch.cat([torch.arange(t0, t1), sc["ii"]]))
    eta_f = torch.zeros(num, ht, wd)
    eta_f[kx] = eta
    D = {k: v.to(dev()) for k, v in dict(intr=sc["intrinsics"][0].contiguous(), sens=sc["disps_sens"], tg=tg, wg=wg,
                                         eta=eta_f, ii=sc["ii"], jj=sc["jj"]).items()}
    bounds = parallel.shard_frames_by_edges(sc["ii"], num, world)
    ranks = []
    for lo, hi in bounds:
        p, d = sc["poses"].clone().to(dev()), sc["disps"].clone().to(dev())
        sel = parallel.local_edges(D["ii"], lo, hi)
        ranks.append(dict(be=parallel.CudaBackend(p, d, D["intr"], D["sens"], t0, t1), p=p, d=d, lo=lo, hi=hi,
                          tg=D["tg"][sel].contiguous(), wg=D["wg"][sel].contiguous(),
                          ii=D["ii"][sel].contiguous(), jj=D["jj"][sel].contiguous()))
    assert sum(r["ii"].numel() for r in ranks) == sc["ii"].numel()
    for _ in range(iters):
        total = None
        for r in ranks:
            s = r["be"].phase1(r["tg"], r["wg"], D["eta"], r["ii"], r["jj"], motion_only)
            total = s if total is None else total + s
        for r in ranks:
            r["dx"], st = r["be"].phase2(total, lm, ep, motion_only, r["lo"], r["hi"], return_status=True)
            assert int(st.item()) == 0
        if not motion_only:
            merged = torch.cat([r["d"][r["lo"]:r["hi"]] for r in ranks])
            for r in ranks:
                r["d"].copy_(merged)
    rp, rd, rdx, _, _ = _oracle(name, motion_only)
    for r in ranks:
        assert torch.equal(r["p"], ranks[0]["p"])                 # replicas stay bit-identical
        assert _rel(r["p"].cpu().numpy(), rp) < 1e-4
        assert _rel(r["dx"].cpu().numpy(), rdx) < 5e-3
        if not motion_only:
            assert _rel(r["d"].cpu().numpy(), rd) < 1e-4


REF_CASES = ["P20", "P31", "cfg4"]


def ref_inputs(name):
    sc, tg, wg, eta, lm, ep, iters = _case(name)
    a = dict(intr=sc["intrinsics"][0].to(dev()).contiguous(), sens=sc["disps_sens"].to(dev()), tg=tg.to(dev()),
             wg=wg.to(dev()), eta=eta.to(dev()), ii=sc["ii"].to(dev()), jj=sc["jj"].to(dev()))
    return sc, a, lm, ep, iters


@pytest.mark.parametrize("motion_only", [False, True])
@pytest.mark.parametrize("name", REF_CASES)
def test_ba_large_vs_reference_kernels(name, motion_only):
    """same systems through the reference's own kernels (projective_transform_kernel, accum, EEt6x6, Ev6x1,
    EvT6x1, pose/disp retraction; src/lib/droid_kernels.cu) + the restated Eigen host code, as recorded in
    tests/golden/ref_kernels.npz (see test_gpu_ref.py)."""
    from goslam_b200 import droid_backends
    from test_gpu_ref import Golden, check_ba
    ref = Golden("ref_kernels.npz")
    sc, a, lm, ep, iters = ref_inputs(name)
    key = "ba_large_%s_mo%d" % (name, motion_only)
    ref.check_inputs(key, sc["poses"], sc["disps"], *a.values())
    t0, t1 = sc["t0"], sc["t1"]
    p1, d1 = sc["poses"].clone().to(dev()), sc["disps"].clone().to(dev())
    dx1, dz1, st1 = droid_backends.ba(p1, d1, a["intr"], a["sens"], a["tg"], a["wg"], a["eta"], a["ii"], a["jj"],
                                      t0, t1, iters, lm, ep, motion_only, return_status=True)
    assert st1.cpu().tolist() == ref[key + "_status"]
    check_ba(ref, key, p1, d1, dx1, dz1, motion_only)


def test_ba_eta_row_mismatch_is_reported_not_misapplied():
    """ADVICE r01: a damping tensor whose row count is neither 1 nor the number of depth slots used to be
    clamped onto the wrong frames silently.  Now: state untouched, dx = 0, status 2 (the reference raises)."""
    from goslam_b200 import droid_backends
    from test_gpu_parity import _ba_case
    sc, tg, wg, eta = _ba_case(num_kf=6, ht=12, wd=16, rgbd=True)
    for bad_eta in (eta[:-1].contiguous(), torch.cat([eta, eta[:2]])):
        poses, disps = sc["poses"].clone().to(dev()), sc["disps"].clone().to(dev())
        dx, dz, status = droid_backends.ba(
            poses, disps, sc["intrinsics"][0].to(dev()).contiguous(), sc["disps_sens"].to(dev()), tg.to(dev()),
            wg.to(dev()), bad_eta.to(dev()), sc["ii"].to(dev()), sc["jj"].to(dev()), 1, 6, 2, 1e-4, 0.1, False,
            return_status=True)
        assert status.cpu().tolist() == [2, 2]
        assert torch.equal(poses.cpu(), sc["poses"]) and torch.equal(disps.cpu(), sc["disps"])
        assert float(dx.abs().max()) == 0.0
    # frame-indexed damping == slot-indexed damping
    num, ht, wd = sc["disps"].shape
    kx = torch.unique(torch.cat([torch.arange(1, 6), sc["ii"]]))
    eta_f = torch.zeros(num, ht, wd)
    eta_f[kx] = eta
    outs = []
    for e, by_frame in ((eta, False), (eta_f, True)):
        poses, disps = sc["poses"].clone().to(dev()), sc["disps"].clone().to(dev())
        droid_backends.ba(poses, disps, sc["intrinsics"][0].to(dev()).contiguous(), sc["disps_sens"].to(dev()),
                          tg.to(dev()), wg.to(dev()), e.to(dev()), sc["ii"].to(dev()), sc["jj"].to(dev()), 1, 6, 2,
                          1e-4, 0.1, False, eta_by_frame=by_frame)
        outs.append((poses, disps))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
