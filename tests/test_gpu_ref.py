"""GPU parity against the REFERENCE'S OWN CUDA KERNELS: tests/golden/ref_kernels.npz holds what src/lib/*.cu of
the reference computed on a B200 (compiled for sm_100a by oracle/build_ref.py, recorded by
tests/golden/make_ref_golden.py) from the seeded inputs built here.  This is the pin for K2/K4/K6-K16: identical
inputs, our C-ABI kernels vs the reference's kernels.

An output of up to FULL elements is stored whole; one that a test wants bit-equal, as a SHA-256 of all of it.  Of any
other output the file keeps a fixed sample of SAMPLE elements, its largest magnitude (the tolerances scale with it)
and its L1 mass; a test checks its per-element bound on the sample and what that bound implies for the L1 mass."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FULL, SAMPLE = 2048, 512


def digest(*ts):
    """SHA-256 of the tensors' values (-0.0 hashed as 0.0, as torch.equal compares)"""
    h = hashlib.sha256()
    for t in ts:
        h.update((t.detach() + 0).contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def sample_index(n):
    """the fixed subset of a flattened n-element output that a golden file keeps (None: all of it)"""
    if n <= FULL:
        return None
    return torch.randperm(n, generator=torch.Generator().manual_seed(n))[:SAMPLE].sort().values


def record(arrays, meta, key, t, exact=False, full=False):
    """store output t under `key`: kept elements in `arrays`, everything else in `meta` (tests/golden/make_ref_golden.py)"""
    flat = t.detach().reshape(-1).cpu()
    meta[key] = {"shape": list(t.shape)}
    if exact:
        meta[key]["sha256"] = digest(t)
        return
    idx = None if full else sample_index(flat.numel())
    arrays[key] = (flat if idx is None else flat[idx]).numpy()
    meta[key]["amax"] = float(flat.double().abs().max()) if flat.numel() else 0.0
    meta[key]["l1"] = float(flat.double().abs().sum())


class Golden:
    """one golden file of reference-kernel outputs: arrays of kept elements + a JSON entry "meta" with, per key,
    shape / amax / l1 / sha256 of an output, the SHA-256 of a case's inputs, or a small list (BA status)"""

    def __init__(self, name):
        self.z = np.load(os.path.join(GOLDEN_DIR, name))
        self.meta = json.loads(str(self.z["meta"]))

    def __getitem__(self, key):
        return self.z[key] if key in self.z.files else self.meta[key]

    def check_inputs(self, key, *ts):
        assert self.meta[key + ".inputs"] == digest(*ts), (
            "%s: inputs differ from those the golden file was recorded from (tests/golden/make_ref_golden.py)" % key)

    def pair(self, key, ours):
        """(ours, theirs) on the elements of output `key` that the file keeps"""
        assert list(ours.shape) == self.meta[key]["shape"], (key, tuple(ours.shape))
        theirs = torch.from_numpy(self.z[key]).to(ours.device)
        flat = ours.reshape(-1)
        if theirs.numel() == flat.numel():
            return flat, theirs
        return flat[sample_index(flat.numel()).to(ours.device)], theirs

    def amax(self, key):
        return self.meta[key]["amax"]

    def equal(self, key, ours):
        """torch.equal(ours, theirs) on the whole output"""
        return list(ours.shape) == self.meta[key]["shape"] and digest(ours) == self.meta[key]["sha256"]

    def l1_within(self, key, ours, atol, rtol=0.0):
        """|L1(ours) - L1(theirs)| is within what |ours - theirs| <= atol + rtol |theirs| per element allows"""
        l1 = self.meta[key]["l1"]
        return abs(float(ours.double().abs().sum()) - l1) <= 1.001 * (ours.numel() * atol + rtol * l1)


@pytest.fixture(scope="module")
def ref():
    return Golden("ref_kernels.npz")


def dev():
    return torch.device("cuda:0")


def _scene(*a, **kw):
    from goslam_b200 import synthetic
    return synthetic.make_scene(*a, **kw)


def corr_index_inputs(dtype):
    """(key, volume, coords) of the 4 pyramid levels"""
    g = torch.Generator().manual_seed(0)
    N, h, w = 4, 40, 80
    for lvl in range(4):
        h2, w2 = h >> lvl, w >> lvl
        vol = torch.randn(N, h, w, h2, w2, generator=g).to(dtype).to(dev())
        base = torch.stack(torch.meshgrid(torch.arange(w).float(), torch.arange(h).float(), indexing="xy"), 0)
        coords = ((base[None].repeat(N, 1, 1, 1) + 4 * torch.randn(N, 2, h, w, generator=g)) / 2 ** lvl).to(dev()).contiguous()
        yield "corr_index_%s_l%d" % (str(dtype).split(".")[-1], lvl), vol, coords


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_corr_index_forward_vs_reference_kernel(ref, dtype):
    from goslam_b200 import droid_backends
    for key, vol, coords in corr_index_inputs(dtype):
        ref.check_inputs(key, vol, coords)
        ours, = droid_backends.corr_index_forward(vol, coords, 3)
        torch.cuda.synchronize()
        if dtype == torch.float16:
            # both are a fixed sequence of correctly rounded half operations
            assert ref.equal(key, ours), key
        else:
            # same FMA chain; allow the compiler one contraction difference
            o, t = ref.pair(key, ours)
            tol = 1e-6 * max(1.0, ref.amax(key))
            assert (o - t).abs().max().item() <= tol
            assert (o == t).float().mean().item() > 0.99
            assert ref.l1_within(key, ours, tol), key


def altcorr_inputs():
    """(key, fmap1, fmap2, coords) of 3 pyramid levels"""
    g = torch.Generator().manual_seed(1)
    B, H, W, C = 5, 30, 40, 128
    f1 = torch.randn(B, H, W, C, generator=g).to(dev())
    for lvl in range(3):
        f2 = torch.randn(B, H >> lvl, W >> lvl, C, generator=g).to(dev())
        base = torch.stack(torch.meshgrid(torch.arange(W).float(), torch.arange(H).float(), indexing="xy"), -1)
        coords = ((base[None, None].repeat(B, 1, 1, 1, 1) + 3 * torch.randn(B, 1, H, W, 2, generator=g)) / 2 ** lvl).to(dev()).contiguous()
        yield "altcorr_l%d" % lvl, f1, f2, coords


def test_altcorr_vs_reference_kernel(ref):
    from goslam_b200 import droid_backends
    for key, f1, f2, coords in altcorr_inputs():
        ref.check_inputs(key, f1, f2, coords)
        ours, = droid_backends.altcorr_forward(f1, f2, coords, 3)
        # fp32 dot products of 128 terms, different association (reference: 4 chunks of 32)
        o, t = ref.pair(key, ours)
        tol = 1e-4 * max(1.0, ref.amax(key))
        assert (o - t).abs().max().item() < tol
        assert ref.l1_within(key, ours, tol), key


def geometry_inputs(size):
    n = size[0]
    sc, g = _scene(*size, with_fmaps=False)
    poses, disps = sc["poses"].to(dev()), sc["disps"].to(dev())
    intr = sc["intrinsics"][0].to(dev()).contiguous()
    ii, jj = torch.meshgrid(torch.arange(n), torch.arange(n), indexing="ij")
    ii, jj = ii.reshape(-1).to(dev()), jj.reshape(-1).to(dev())
    ix = torch.arange(n, device=dev())
    th = torch.full((n,), 0.02, device=dev())
    return "geometry_%d_%d_%d" % tuple(size), poses, disps, intr, ii, jj, ix, th


@pytest.mark.parametrize("size", [(8, 40, 80), (12, 30, 40)])
def test_geometry_vs_reference_kernels(ref, size):
    from goslam_b200 import droid_backends
    key, poses, disps, intr, ii, jj, ix, th = geometry_inputs(size)
    ref.check_inputs(key, poses, disps, intr, ii, jj, ix, th)
    for beta in (0.3, 0.75):
        ours = droid_backends.frame_distance(poses, disps, intr, ii, jj, beta)
        _, theirs = ref.pair("%s_fd%g" % (key, beta), ours)
        theirs = theirs.view_as(ours)
        # same per-thread order and the same reduction tree; what remains is the compiler's choice
        # of FMA contractions inside the projection: <= 2 ulp, and the edge lists the frontend /
        # backend derive from the distances (thresholds, sort order) are identical
        assert (ours - theirs).abs().max().item() <= 2 * 4.8e-7 * max(1.0, theirs[theirs < 999].abs().max().item())
        assert torch.equal(ours >= 999, theirs >= 999)
        for thresh in (1.0, 4.0, 16.0, 25.0):
            assert torch.equal(ours < thresh, theirs < thresh)
        ko = torch.argsort(ours, stable=True)
        kt = torch.argsort(theirs, stable=True)
        assert torch.equal(ii[ko], ii[kt]) and torch.equal(jj[ko], jj[kt])
    c, v = droid_backends.projmap(poses, disps, intr, ii, jj)
    o, t = ref.pair(key + "_projmap", c[..., :2].contiguous())
    assert torch.allclose(o, t, rtol=1e-6, atol=1e-5) and ref.l1_within(key + "_projmap", c[..., :2], 1e-5, 1e-6)
    assert ref.equal(key + "_valid", v)
    o, t = ref.pair(key + "_iproj", droid_backends.iproj(poses, disps, intr))
    assert torch.allclose(o, t, rtol=1e-6, atol=1e-6)
    a, b = ref.pair(key + "_depth_filter", droid_backends.depth_filter(poses, disps, intr, ix, th))
    assert a.numel() == int(np.prod(ref.meta[key + "_depth_filter"]["shape"]))     # stored whole
    assert (a == b).float().mean().item() > 0.999


BA_CASES = [dict(num_kf=8, ht=40, wd=80, rgbd=True), dict(num_kf=8, ht=40, wd=80, rgbd=False),
            dict(num_kf=6, ht=30, wd=40, rgbd=True, stereo_edges=2)]


def ba_key(case, motion_only):
    return "ba_%d_%d_%d_rgbd%d_st%d_mo%d" % (case["num_kf"], case["ht"], case["wd"], case["rgbd"],
                                             case.get("stereo_edges", 0), motion_only)


def ba_inputs(case):
    from test_gpu_parity import _ba_case
    sc, targets, weights, eta = _ba_case(**case)
    args = dict(intr=sc["intrinsics"][0].to(dev()).contiguous(), sens=sc["disps_sens"].to(dev()),
                tg=targets.to(dev()), wg=weights.to(dev()), eta=eta.to(dev()),
                ii=sc["ii"].to(dev()), jj=sc["jj"].to(dev()))
    return sc, args


@pytest.mark.parametrize("case", BA_CASES)
@pytest.mark.parametrize("motion_only", [False, True])
def test_ba_vs_reference_kernels(ref, case, motion_only):
    """our fused device-side BA vs the reference's kernels + restated Eigen host code (oracle/ref_ba_driver.py)."""
    from goslam_b200 import droid_backends
    sc, args = ba_inputs(case)
    key = ba_key(case, motion_only)
    ref.check_inputs(key, sc["poses"], sc["disps"], *args.values())
    t0, t1 = sc["t0"], sc["t1"]
    p1, d1 = sc["poses"].clone().to(dev()), sc["disps"].clone().to(dev())
    dx1, dz1, st1 = droid_backends.ba(p1, d1, args["intr"], args["sens"], args["tg"], args["wg"], args["eta"],
                                      args["ii"], args["jj"], t0, t1, 2, 1e-4, 0.1, motion_only, return_status=True)
    assert st1.cpu().tolist() == ref[key + "_status"]
    check_ba(ref, key, p1, d1, dx1, dz1, motion_only)


def check_ba(ref, key, p1, d1, dx1, dz1, motion_only):
    """the BA state and last step against the reference run stored under `key`"""
    def rel(name, ours):
        o, t = ref.pair(key + name, ours)
        return ((o - t).abs().max() / max(ref.amax(key + name), 1e-12)).item()
    assert rel("_poses", p1) < 1e-4, rel("_poses", p1)
    assert rel("_disps", d1) < 1e-4, rel("_disps", d1)
    assert ref.l1_within(key + "_disps", d1, 1e-4 * ref.amax(key + "_disps"))
    assert rel("_dx", dx1) < 5e-3
    if not motion_only:
        kx = torch.from_numpy(ref[key + "_kx"]).to(dz1.device)
        o, t = ref.pair(key + "_dz", dz1[kx])
        tol = 1e-4 * max(1.0, ref.amax(key + "_disps"))
        assert (o - t).abs().max().item() < tol
        assert ref.l1_within(key + "_dz", dz1[kx], tol)
