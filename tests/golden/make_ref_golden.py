"""Generate tests/golden/ref_kernels.npz: outputs of THE REFERENCE'S OWN CUDA KERNELS (oracle/_ref, built by
oracle/build_ref.py from the reference's src/lib/*.cu) on the seeded inputs of tests/test_gpu_ref.py and
tests/test_gpu_ba_large.py.  Needs a B200 and oracle/_ref; the tests themselves need neither the reference nor
oracle/_ref.  Which elements of an output are stored is described in tests/test_gpu_ref.py.

Run:  python tests/golden/make_ref_golden.py [OUT_DIR]      (default: next to this file)
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import test_gpu_ba_large as L  # noqa: E402
import test_gpu_ref as T  # noqa: E402
from oracle import build_ref, ref_ba_driver  # noqa: E402


def ba_entry(z, meta, ref, key, sc, a, iters, lm, ep, motion_only):
    meta[key + ".inputs"] = T.digest(sc["poses"], sc["disps"], *a.values())
    p, d = sc["poses"].clone().to(T.dev()), sc["disps"].clone().to(T.dev())
    dx, dz, status, kx = ref_ba_driver.ba(ref, p, d, a["intr"], a["sens"], a["tg"], a["wg"], a["eta"], a["ii"], a["jj"],
                                          sc["t0"], sc["t1"], iters, lm, ep, motion_only)
    meta[key + "_status"] = status
    T.record(z, meta, key + "_poses", p)
    T.record(z, meta, key + "_disps", d)
    T.record(z, meta, key + "_dx", dx)
    if not motion_only:
        z[key + "_kx"] = kx.cpu().numpy()
        T.record(z, meta, key + "_dz", dz)


def main(out_dir):
    ref = build_ref.load_ref()
    assert ref is not None, "oracle/_ref is not built (python oracle/build_ref.py)"
    z, meta = {}, {}
    for dtype in (torch.float16, torch.float32):
        for key, vol, coords in T.corr_index_inputs(dtype):
            meta[key + ".inputs"] = T.digest(vol, coords)
            T.record(z, meta, key, ref.corr_index_forward(vol, coords, 3)[0], exact=dtype == torch.float16)
    for key, f1, f2, coords in T.altcorr_inputs():
        meta[key + ".inputs"] = T.digest(f1, f2, coords)
        T.record(z, meta, key, ref.altcorr_forward(f1, f2, coords, 3)[0])
    for size in ((8, 40, 80), (12, 30, 40)):
        key, poses, disps, intr, ii, jj, ix, th = T.geometry_inputs(size)
        meta[key + ".inputs"] = T.digest(poses, disps, intr, ii, jj, ix, th)
        for beta in (0.3, 0.75):
            T.record(z, meta, "%s_fd%g" % (key, beta), ref.frame_distance(poses, disps, intr, ii, jj, beta), full=True)
        c, v = ref.projmap(poses, disps, intr, ii, jj)
        T.record(z, meta, key + "_projmap", c[..., :2].contiguous())
        T.record(z, meta, key + "_valid", v, exact=True)
        T.record(z, meta, key + "_iproj", ref.iproj(poses, disps, intr))
        T.record(z, meta, key + "_depth_filter", ref.depth_filter(poses, disps, intr, ix, th), full=True)
    for case in T.BA_CASES:
        for motion_only in (False, True):
            sc, a = T.ba_inputs(case)
            ba_entry(z, meta, ref, T.ba_key(case, motion_only), sc, a, 2, 1e-4, 0.1, motion_only)
    for name in L.REF_CASES:
        for motion_only in (False, True):
            sc, a, lm, ep, iters = L.ref_inputs(name)
            ba_entry(z, meta, ref, "ba_large_%s_mo%d" % (name, motion_only), sc, a, iters, lm, ep, motion_only)
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "ref_kernels.npz")
    np.savez_compressed(path, meta=np.array(json.dumps(meta, sort_keys=True)), **z)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
