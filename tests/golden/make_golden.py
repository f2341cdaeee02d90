"""Generate tests/golden/*.npz by running THE REFERENCE'S OWN PYTHON (imported from
/root/reference, which exists only in the build container) on small seeded inputs.

Stub modules stand in for natives that are absent from the snapshot:
    droid_backends -> oracle.corr_oracle lookup (only CorrBlock.__call__ needs it)
    lietorch       -> go-slam_b200/lietorch.py (host-side SE3 algebra, pinned by the CUDA twins)
    torch_scatter  -> 6-line scatter_sum / scatter_mean
    tinycudann     -> oracle.neus_oracle restatement (hash grid with autograd input-gradient, MLP)
    mcubes, trimesh-> empty modules (only used by mesh extraction)
What each fixture pins:
    corr_block.npz    CorrBlock.__init__/corr/__call__           src/modules/corr.py:25-76
    reproject.npz     pops.projective_transform (jacobian=False)  src/geom/projective_ops.py:114-144
    ba_torch.npz      dx of the reference's dense pure-torch BA   src/geom/ba.py:26-101 + chol.py
    neus.npz          InstantNeuS.forward (9 outputs)             src/InstantNeuS.py:295-370
    render_z.npz      Renderer.render_batch_ray z-sampling        src/render.py:99-171
    cvx_upsample.npz  cvx_upsample (f32 and f16 masks)            src/droid_net.py:9-23
    proximity.npz     FactorGraph.add_proximity_factors edges     src/factor_graph.py:384-450
    altcorr_pyramid.npz AltCorrBlock.__init__ pyramid            src/modules/corr.py:97-111
    backend_edges.npz Backend.ba edge selection (loop=False)      src/backend.py:25-99
    factor_graph.npz  FactorGraph + DepthVideo state machine      src/factor_graph.py:85-450, src/depth_video.py:194-269
    conv_gru.npz      ConvGRU.forward (fp32)                      src/modules/gru.py:21-39
    update_module.npz UpdateModule.forward incl. GraphAgg (fp32)  src/droid_net.py:33-140
Run:  python tests/golden/make_golden.py      (writes next to this file)
"""
import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)

from oracle import corr_oracle, neus_oracle  # noqa: E402


def install_stubs():
    import goslam_b200  # noqa: F401
    from goslam_b200 import lietorch as lt
    sys.modules["lietorch"] = lt

    db = types.ModuleType("droid_backends")

    def corr_index_forward(volume, coords, radius):
        out = corr_oracle.corr_index_forward(volume.numpy(), coords.numpy(), radius)
        return [torch.from_numpy(out)]
    db.corr_index_forward = corr_index_forward
    sys.modules["droid_backends"] = db

    ts = types.ModuleType("torch_scatter")

    def scatter_sum(src, index, dim=-1, dim_size=None):
        shape = list(src.shape)
        shape[dim] = dim_size if dim_size is not None else int(index.max()) + 1
        out = torch.zeros(shape, dtype=src.dtype)
        return out.index_add_(dim, index, src)

    def scatter_mean(src, index, dim=-1, dim_size=None):
        s = scatter_sum(src, index, dim, dim_size)
        c = scatter_sum(torch.ones_like(src), index, dim, dim_size).clamp_min(1)
        return s / c
    ts.scatter_sum, ts.scatter_mean = scatter_sum, scatter_mean
    sys.modules["torch_scatter"] = ts

    for name in ("mcubes", "trimesh"):
        sys.modules[name] = types.ModuleType(name)

    # ---- tinycudann restatement ----------------------------------------------------------
    tcnn = types.ModuleType("tinycudann")
    metas, total_entries = neus_oracle.hashgrid_meta()

    class _GridFn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x, params):
            table = params.detach().half().numpy().reshape(-1, 2)
            ctx.save_for_backward(x, params)
            enc = neus_oracle.hashgrid_encode(x.detach().numpy().astype(np.float32), table)
            return torch.from_numpy(enc)          # float16, like tcnn

        @staticmethod
        def backward(ctx, dy):
            x, params = ctx.saved_tensors
            table = params.detach().half().numpy().reshape(-1, 2)
            # tcnn: per-sample dL/dy (cast to half) times d(enc)/dx in fp32
            dyn = dy.detach().float().numpy()
            assert np.allclose(dyn, dyn[:1]), "restatement assumes a sample-independent dL/dy"
            g = neus_oracle.hashgrid_input_grad(x.detach().numpy().astype(np.float32), table, dyn[0])
            return torch.from_numpy(g), None

    class Encoding(torch.nn.Module):
        def __init__(self, n_input_dims, encoding_config):
            super().__init__()
            assert encoding_config["otype"] == "HashGrid"
            self.n_output_dims = 32
            self.params = torch.nn.Parameter((torch.rand(total_entries * 2) * 2 - 1) * 1e-4)

        def forward(self, x):
            return _GridFn.apply(x, self.params)

    class Network(torch.nn.Module):
        def __init__(self, n_input_dims, n_output_dims, network_config):
            super().__init__()
            assert (n_input_dims, n_output_dims, network_config["n_neurons"]) == (67, 3, 64)
            self.params = torch.nn.Parameter(torch.zeros(64 * 80 + 64 * 64 + 16 * 64))

        def forward(self, x):
            out = neus_oracle.mlp_forward(x.detach().float().numpy(), self.params.detach().half().numpy())
            return torch.from_numpy(out)          # float16 [n,3]

    tcnn.Encoding, tcnn.Network = Encoding, Network
    sys.modules["tinycudann"] = tcnn

    # torch.cuda.device(...) context is used at model construction; make it a no-op on CPU
    class _NoDev:
        def __init__(self, *a, **k):
            pass

        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False
    torch.cuda.device = _NoDev


def ref_import(name):
    if REF not in sys.path:
        sys.path.insert(0, REF)
    return importlib.import_module(name)


def gen_corr_block():
    corr_mod = ref_import("src.modules.corr")
    g = torch.Generator().manual_seed(43)
    N, h, w = 2, 16, 24      # >= 16: the reference pools once more after the last level
    out = {}
    for tag, dt in (("f32", torch.float32), ("f16", torch.float16)):
        f1 = torch.randn(1, N, 128, h, w, generator=g).to(dt)
        f2 = torch.randn(1, N, 128, h, w, generator=g).to(dt)
        blk = corr_mod.CorrBlock(f1, f2)
        coords = torch.stack(torch.meshgrid(torch.arange(w).float(), torch.arange(h).float(), indexing="xy"), -1)
        coords = coords[None, None].repeat(1, N, 1, 1, 1) + 2.0 * torch.randn(1, N, h, w, 2, generator=g)
        sampled = blk(coords)
        out.update({tag + "_fmap1": f1.numpy(), tag + "_fmap2": f2.numpy(), tag + "_coords": coords.numpy(),
                    tag + "_sampled": sampled.numpy()})
        for i, p in enumerate(blk.corr_pyramid):
            out["%s_level%d" % (tag, i)] = p.numpy()
    np.savez_compressed(os.path.join(HERE, "corr_block.npz"), **out)


def small_scene():
    from goslam_b200 import synthetic
    return synthetic.make_scene(num_kf=6, ht=12, wd=16, seed=43, rgbd=False, with_fmaps=False)


def gen_reproject():
    pops = ref_import("src.geom.projective_ops")
    import lietorch
    sc, g = small_scene()
    ii = torch.cat([sc["ii"], torch.tensor([2, 3])])       # + two stereo (ii == jj) edges
    jj = torch.cat([sc["jj"], torch.tensor([2, 3])])
    coords, valid = pops.projective_transform(lietorch.SE3(sc["poses"][None]), sc["disps"][None],
                                              sc["intrinsics"][None], ii, jj)
    np.savez_compressed(os.path.join(HERE, "reproject.npz"), poses=sc["poses"].numpy(), disps=sc["disps"].numpy(),
                        intrinsics=sc["intrinsics"].numpy(), ii=ii.numpy(), jj=jj.numpy(),
                        coords=coords.numpy(), valid=valid.numpy())


def gen_ba_torch():
    """dx / dz of the reference's dense torch BA on a scene where its formulation and the CUDA one
    coincide: no sensor depth (no prior), all points in front of both cameras (no MIN_DEPTH
    clipping: 0.2 vs 0.25 never triggers), no stereo edges."""
    sys.path.insert(0, os.path.join(REF, "src", "geom"))     # `import projective_ops` inside ba.py
    ba_mod = ref_import("src.geom.ba")
    import lietorch
    from goslam_b200 import synthetic
    from oracle import geom_oracle
    sc, g = small_scene()
    coords, _ = geom_oracle.reproject(sc["poses"].numpy(), sc["disps"].numpy(), sc["intrinsics"].numpy(),
                                      sc["ii"].numpy(), sc["jj"].numpy())
    targets, weights, eta = synthetic.make_update(sc, torch.from_numpy(coords[0]), g, noise=0.7)
    cap = {}
    orig = ba_mod.schur_solve

    def spy(H, E, C, v, w, **kw):
        dx, dz = orig(H, E, C, v, w, **kw)
        cap["dx"], cap["dz"] = dx, dz
        return dx, dz
    ba_mod.schur_solve = spy
    N, ht, wd = sc["ii"].numel(), sc["ht"], sc["wd"]
    tgt = targets.permute(0, 2, 3, 1)[None].contiguous()   # [1,N,h,w,2]
    wgt = weights.permute(0, 2, 3, 1)[None].contiguous()
    t0 = 1
    kx = torch.unique(sc["ii"])
    assert kx.numel() == eta.shape[0]
    res = {}
    for tag, dt in (("", torch.float32), ("64", torch.float64)):
        torch.set_default_dtype(dt)      # the reference builds its stereo constant with torch.tensor([...])
        poses = lietorch.SE3(sc["poses"][None].clone().to(dt))
        ba_mod.BA(tgt.to(dt), wgt.to(dt), (eta[None] - 1e-7).to(dt), poses, sc["disps"][None].clone().to(dt),
                  sc["intrinsics"][None].to(dt), sc["ii"], sc["jj"], fixedp=t0)
        res["dx" + tag] = cap["dx"][0].numpy()
        res["dz" + tag] = cap["dz"][0].numpy()
    torch.set_default_dtype(torch.float32)
    np.savez_compressed(os.path.join(HERE, "ba_torch.npz"), poses=sc["poses"].numpy(), disps=sc["disps"].numpy(),
                        intrinsics=sc["intrinsics"].numpy(), ii=sc["ii"].numpy(), jj=sc["jj"].numpy(),
                        targets=targets.numpy(), weights=weights.numpy(), eta=eta.numpy(), t0=t0, **res)


def gen_neus():
    neus_mod = ref_import("src.InstantNeuS")
    from goslam_b200 import synthetic
    metas, total_entries = neus_oracle.hashgrid_meta()
    offs = [m["offset"] * 2 for m in metas] + [total_entries * 2]
    ress = [m["res"] for m in metas]
    w = synthetic.make_neus_weights(seed=7, total_grid_params=total_entries * 2, layout=(offs, ress))
    bound = [[-2.0, 2.0], [-2.0, 2.0], [-2.0, 2.0]]
    net = neus_mod.InstantNeuS(synthetic.NEUS_CFG, bound, device="cpu")
    with torch.no_grad():
        net.sdf_network.encoding.encoding.params.copy_(w["grid"])
        net.sdf_network.sdf_layer.weight.copy_(w["sdf_w"])
        net.sdf_network.sdf_layer.bias.copy_(w["sdf_b"])
        net.color_network._B.copy_(w["color_B"])
        net.color_network.network.params.copy_(w["mlp"])
    rt = torch.tensor([[-1.8, 1.9], [-2.0, 2.0], [-1.5, 2.0]])
    net.update_bound(rt)
    ro, rd, zv, ds = synthetic.make_rays(48, S=72, seed=11)
    out = net(ro, rd, zv, ds)
    np.savez_compressed(os.path.join(HERE, "neus.npz"), rays_o=ro.numpy(), rays_d=rd.numpy(), z_vals_in=zv.numpy(),
                        dists=ds.numpy(), rt_bound=rt.numpy(), bound=np.array(bound, np.float32), weights_seed=7,
                        **{"out_" + k: v.detach().float().numpy() for k, v in out.items()})


def gen_neus_grad():
    """Renderer backward golden: the REFERENCE's InstantNeuS.forward (its own autograd.grad normal included) under
    enable_grad with the tcnn modules replaced by the differentiable restatements of oracle/neus_grad_oracle.py, the
    loss of Mapper.optimize_map (src/mapping.py:97-128, weights of configs/go_slam.yaml, uncertainty weighting on) and
    .backward().  Stored: inputs, the loss, the forward outputs and every parameter gradient (the 12.6 M-entry hash-grid
    gradient as its non-zero entries)."""
    neus_mod = ref_import("src.InstantNeuS")
    import tinycudann
    from oracle import neus_grad_oracle as ngo
    from goslam_b200 import synthetic
    old = tinycudann.Encoding, tinycudann.Network
    tinycudann.Encoding, tinycudann.Network = ngo.TorchHashGrid, ngo.TorchMLP
    try:
        metas, total_entries = neus_oracle.hashgrid_meta()
        offs = [m["offset"] * 2 for m in metas] + [total_entries * 2]
        ress = [m["res"] for m in metas]
        w = synthetic.make_neus_weights(seed=9, total_grid_params=total_entries * 2, layout=(offs, ress))
        bound = [[-2.0, 2.0], [-2.0, 2.0], [-2.0, 2.0]]
        net = neus_mod.InstantNeuS(synthetic.NEUS_CFG, bound, device="cpu")
        with torch.no_grad():
            net.sdf_network.encoding.encoding.params.copy_(w["grid"])
            net.sdf_network.sdf_layer.weight.copy_(w["sdf_w"])
            net.sdf_network.sdf_layer.bias.copy_(w["sdf_b"])
            net.color_network._B.copy_(w["color_B"])
            net.color_network.network.params.copy_(w["mlp"])
        rt = torch.tensor([[-1.8, 1.9], [-2.0, 2.0], [-1.5, 2.0]])
        net.update_bound(rt)
        R, S = 40, 32
        ro, rd, zv, ds = synthetic.make_rays(R, S=S, seed=13, n_uniform=12)
        g = torch.Generator().manual_seed(17)
        rays_color = torch.rand(R, 3, generator=g)
        rays_depth = 0.5 + 2.5 * torch.rand(R, generator=g)
        rays_depth[::9] = 0.0                                     # invalid sensor depth: ray excluded from the losses
        with torch.enable_grad():
            out = net(ro, rd, zv, ds)
            # src/mapping.py:97-128
            depth = rays_depth.reshape(-1, 1)
            valid = (depth > 0).reshape(-1)
            unc = 1.0 / torch.sqrt(out["depth_variance"][valid].detach() + 1e-10)
            color_loss = torch.abs(out["color"][valid] - rays_color[valid]).mean()
            depth_loss = (torch.abs(out["depth"][valid] - depth[valid]) * unc).mean()
            sdf_loss, sparse_loss = net.compute_sdf_error(sdf=out["sdf"][valid], z_vals=out["z_vals"][valid], gt_depth=depth[valid])
            total = color_loss * 2.0 + depth_loss * 1.0 + (sdf_loss + sparse_loss) * 2.0 + 0.1 * out["gradient_error"].mean()
            total.backward()
        gg = net.sdf_network.encoding.encoding.params.grad.numpy()
        nz = np.nonzero(gg)[0]
        np.savez_compressed(
            os.path.join(HERE, "neus_grad.npz"), rays_o=ro.numpy(), rays_d=rd.numpy(), z_vals_in=zv.numpy(), dists=ds.numpy(),
            rt_bound=rt.numpy(), bound=np.array(bound, np.float32), weights_seed=9, rays_color=rays_color.numpy(),
            rays_depth=rays_depth.numpy(), loss=np.float32(total.item()),
            parts=np.array([color_loss.item(), depth_loss.item(), sdf_loss.item(), sparse_loss.item(), out["gradient_error"].item()], np.float32),
            grid_grad_idx=nz.astype(np.int64), grid_grad_val=gg[nz].astype(np.float32),
            g_sdf_w=net.sdf_network.sdf_layer.weight.grad.numpy(), g_sdf_b=net.sdf_network.sdf_layer.bias.grad.numpy(),
            g_color_B=net.color_network._B.grad.numpy(), g_mlp=net.color_network.network.params.grad.numpy(),
            g_variance=net.variance_network.variance.grad.numpy(),
            **{"out_" + k: v.detach().float().numpy() for k, v in out.items()})
        print("neus_grad: loss %.6f, %d non-zero grid gradients, |g_sdf_w| %.4e |g_mlp| %.4e |g_B| %.4e g_var %.4e" % (
            total.item(), nz.size, np.linalg.norm(net.sdf_network.sdf_layer.weight.grad.numpy()),
            np.linalg.norm(net.color_network.network.params.grad.numpy()), np.linalg.norm(net.color_network._B.grad.numpy()),
            float(net.variance_network.variance.grad)))
    finally:
        tinycudann.Encoding, tinycudann.Network = old


def gen_neus_adamw():
    """Mapping-step trajectory golden: 8 iterations of Mapper.optimize_map's loop body (src/mapping.py:84-131: forward
    under enable_grad, loss, backward, clip_grad_norm_(35), AdamW step with the two parameter groups of :55-58) run by the
    REFERENCE's InstantNeuS on the inputs of neus_grad.npz, with uncertainty weighting off and both learning rates x0.1
    (with the config's rates this synthetic scene's uncertainty-weighted depth loss grows 20x in one step — in the
    reference as well).  Stored: the 8 losses and their parts."""
    neus_mod = ref_import("src.InstantNeuS")
    import tinycudann
    from oracle import neus_grad_oracle as ngo
    from goslam_b200 import synthetic
    old = tinycudann.Encoding, tinycudann.Network
    tinycudann.Encoding, tinycudann.Network = ngo.TorchHashGrid, ngo.TorchMLP
    try:
        g = np.load(os.path.join(HERE, "neus_grad.npz"))
        metas, total_entries = neus_oracle.hashgrid_meta()
        offs = [m["offset"] * 2 for m in metas] + [total_entries * 2]
        ress = [m["res"] for m in metas]
        w = synthetic.make_neus_weights(seed=int(g["weights_seed"]), total_grid_params=total_entries * 2, layout=(offs, ress))
        net = neus_mod.InstantNeuS(synthetic.NEUS_CFG, g["bound"].tolist(), device="cpu")
        with torch.no_grad():
            net.sdf_network.encoding.encoding.params.copy_(w["grid"])
            net.sdf_network.sdf_layer.weight.copy_(w["sdf_w"])
            net.sdf_network.sdf_layer.bias.copy_(w["sdf_b"])
            net.color_network._B.copy_(w["color_B"])
            net.color_network.network.params.copy_(w["mlp"])
        net.update_bound(torch.from_numpy(g["rt_bound"]))
        net_lr, grid_lr = 1e-4, 1e-3
        opt = torch.optim.AdamW([{"params": net.get_training_parameters(), "lr": net_lr},
                                 {"params": net.get_volume_parameters(), "lr": grid_lr}], betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
        args = [torch.from_numpy(g[k]) for k in ("rays_o", "rays_d", "z_vals_in", "dists")]
        rc, rdp = torch.from_numpy(g["rays_color"]), torch.from_numpy(g["rays_depth"])
        rows = []
        for it in range(8):
            opt.zero_grad()
            with torch.enable_grad():
                out = net(*args)
                depth = rdp.reshape(-1, 1)
                valid = (depth > 0).reshape(-1)
                cl = torch.abs(out["color"][valid] - rc[valid]).mean()
                dl = torch.abs(out["depth"][valid] - depth[valid]).mean()
                sl, spl = net.compute_sdf_error(sdf=out["sdf"][valid], z_vals=out["z_vals"][valid], gt_depth=depth[valid])
                total = cl * 2.0 + dl * 1.0 + (sl + spl) * 2.0 + 0.1 * out["gradient_error"].mean()
                total.backward()
            torch.nn.utils.clip_grad_norm_(net.get_training_parameters() + net.get_volume_parameters(), max_norm=35.0)
            opt.step()
            rows.append([total.item(), cl.item(), dl.item(), sl.item(), spl.item(), out["gradient_error"].item()])
            print("neus_adamw step %d: %s" % (it, " ".join("%.5f" % v for v in rows[-1])))
        np.savez_compressed(os.path.join(HERE, "neus_adamw.npz"), rows=np.array(rows, np.float32), net_lr=net_lr, grid_lr=grid_lr)
    finally:
        tinycudann.Encoding, tinycudann.Network = old


def gen_render_z():
    render_mod = ref_import("src.render")
    cfg = {"rendering": {"lindisp": False, "perturb": 1.0, "N_samples": 24, "N_surface": 48}}
    slam = types.SimpleNamespace(H=64, W=64, fx=50.0, fy=50.0, cx=32.0, cy=32.0)
    r = render_mod.Renderer(cfg, None, slam)
    cap = {}

    class Net:
        bound = torch.tensor([[-2.0, 2.0], [-2.0, 2.0], [-2.0, 2.0]])

        def __call__(self, ro, rd, zv, dst, render_params=None):
            cap["z"], cap["d"] = zv, dst
            return {"z": zv}
    from goslam_b200 import synthetic
    ro, rd, _, _ = synthetic.make_rays(32, S=72, seed=5)
    depth = 0.5 + 2.0 * torch.rand(32, generator=torch.Generator().manual_seed(5))
    depth[::7] = 0.0
    torch.manual_seed(1234)
    r.render_batch_ray(ro, rd, Net(), None, device="cpu", gt_depth=depth)
    np.savez_compressed(os.path.join(HERE, "render_z.npz"), rays_o=ro.numpy(), rays_d=rd.numpy(), gt_depth=depth.numpy(),
                        z_vals=cap["z"].numpy(), dists=cap["d"].numpy(), torch_seed=1234)


def gen_cvx_upsample():
    dn = ref_import("src.droid_net")
    g = torch.Generator().manual_seed(77)
    # one thread: torch's float16 softmax then rounds the same on every host (see oracle/upsample_oracle.py)
    torch.set_num_threads(1)
    out = {}
    for tag, (b, ht, wd, dim) in {"disp": (3, 6, 9, 1), "flow": (2, 5, 7, 2)}.items():
        data = torch.rand(b, ht, wd, dim, generator=g) + 0.1
        mask = 2.0 * torch.randn(b, 576, ht, wd, generator=g)
        out[tag + "_data"], out[tag + "_mask"] = data.numpy(), mask.numpy()
        out[tag + "_out_f32"] = dn.cvx_upsample(data, mask).numpy()
        out[tag + "_out_f16mask"] = dn.cvx_upsample(data, mask.half()).float().numpy()
    np.savez_compressed(os.path.join(HERE, "cvx_upsample.npz"), **out)


def gen_proximity():
    """FactorGraph.add_proximity_factors (src/factor_graph.py:384-450) itself, with a stub video whose
    distance() returns a prepared matrix; the edges handed to add_factors are the golden output."""
    fg_mod = ref_import("src.factor_graph")
    rng = np.random.default_rng(21)
    cases = []
    for (t0, t1, t, rad, nms, thresh, maxf, stereo, n_old) in [
            (7, 0, 12, 2, 2, 16.0, 48, False, 6), (0, 0, 9, 2, 2, 16.0, 60, False, 0),
            (10, 3, 22, 3, 1, 20.0, 40, True, 9), (4, 0, 10, 2, 2, 12.0, 14, False, 3),
            (5, 9, 30, 2, 2, 25.0, 200, True, 20),       # t1 > t0: negative column indices wrap (Python semantics)
            (6, 8, 20, 3, 2, 30.0, 90, False, 5), (0, 0, 40, 2, 2, 14.0, 400, False, 60),
            (3, 0, 14, 2, 3, 30.0, -1, False, 0)]:
        ilen, jlen = t - t0, t - t1
        dist = (rng.random(ilen * jlen) * 40).astype(np.float32)
        dist[rng.random(ilen * jlen) < 0.1] = 150.0
        old = rng.integers(0, t, size=(n_old, 2)).astype(np.int64)
        cap = {}
        g = fg_mod.FactorGraph.__new__(fg_mod.FactorGraph)
        g.device = "cpu"
        g.max_factors = maxf
        g.ii, g.jj = torch.from_numpy(old[:, 0].copy()), torch.from_numpy(old[:, 1].copy())
        g.ii_bad = g.jj_bad = g.ii_inac = g.jj_inac = torch.zeros(0, dtype=torch.long)
        g.video = types.SimpleNamespace(counter=types.SimpleNamespace(value=t), stereo=stereo,
                                        distance=lambda ii, jj, beta, _d=dist: torch.from_numpy(_d.copy()))
        g.add_factors = lambda ii, jj, remove=False, _c=cap: _c.update(ii=ii.numpy().copy(), jj=jj.numpy().copy())
        g.add_proximity_factors(t0, t1, rad=rad, nms=nms, thresh=thresh, remove=False)
        cases.append(dict(params=np.array([t0, t1, t, rad, nms, maxf, int(stereo)], np.int64), thresh=np.float32(thresh),
                          dist=dist, old=old, es=np.stack([cap["ii"], cap["jj"]], 1)))
    out = {}
    for n, c in enumerate(cases):
        for k, v in c.items():
            out["c%d_%s" % (n, k)] = v
    out["n_cases"] = np.int64(len(cases))
    np.savez_compressed(os.path.join(HERE, "proximity.npz"), **out)


def gen_backend_edges():
    """Backend.ba (src/backend.py:25-128) with loop=False and stubbed graph/video: the edges handed to
    graph.add_factors are the golden output (None when it returns early)."""
    be_mod = ref_import("src.backend")
    rng = np.random.default_rng(33)
    out, n = {}, 0
    for (ts, te, radius, nms, thresh, maxf, stereo, tsl, loop) in [
            (0, 14, 2, 2, 18.0, 96, False, None, False), (3, 25, 3, 1, 25.0, 80, True, None, False),
            (0, 3, 2, 2, 10.0, 20, False, None, False), (5, 30, 1, 2, 15.0, 30, False, None, False),
            (0, 40, 2, 2, 22.0, 300, False, 25, True), (2, 30, 3, 1, 30.0, 120, True, 18, True)]:
        ilen = te - (tsl if loop else ts)
        jlen = te - ts
        dist = (rng.random(ilen * jlen) * 40).astype(np.float32)
        if loop:                                   # smooth field so that 3x3 neighbourhoods agree often enough
            dist = (dist.reshape(ilen, jlen) * 0.25 + 30.0 * np.abs(np.sin(np.arange(ilen)[:, None] * 0.4 + np.arange(jlen)[None] * 0.3))).astype(np.float32).reshape(-1)
        cap = {}
        b = be_mod.Backend.__new__(be_mod.Backend)
        b.beta, b.device = 0.75, "cpu"
        b.video = types.SimpleNamespace(stereo=stereo, dirty=torch.zeros(te + 1, dtype=torch.bool),
                                        distance=lambda ii, jj, beta, _d=dist: torch.from_numpy(_d.copy()))
        graph = types.SimpleNamespace(ii=[], update_lowmem=lambda **k: None, clear_edges=lambda: None,
                                      add_factors=lambda ii, jj, remove=False, _c=cap: _c.update(ii=ii.numpy().copy(), jj=jj.numpy().copy()))
        b.ba(ts, te, 4, graph, nms, radius, thresh, maxf, t_start_loop=tsl, loop=loop)
        out["b%d_params" % n] = np.array([ts, te, radius, nms, maxf, int(stereo), -1 if tsl is None else tsl, int(loop)], np.int64)
        out["b%d_thresh" % n] = np.float32(thresh)
        out["b%d_dist" % n] = dist
        out["b%d_es" % n] = np.stack([cap["ii"], cap["jj"]], 1) if cap else np.zeros((0, 2), np.int64)
        out["b%d_early" % n] = np.int64(0 if cap else 1)
        n += 1
    out["n_cases"] = np.int64(n)
    np.savez_compressed(os.path.join(HERE, "backend_edges.npz"), **out)


def gen_altcorr_block():
    """AltCorrBlock.__call__ plumbing (src/modules/corr.py:113-145) with the oracle standing in for the
    CUDA op: pins the gather / per-level scaling / channel layout of the reference class."""
    def alt_fwd(f1, f2, coords, r):
        return [torch.from_numpy(corr_oracle.altcorr_forward(f1.numpy(), f2.numpy(), coords.numpy(), r))]
    sys.modules["droid_backends"].altcorr_forward = alt_fwd
    corr_mod = ref_import("src.modules.corr")
    g = torch.Generator().manual_seed(13)
    h, w = 16, 24
    fm = torch.randn(1, 4, 128, h, w, generator=g)
    ii, jj = torch.tensor([0, 3, 2]), torch.tensor([1, 0, 3])
    base = torch.stack(torch.meshgrid(torch.arange(w).float(), torch.arange(h).float(), indexing="xy"), -1)
    coords = base[None, None].repeat(1, 3, 1, 1, 1) + 2 * torch.randn(1, 3, h, w, 2, generator=g)
    out5 = corr_mod.AltCorrBlock(fm)(coords, ii, jj)
    c6 = coords.unsqueeze(-2).repeat(1, 1, 1, 1, 2, 1) + torch.tensor([0.0, 0.5]).view(1, 1, 1, 1, 2, 1)
    out6 = corr_mod.AltCorrBlock(fm)(c6, ii, jj)
    np.savez_compressed(os.path.join(HERE, "altcorr_block.npz"), fmaps=fm.numpy(), ii=ii.numpy(), jj=jj.numpy(),
                        coords=coords.numpy(), coords6=c6.numpy(), out5=out5[:, :, ::7].numpy(), out6=out6[:, :, ::7].numpy())


def gen_altcorr_pyramid():
    """AltCorrBlock.__init__ (src/modules/corr.py:97-111): the /4-scaled, average-pooled NHWC pyramid."""
    corr_mod = ref_import("src.modules.corr")
    g = torch.Generator().manual_seed(12)
    fm = torch.randn(1, 3, 128, 16, 24, generator=g).half()   # the reference pools once more than it needs: h >= 16
    blk = corr_mod.AltCorrBlock(fm)
    out = {"fmaps": fm.numpy()}
    for i, lvl in enumerate(blk.pyramid):
        out["level%d" % i] = lvl.numpy()
    np.savez_compressed(os.path.join(HERE, "altcorr_pyramid.npz"), **out)


def gen_factor_graph():
    """The REFERENCE FactorGraph + DepthVideo (src/factor_graph.py, src/depth_video.py) driven through
    tests/tools/fg_scenario.py on the CPU.  Natives are the oracle: droid_backends.{ba, frame_distance,
    corr_index_forward, altcorr_forward}; lietorch = the host SE3 shim; update_op = tests/tools/stub_update_op."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "tools"))
    import fg_scenario
    from oracle import ba_oracle, geom_oracle
    db = sys.modules["droid_backends"]

    def ba(poses, disps, intrinsics, disps_sens, targets, weights, eta, ii, jj, t0, t1, iters, lm, ep, motion_only):
        rp, rd, dx, dz, st = ba_oracle.ba(poses.numpy(), disps.numpy(), intrinsics.numpy(), disps_sens.numpy(),
                                          targets.numpy(), weights.numpy(), eta.numpy(), ii.numpy(), jj.numpy(),
                                          int(t0), int(t1), int(iters), lm, ep, bool(motion_only))
        assert list(st) == [0] * int(iters)
        poses.copy_(torch.from_numpy(rp))
        disps.copy_(torch.from_numpy(rd))
        return [torch.from_numpy(dx), torch.from_numpy(dz)]

    def frame_distance(poses, disps, intrinsics, ii, jj, beta):
        return torch.from_numpy(geom_oracle.frame_distance(poses.numpy(), disps.numpy(), intrinsics.numpy(),
                                                           ii.numpy(), jj.numpy(), beta))

    def altcorr_forward(f1, f2, coords, r):
        return [torch.from_numpy(corr_oracle.altcorr_forward(f1.numpy(), f2.numpy(), coords.numpy(), r))]
    db.ba, db.frame_distance, db.altcorr_forward = ba, frame_distance, altcorr_forward
    dv_mod = ref_import("src.depth_video")
    fg_mod = ref_import("src.factor_graph")

    # DepthVideo.format_indices defaults to device='cuda' (src/depth_video.py:184) and distance() relies on it
    orig_fmt = dv_mod.DepthVideo.format_indices
    dv_mod.DepthVideo.format_indices = staticmethod(lambda ii, jj, device="cpu": orig_fmt(ii, jj, "cpu"))
    CpuVideo = dv_mod.DepthVideo

    # the reference's age eviction uses an UNSTABLE argsort (src/factor_graph.py:103); record whether it and the
    # stable order we use ever disagree in this scenario
    disagreements = []
    orig_argsort = torch.argsort

    def spy_argsort(x, *a, **k):
        got = orig_argsort(x, *a, **k)
        if x.dim() == 1 and not k.get("stable", False):
            disagreements.append(not torch.equal(got, orig_argsort(x, *a, stable=True, **k)))
        return got
    torch.argsort = spy_argsort
    try:
        cfg, args = fg_scenario.cfg_and_args("cpu")
        video = CpuVideo(cfg, args)
        fg_scenario.fill_video(video, fg_scenario.make_inputs())
        with torch.no_grad():
            out = fg_scenario.run(fg_mod.FactorGraph, video, "cpu")
    finally:
        torch.argsort = orig_argsort
    print("argsort calls (True = differs from the stable order):", disagreements,
          [int(out["s%02d_ii" % k].size) for k in range(int(out["n_steps"]))])
    assert disagreements and not any(disagreements), "age eviction hit an argsort tie that the stable order resolves differently"
    out["evictions"] = np.int64(len(disagreements))
    np.savez_compressed(os.path.join(HERE, "factor_graph.npz"), **out)
    print("factor_graph: %d snapshots, %d age evictions, final edges %s" % (int(out["n_steps"]), len(disagreements),
                                                                            [int(out["s%02d_ii" % k].size) for k in range(int(out["n_steps"]))]))


def gen_conv_gru():
    """ConvGRU.forward (src/modules/gru.py:21-39) itself, fp32 on the CPU, default-initialised weights under
    torch.manual_seed(77) (the test rebuilds them the same way); ragged sizes (w % 16 != 0, h % 8 != 0)."""
    gru_mod = ref_import("src.modules.gru")
    out = {}
    for tag, (B, h, w) in {"a": (3, 16, 24), "b": (2, 12, 20)}.items():
        torch.manual_seed(77)
        gru = gru_mod.ConvGRU(128, 128 + 128 + 64)
        g = torch.Generator().manual_seed(5 + B)
        # inputs are fp16-representable (stored as fp16): the graph keeps net / inp / corr / flow in half anyway
        net = torch.tanh(torch.randn(B, 128, h, w, generator=g)).half()
        inp = torch.relu(torch.randn(B, 128, h, w, generator=g)).half()
        corr = torch.relu(torch.randn(B, 128, h, w, generator=g)).half()
        flow = torch.relu(torch.randn(B, 64, h, w, generator=g)).half()
        with torch.no_grad():
            res = gru(net.float(), inp.float(), corr.float(), flow.float())
        out.update({tag + "_net": net.numpy(), tag + "_inp": inp.numpy(), tag + "_corr": corr.numpy(), tag + "_flow": flow.numpy(),
                    tag + "_out": res.numpy(), tag + "_wsum": np.float64(sum(float(p.double().sum()) for p in gru.parameters()))})
    np.savez_compressed(os.path.join(HERE, "conv_gru.npz"), **out)


def gen_update_module():
    """UpdateModule.forward (src/droid_net.py:107-140) of the reference, fp32 on the CPU, default-initialised weights
    under torch.manual_seed(78); inputs are fp16-representable (the graph holds them in half)."""
    dn = ref_import("src.droid_net")
    torch.manual_seed(78)
    upd = dn.UpdateModule()
    g = torch.Generator().manual_seed(9)
    num, h, w = 6, 16, 24
    net = torch.tanh(torch.randn(1, num, 128, h, w, generator=g)).half()
    inp = torch.relu(torch.randn(1, num, 128, h, w, generator=g)).half()
    corr = (0.7 * torch.randn(1, num, 196, h, w, generator=g)).half()
    flow = (4.0 * torch.randn(1, num, 4, h, w, generator=g)).clamp(-64, 64).half()
    ii = torch.tensor([0, 0, 1, 3, 3, 1])
    jj = torch.tensor([1, 2, 0, 1, 2, 3])
    with torch.no_grad():
        n2, delta, weight, eta, upmask = upd(net.float(), inp.float(), corr.float(), flow.float(), ii, jj)
    np.savez_compressed(os.path.join(HERE, "update_module.npz"), net=net.numpy(), inp=inp.numpy(), corr=corr.numpy(),
                        flow=flow.numpy(), ii=ii.numpy(), jj=jj.numpy(), out_net=n2.half().numpy(), out_delta=delta.numpy(),
                        out_weight=weight.numpy(), out_eta=eta.numpy(), out_upmask=upmask[:, :, ::9].numpy(),
                        wsum=np.float64(sum(float(p.detach().double().sum()) for p in upd.parameters())))


if __name__ == "__main__":
    if not os.path.isdir(REF):
        raise SystemExit("needs /root/reference (build container only)")
    install_stubs()
    which = sys.argv[1:] or ["corr_block", "reproject", "ba_torch", "neus", "render_z", "cvx_upsample", "proximity", "backend_edges", "altcorr_pyramid", "altcorr_block"]
    for name in which:
        globals()["gen_" + name]()
        print("wrote", name)
