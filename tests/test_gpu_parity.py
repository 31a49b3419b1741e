"""-m gpu: the CUDA path (through the C ABI) against the oracle on the same seeded inputs.

Bars: bit-exact for integer / index work (winner selection, index maps, lists, counts, NN
indices, sort order); fp32 losses within 1e-5 rel of the oracle (BASELINE.json north_star);
the 12-float transform gradient within 1e-5 of its max-abs entry; normals p99 <= 1e-6 and max <= 5e-5
against the reference's LAPACK eigenvectors (see test_normals_and_lists)."""
import math
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, case_inputs, digest, unsort_uv
from oracle import delora_oracle as orc

pytestmark = pytest.mark.gpu

DEV = "cuda"
CASES = ["small_16x180", "kitti_64x720", "kitti_64x2048"]
_cache = {}


def oracle_case(name, golden):
    if name not in _cache:
        meta = golden[name]
        cfg, (scan_1, scan_2, t_gt, t_pred) = case_inputs(meta)
        out = orc.pair_forward_backward(scan_1, scan_2, t_pred, cfg)
        _cache[name] = (meta, cfg, scan_1, scan_2, t_pred, out)
    return _cache[name]


def fov(cfg):
    return cfg["horizontal_field_of_view"], cfg["kitti"]["vertical_field_of_view"]


def gpu_project(cloud, h, w, hf, vf, div_mode=0):
    from delora_b200 import ops
    pts = cloud[None].contiguous().to(DEV)
    n = torch.tensor([cloud.shape[1]], dtype=torch.int32, device=DEV)
    image, index_map = ops.project(pts, n, h, w, hf, vf, div_mode)
    u, v, r = ops.project_uv(pts, n, h, w, hf, vf, div_mode)
    return image[0].cpu(), index_map[0].cpu(), u[0].cpu(), v[0].cpu(), r[0].cpu()


def check_projection(cloud, h, w, hf, vf, label, max_flip_fraction=2e-3):
    """(1) range bit-exact, (u,v) within 1e-3 px of the CPU reference arithmetic; (2) rounding
    flips only within 2e-3 px of a pixel boundary and rare; (3) on the kernel's own (u,v) the
    integer stage is bit-exact; (4) with no flips the whole image is bit-exact vs the oracle."""
    image_o, u_o, v_o, idx_o, i2p_o = orc.project_to_img(cloud[None], h, w, hf, vf)
    uo, vo, rng_o = unsort_uv(cloud, u_o[0], v_o[0])
    image_g, imap_g, u_g, v_g, r_g = gpu_project(cloud, h, w, hf, vf)
    assert torch.equal(r_g, rng_o), "range must be bit-exact (sqrt((x*x+y*y)+z*z), no FMA)"
    fin = torch.isfinite(uo) & torch.isfinite(vo)
    du = (u_g - uo)[fin].abs().max().item()
    dv = (v_g - vo)[fin].abs().max().item()
    assert du < 1e-3 and dv < 1e-3, (du, dv)
    # the kernel's atan2 is SLEEF's algorithm (common.cuh `sleef_atan2f_u10`): bit-identical to torch-CPU
    # except for the < 32 trailing elements that torch (one thread) evaluates with the scalar libm
    mism_u = int(((u_g != uo) & fin).sum())
    mism_v = int(((v_g != vo) & fin).sum())
    print(f"[{label}] float (u,v) not bit-identical to torch-CPU: u {mism_u}, v {mism_v} of {cloud.shape[1]}")
    assert mism_u <= 31 and mism_v <= 31, (mism_u, mism_v)
    flips = ((torch.round(u_g) != torch.round(uo)) | (torch.round(v_g) != torch.round(vo))) & fin
    nflip = int(flips.sum())
    fu = (uo[flips] - torch.floor(uo[flips]) - 0.5).abs()
    fv = (vo[flips] - torch.floor(vo[flips]) - 0.5).abs()
    near = torch.minimum(fu, fv)
    print(f"[{label}] N={cloud.shape[1]} max|du|={du:.2e} max|dv|={dv:.2e} rounding flips={nflip} "
          f"max boundary distance={near.max().item() if nflip else 0:.2e}")
    assert nflip <= max(2, int(max_flip_fraction * cloud.shape[1]))
    if nflip:
        assert near.max().item() < 2e-3
    # integer stage, bit-exact on the kernel's own coordinates
    image_e, _, _, idx_e, i2p_e = orc.project_to_img(cloud[None], h, w, hf, vf, uv_override=(u_g, v_g))
    assert torch.equal(image_g, image_e[0]), "image differs from the oracle's integer stage"
    imap_e = torch.full((h, w), -1, dtype=torch.int32)
    imap_e[i2p_e[0, :, 0], i2p_e[0, :, 1]] = idx_e.to(torch.int32)
    assert torch.equal(imap_g, imap_e), "pixel -> point index map differs"
    if nflip == 0:
        assert torch.equal(image_g, image_o[0])
    else:
        diff = (image_g != image_o[0]).any(dim=0).sum().item()
        assert diff <= 2 * nflip, (diff, nflip)
    return nflip


@pytest.mark.parametrize("name", CASES)
def test_projection(name, golden, cuda_lib):
    meta, cfg, scan_1, scan_2, _, _ = oracle_case(name, golden)
    hf, vf = fov(cfg)
    check_projection(scan_1, meta["H"], meta["W"], hf, vf, name + "/scan_1")
    check_projection(scan_2, meta["H"], meta["W"], hf, vf, name + "/scan_2")


@pytest.mark.parametrize("name", ["edge_16x180", "tie_16x512"])
def test_projection_stress(name, golden, cuda_lib):
    from delora_b200 import synthetic
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    meta = golden[name]
    cfg = synthetic.fov_config(h=meta["H"], w=meta["W"], vfov_deg=tuple(meta["vfov_deg"]))
    hf, vf = fov(cfg)
    cloud = torch.from_numpy(z["cloud"])
    # the edge cloud sits ON the rounding boundaries (k + 0.5 px): flips between SLEEF (CPU torch)
    # and libdevice atan2f are expected there; they must all be boundary points
    check_projection(cloud, meta["H"], meta["W"], hf, vf, name, max_flip_fraction=0.2)


def test_projection_empty_and_ragged_batch(cuda_lib):
    from delora_b200 import ops, synthetic
    cfg = synthetic.fov_config(h=16, w=180, vfov_deg=(-15.0, 15.0))
    hf, vf = fov(cfg)
    a, b, _, _ = synthetic.make_pair(3, w_raw=192, rings=16, vfov_deg=(-15.0, 15.0))
    nmax = max(a.shape[1], b.shape[1]) + 5
    pts = torch.full((3, 3, nmax), float("nan"))
    pts[0, :, :a.shape[1]] = a
    pts[1, :, :b.shape[1]] = b
    n = torch.tensor([a.shape[1], b.shape[1], 0], dtype=torch.int32)
    image, imap = ops.project(pts.to(DEV), n.to(DEV), 16, 180, hf, vf)
    for i, cloud in enumerate((a, b)):
        img_i, imap_i, _, _, _ = gpu_project(cloud, 16, 180, hf, vf)
        assert torch.equal(image[i].cpu(), img_i) and torch.equal(imap[i].cpu(), imap_i)
    assert float(image[2].abs().sum()) == 0.0 and bool((imap[2] == -1).all())
    # the key scratch is re-armed: a second call gives the same answer
    image2, _ = ops.project(pts.to(DEV), n.to(DEV), 16, 180, hf, vf)
    assert torch.equal(image, image2)


def test_projection_matches_torch_cuda_op_sequence(golden, cuda_lib):
    """The reference's default config is device: "cuda".  Run its op sequence (the oracle's torch
    calls) on the GPU and compare: div_mode=1 mirrors torch-CUDA's scalar divide (a * (1/b))."""
    meta, cfg, scan_1, _, _, _ = oracle_case("kitti_64x720", golden)
    hf, vf = fov(cfg)
    image_t, u_t, v_t, idx_t, _ = orc.project_to_img(scan_1[None], meta["H"], meta["W"], hf, vf, device="cuda")
    image_g, _, u_g, v_g, r_g = gpu_project(scan_1, meta["H"], meta["W"], hf, vf, div_mode=1)
    order = torch.argsort(torch.norm(scan_1[None].to(DEV)[:, :3, :], dim=1), dim=1, stable=True)[0].cpu()
    ut = torch.empty_like(u_g)
    vt = torch.empty_like(v_g)
    ut[order] = u_t[0].cpu()
    vt[order] = v_t[0].cpu()
    same_uv = float(((ut == u_g) & (vt == v_g)).float().mean())
    same_img = float((image_t[0].cpu() == image_g).float().mean())
    print(f"[torch-cuda op sequence] identical (u,v): {same_uv:.6f}, identical image entries: {same_img:.6f}")
    # torch-CUDA's own float pipeline differs from torch-CPU's by an ulp in most (u, v) (measured: only
    # ~14 % of the float coordinates are bit-identical), yet the IMAGES agree except at rounding
    # boundaries -- the same statement as for CPU-vs-kernel.  Informational for (u,v); asserted for pixels.
    assert same_img > 0.9995


def test_sort_by_range(golden, cuda_lib):
    from delora_b200 import ops
    meta, cfg, scan_1, scan_2, _, _ = oracle_case("kitti_64x720", golden)
    n1, n2 = scan_1.shape[1], scan_2.shape[1]
    nmax = max(n1, n2)
    rng = torch.zeros((3, nmax))
    rng[0, :n1] = torch.norm(scan_1, dim=0)
    rng[1, :n2] = torch.norm(scan_2, dim=0)
    rng[2, :1000] = torch.randint(0, 7, (1000,)).float()          # heavy ties -> stability matters
    n = torch.tensor([n1, n2, 1000], dtype=torch.int32)
    order = ops.sort_by_range(rng.to(DEV), n.to(DEV)).cpu()
    for i in range(3):
        ref = torch.argsort(rng[i, :n[i]], stable=True)
        assert torch.equal(order[i, :n[i]].long(), ref)


@pytest.mark.parametrize("name", CASES)
def test_normals_and_lists(name, golden, cuda_lib):
    from delora_b200 import ops
    meta, cfg, _, _, _, out = oracle_case(name, golden)
    h, w = meta["H"], meta["W"]
    for k in ("1", "2"):
        image = out["image_" + k]
        nrm_img = ops.normals(image.to(DEV))
        pts4, nrm4, cell_start, counts = ops.lists_from_images(image.to(DEV), nrm_img)
        p = int(counts[0])
        assert p == out["points_" + k].shape[0]
        pts4, nrm4 = pts4[0, :p].cpu(), nrm4[0, :p].cpu()
        assert torch.equal(pts4[:, :3], out["points_" + k]), "point list (row-major valid pixels) must be exact"
        n_o, n_g = out["normals_" + k], nrm4[:, :3]
        has_o = (n_o != 0).any(dim=1)
        assert torch.equal(nrm4[:, 3] != 0, has_o), "has-normal mask (>= 10 gated neighbours) must be exact"
        # cell_start is the exclusive prefix of the valid flags
        valid = (image[0, 0] != 0) & (image[0, 1] != 0) & (image[0, 2] != 0)
        cs = torch.cat((torch.zeros(1, dtype=torch.long), torch.cumsum(valid.reshape(-1).long(), 0)))
        assert torch.equal(cell_start[0].cpu().long(), cs)
        pix = pts4[:, 3].view(torch.int32)
        assert torch.equal(pix.long(), torch.nonzero(valid.reshape(-1))[:, 0])
        # normals: unit length, oriented toward the sensor, close to the reference's LAPACK result
        err = (n_g - n_o).norm(dim=1)[has_o]
        unit = (n_g[has_o].norm(dim=1) - 1).abs().max().item()
        q = torch.quantile(err, torch.tensor([0.5, 0.99, 0.999])).tolist()
        print(f"[{name}/normals_{k}] P={p} with normal={int(has_o.sum())} |dn| median={q[0]:.2e} "
              f"p99={q[1]:.2e} p99.9={q[2]:.2e} max={err.max().item():.2e} unit err={unit:.1e}")
        assert unit < 1e-5
        # measured on B200 (scripts/gpu_normals_stats.py, six image sizes): p99 <= 4.3e-7, max <= 1.14e-5 (at an
        # eigen-gap of 1e-3 of the largest eigenvalue, where LAPACK's own fp32 result is no better determined)
        assert q[1] <= 1e-6, "99% of the normals must agree with the reference's LAPACK result to 1e-6"
        assert err.max().item() <= 5e-5, "every normal within 5e-5"


@pytest.mark.parametrize("name", CASES)
def test_nn_exact_and_losses(name, golden, cuda_lib):
    """Drop-in shape of ICPLosses.forward: already transformed source lists (T = None)."""
    from delora_b200 import ops
    meta, cfg, _, _, t_pred, out = oracle_case(name, golden)
    h, w = meta["H"], meta["W"]
    hf, vf = fov(cfg)
    tm = t_pred.view(1, 4, 4)
    src = orc.transform_point_cloud(tm, out["points_2"].t()[None]).contiguous()
    src_n = orc.rotate_point_cloud(tm, out["normals_2"].t()[None]).contiguous()
    tgt, tgt_n = out["points_1"].t()[None].contiguous(), out["normals_1"].t()[None].contiguous()
    losses_o, aux = orc.icp_losses(src, src_n, tgt, tgt_n, return_aux=True)
    ns = torch.tensor([src.shape[2]], dtype=torch.int32, device=DEV)
    nt = torch.tensor([tgt.shape[2]], dtype=torch.int32, device=DEV)
    s4, sn4 = ops.pack_lists(src.to(DEV), src_n.to(DEV), ns)
    t4, tn4, cs = ops.grid_build(tgt.to(DEV), tgt_n.to(DEV), nt, h, w, hf, vf)
    losses, grad_t, nn_index, pdir, ndir = ops.icp_fwd_bwd(s4, sn4, ns, None, t4, tn4, cs, h, w, hf, vf,
                                                           pointwise=True)
    nn_g = nn_index[0].cpu().long()
    mism = int((nn_g != aux["nn_index"]).sum())
    print(f"[{name}] NN mismatches vs cKDTree: {mism} of {nn_g.shape[0]}")
    assert mism == 0, "nearest neighbours must be the exact float64 NN"
    row = losses[0].cpu()
    assert int(row[3]) == aux["num_pairs"]
    rel_pl = abs(row[1].item() - float(losses_o["loss_po2pl"])) / float(losses_o["loss_po2pl"])
    rel_nn = abs(row[2].item() - float(losses_o["loss_pl2pl"])) / float(losses_o["loss_pl2pl"])
    print(f"[{name}] loss rel err po2pl={rel_pl:.2e} pl2pl={rel_nn:.2e}")
    assert rel_pl < 1e-5 and rel_nn < 1e-5
    # per-point gradients for the autograd path
    srcg = src.clone().requires_grad_(True)
    srcng = src_n.clone().requires_grad_(True)
    lo = orc.icp_losses(srcg, srcng, tgt, tgt_n)
    (lo["loss_po2pl"] + lo["loss_pl2pl"]).sum().backward()
    up = torch.tensor([[0.0, 1.0, 1.0]], device=DEV)
    gp, gn = ops.icp_point_grads(pdir, ndir, ns, losses, up)
    assert torch.allclose(gp[0].cpu(), srcg.grad[0], rtol=1e-4, atol=1e-9)
    assert torch.allclose(gn[0].cpu(), srcng.grad[0], rtol=1e-4, atol=1e-9)


@pytest.mark.parametrize("name", CASES)
def test_pair_pipeline_end_to_end(name, golden, cuda_lib):
    """Raw scans -> losses + dL/dT through the batched pipeline vs the oracle / reference golden."""
    from delora_b200.pipeline import ScanPairPipeline
    meta, cfg, scan_1, scan_2, t_pred, out = oracle_case(name, golden)
    hf, vf = fov(cfg)
    B = 2                                               # the same pair twice + ragged padding
    nmax = max(scan_1.shape[1], scan_2.shape[1]) + 7
    pipe = ScanPairPipeline(B, nmax, meta["H"], meta["W"], hf, vf, device=DEV)
    pipe.load([scan_1, scan_1], [scan_2, scan_2], torch.stack((t_pred, t_pred)))
    losses, grad_t = pipe.step()
    torch.cuda.synchronize()
    losses, grad_t = losses.cpu(), grad_t.cpu()
    assert torch.equal(losses[0], losses[1]) and torch.equal(grad_t[0], grad_t[1]), "deterministic per pair"
    g_ref = np.asarray(meta["grad_T"], dtype=np.float64)
    rel_pl = abs(losses[0, 1].item() - meta["loss_po2pl"]) / meta["loss_po2pl"]
    rel_nn = abs(losses[0, 2].item() - meta["loss_pl2pl"]) / meta["loss_pl2pl"]
    gerr = np.abs(grad_t[0].numpy().reshape(3, 4) - g_ref).max() / np.abs(g_ref).max()
    print(f"[{name}] end-to-end vs reference golden: po2pl rel={rel_pl:.2e} pl2pl rel={rel_nn:.2e} "
          f"grad_T rel(max)={gerr:.2e} pairs={int(losses[0, 3])} (ref {meta['num_pairs']})")
    # with the SLEEF-exact atan2 the projection reproduces the CPU reference's pixels, so the whole chain
    # meets the 1e-5 bar against the REFERENCE's own numbers (not only against the oracle on equal inputs)
    assert int(losses[0, 3]) == meta["num_pairs"]
    assert rel_pl < 1e-5 and rel_nn < 1e-5 and gerr < 1e-5


def test_pair_pipeline_sub_batches_on_streams_are_bit_identical(golden, cuda_lib):
    """`concurrency` > 1 runs sub-batches of pairs on their own streams (forked from / joined into the caller's stream):
    5 different pairs, uneven splits, two consecutive steps -- every output buffer equals the single-stream run."""
    from delora_b200 import synthetic
    from delora_b200.pipeline import ScanPairPipeline
    h, w = 16, 180
    vf = (-15.0, 15.0)
    cfg = synthetic.fov_config(h=h, w=w, vfov_deg=vf)
    hf, vfr = cfg["horizontal_field_of_view"], cfg["kitti"]["vertical_field_of_view"]
    pairs = [synthetic.make_pair(20 + i, w_raw=192, rings=16, vfov_deg=vf) for i in range(5)]
    nmax = max(max(p[0].shape[1], p[1].shape[1]) for p in pairs) + 3
    outs = []
    for conc in (1, 2, 3, 5, None):
        pipe = ScanPairPipeline(5, nmax, h, w, hf, vfr, device=DEV, concurrency=conc)
        assert pipe.concurrency == (conc if conc is not None else 2)
        pipe.load([p[0] for p in pairs], [p[1] for p in pairs], torch.stack([p[3] for p in pairs]))
        for _ in range(2):
            losses, grad_t = pipe.step()
        torch.cuda.synchronize()
        outs.append([t.clone() for t in (losses, grad_t, pipe.image, pipe.index_map, pipe.pts_grid, pipe.nrm_grid)])
        assert (pipe.keys == -1).all(), "key buffer re-armed"
    for other in outs[1:]:
        for a, b in zip(outs[0], other):
            assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert float(outs[0][0][:, 3].min()) > 100                          # every pair found correspondences


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path, cuda_lib):
    """`bench.py --dump-outputs DIR`: the losses and transform gradients of the last timed step, bit for bit what the
    pipeline returns for the same seeded pairs (one input set, so every step sees pairs 0..7)."""
    import json
    import subprocess
    import sys
    from delora_b200 import synthetic
    from delora_b200.pipeline import ScanPairPipeline
    from helpers import ROOT
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--rotate", "1",
                          "--cpu-pairs", "0", "--train-steps", "0", "--stream-frames", "0",
                          "--dump-outputs", str(tmp_path / "dump")], capture_output=True, text=True, timeout=900, check=True)
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3
    losses, grad_t = np.load(tmp_path / "dump" / "losses.npy"), np.load(tmp_path / "dump" / "grad_T.npy")
    assert losses.dtype == np.float32 and losses.shape == (8, 8) and grad_t.dtype == np.float32 and grad_t.shape == (8, 12)
    cfg = synthetic.fov_config(h=64, w=2048)
    pairs = [synthetic.make_pair(i, w_raw=2048) for i in range(8)]
    n_max = max(max(p[0].shape[1], p[1].shape[1]) for p in pairs)
    pipe = ScanPairPipeline(8, n_max, 64, 2048, *fov(cfg), device=DEV)
    pipe.load([p[0] for p in pairs], [p[1] for p in pairs], torch.stack([p[3] for p in pairs]))
    want_losses, want_grad = pipe.step()
    assert np.array_equal(losses, want_losses.cpu().numpy()) and np.array_equal(grad_t, want_grad.cpu().numpy())
    assert float(losses[:, 3].min()) > 1000                               # every pair found correspondences


@pytest.mark.parametrize("name", CASES)
def test_dense_icp_matches_list_icp(name, golden, cuda_lib):
    """The dense-grid kernel (training fast path) against the oracle and against the CSR kernel."""
    from delora_b200 import ops
    meta, cfg, _, _, t_pred, out = oracle_case(name, golden)
    h, w = meta["H"], meta["W"]
    hf, vf = fov(cfg)
    images = torch.cat((out["image_1"], out["image_2"])).to(DEV)
    _, pg, ng = ops.normals(images, grids=True)
    T = t_pred[:3, :].reshape(1, 12).contiguous().to(DEV)
    losses, grad_t = ops.icp_dense_fwd_bwd(pg[1:2].contiguous(), ng[1:2].contiguous(), T, pg[0:1].contiguous(),
                                           ng[0:1].contiguous(), h, w, hf, vf)
    # the oracle on the oracle's lists (normals differ at the 1e-7 level, so not bit-identical)
    row = losses[0].cpu()
    assert int(row[3]) == out["num_pairs"]
    assert row[1].item() == pytest.approx(out["loss_po2pl"], rel=1e-5)
    assert row[2].item() == pytest.approx(out["loss_pl2pl"], rel=1e-5)
    g_ref = out["grad_T"].numpy()
    assert np.abs(grad_t[0].cpu().numpy().reshape(3, 4) - g_ref).max() <= 1e-5 * np.abs(g_ref).max()
    # CSR kernel on the lists of the same images: same pair count, same sums up to summation order
    nrm_img = ops.normals(images)
    pts4, nrm4, cs, counts = ops.lists_from_images(images, nrm_img)
    l2, g2, _, _, _ = ops.icp_fwd_bwd(pts4[1:2].contiguous(), nrm4[1:2].contiguous(), counts[1:2].contiguous(), T,
                                      pts4[0:1].contiguous(), nrm4[0:1].contiguous(), cs[0:1].contiguous(), h, w,
                                      hf, vf)
    assert float(l2[0, 3]) == float(row[3])
    assert torch.allclose(l2[0, :3].cpu(), row[:3], rtol=2e-6, atol=0)
    assert torch.allclose(g2.cpu(), grad_t.cpu(), rtol=1e-4, atol=1e-9)
    # empty / invalid pixels of the dense grids
    assert bool(((pg[:, :, 3].view(torch.int32) >= 0) == ((images[:, 0] != 0) & (images[:, 1] != 0)
                                                          & (images[:, 2] != 0)).reshape(2, -1)).all())


@pytest.mark.parametrize("name,dx,yaw_deg", [("kitti_64x720", 1.5, 4.0), ("small_16x180", 0.8, 10.0),
                                             ("kitti_64x2048", 0.6, 1.5),
                                             # re-projections that cross the +-180 deg seam; W = 180 is not a
                                             # multiple of the 16-column range blocks (ragged last block column)
                                             ("small_16x180", 0.5, 178.0), ("small_16x180", 2.0, -95.0),
                                             ("kitti_64x720", 0.3, 181.0)])
def test_dense_icp_large_misalignment(name, dx, yaw_deg, golden, cuda_lib):
    """A poor transform (untrained network): NN distances of ~1 m force the range-pruned block search.
    The dense kernel must still return the exact NN statistics: same pair count and sums as the CSR kernel
    (independent search code) and as the oracle (cKDTree)."""
    from delora_b200 import ops, synthetic
    meta, cfg, _, _, _, out = oracle_case(name, golden)
    h, w = meta["H"], meta["W"]
    hf, vf = fov(cfg)
    t_bad = synthetic.transform_matrix(dx, -0.3, 0.1, math.radians(yaw_deg), math.radians(1.0), 0.0)
    t_bad = torch.from_numpy(t_bad).float()
    images = torch.cat((out["image_1"], out["image_2"])).to(DEV)
    nrm_img, pg, ng = ops.normals(images, grids=True)
    T = t_bad[:3, :].reshape(1, 12).contiguous().to(DEV)
    losses, grad_t = ops.icp_dense_fwd_bwd(pg[1:2].contiguous(), ng[1:2].contiguous(), T, pg[0:1].contiguous(),
                                           ng[0:1].contiguous(), h, w, hf, vf)
    pts4, nrm4, cs, counts = ops.lists_from_images(images, nrm_img)
    l2, g2, _, _, _ = ops.icp_fwd_bwd(pts4[1:2].contiguous(), nrm4[1:2].contiguous(), counts[1:2].contiguous(), T,
                                      pts4[0:1].contiguous(), nrm4[0:1].contiguous(), cs[0:1].contiguous(), h, w,
                                      hf, vf)
    assert float(l2[0, 3]) == float(losses[0, 3])
    assert torch.allclose(l2[0, :3].cpu(), losses[0, :3].cpu(), rtol=2e-6, atol=0)
    assert torch.allclose(g2.cpu(), grad_t.cpu(), rtol=1e-4, atol=1e-7)
    if name != "kitti_64x2048":          # oracle (cKDTree) cross-check on the smaller cases
        tm = t_bad.view(1, 4, 4)
        # same normals as the kernel so that only the search differs
        p1, n1 = pts4[0, :int(counts[0]), :3].cpu(), nrm4[0, :int(counts[0]), :3].cpu()
        p2, n2 = pts4[1, :int(counts[1]), :3].cpu(), nrm4[1, :int(counts[1]), :3].cpu()
        lo, aux = orc.icp_losses(orc.transform_point_cloud(tm, p2.t()[None]), orc.rotate_point_cloud(tm, n2.t()[None]),
                                 p1.t()[None].contiguous(), n1.t()[None].contiguous(), return_aux=True)
        assert aux["num_pairs"] == int(losses[0, 3])
        assert float(losses[0, 1]) == pytest.approx(float(lo["loss_po2pl"]), rel=1e-5)
        assert float(losses[0, 2]) == pytest.approx(float(lo["loss_pl2pl"]), rel=1e-5)


@pytest.mark.parametrize("name,n_transforms", [("small_16x180", 12), ("kitti_64x720", 4)])
def test_dense_icp_arbitrary_transforms_vs_kdtree(name, n_transforms, golden, cuda_lib):
    """Untrained-network regime: arbitrary rotations (any axis, up to 180 deg) and translations of metres.
    Sources re-project anywhere (across the seam, outside the vertical FOV); the strip search gives up
    and the range-pruned block search takes over.  Exactness is checked against cKDTree (oracle)."""
    from delora_b200 import ops
    meta, cfg, _, _, _, out = oracle_case(name, golden)
    h, w = meta["H"], meta["W"]
    hf, vf = fov(cfg)
    images = torch.cat((out["image_1"], out["image_2"])).to(DEV)
    nrm_img, pg, ng = ops.normals(images, grids=True)
    pts4, nrm4, cs, counts = ops.lists_from_images(images, nrm_img)
    p1, n1 = pts4[0, :int(counts[0]), :3].cpu(), nrm4[0, :int(counts[0]), :3].cpu()
    p2, n2 = pts4[1, :int(counts[1]), :3].cpu(), nrm4[1, :int(counts[1]), :3].cpu()
    gen = torch.Generator().manual_seed(77)
    for k in range(n_transforms):
        axis = torch.randn(3, generator=gen)
        axis = axis / axis.norm()
        ang = float(torch.rand(1, generator=gen)) * math.pi * (1.0 if k % 3 else 0.1)
        kx = torch.tensor([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
        rot = torch.eye(3) + math.sin(ang) * kx + (1 - math.cos(ang)) * (kx @ kx)
        tm = torch.eye(4)
        tm[:3, :3] = rot
        tm[:3, 3] = (torch.rand(3, generator=gen) - 0.5) * torch.tensor([16.0, 16.0, 2.0]) * (1.0 if k % 2 else 0.1)
        T = tm[:3, :].reshape(1, 12).contiguous().to(DEV)
        losses, _ = ops.icp_dense_fwd_bwd(pg[1:2].contiguous(), ng[1:2].contiguous(), T, pg[0:1].contiguous(),
                                          ng[0:1].contiguous(), h, w, hf, vf)
        t4 = tm.view(1, 4, 4)
        lo, aux = orc.icp_losses(orc.transform_point_cloud(t4, p2.t()[None]), orc.rotate_point_cloud(t4, n2.t()[None]),
                                 p1.t()[None].contiguous(), n1.t()[None].contiguous(), return_aux=True)
        assert aux["num_pairs"] == int(losses[0, 3]), (k, ang, tm[:3, 3])
        assert float(losses[0, 1]) == pytest.approx(float(lo["loss_po2pl"]), rel=2e-5), (k, ang, tm[:3, 3])
        assert float(losses[0, 2]) == pytest.approx(float(lo["loss_pl2pl"]), rel=2e-5), (k, ang, tm[:3, 3])


def test_dense_icp_handover_limit_and_determinism(golden, cuda_lib, monkeypatch):
    """The two-kernel split is an implementation detail: any hand-over limit (DELORA_ICP_MAX_STRIPS) must give the
    same pairs and, up to fp32 summation order, the same losses / gradient; and for a fixed limit repeated calls are
    BIT-identical although the work list of the second kernel is appended by atomics in arbitrary order."""
    from delora_b200 import ops, synthetic
    meta, cfg, _, _, _, out = oracle_case("kitti_64x720", golden)
    h, w = meta["H"], meta["W"]
    hf, vf = fov(cfg)
    images = torch.cat((out["image_1"], out["image_2"])).to(DEV)
    _, pg, ng = ops.normals(images, grids=True)
    t = torch.from_numpy(synthetic.transform_matrix(0.6, -0.2, 0.05, math.radians(2.0), 0.0, 0.0)).float()
    T = t[:3, :].reshape(1, 12).contiguous().to(DEV)
    scratch = ops.icp_scratch(1, h * w, DEV)

    def run():
        losses, grad = ops.icp_dense_fwd_bwd(pg[1:2].contiguous(), ng[1:2].contiguous(), T, pg[0:1].contiguous(),
                                             ng[0:1].contiguous(), h, w, hf, vf, scratch=scratch)
        return losses.cpu().clone(), grad.cpu().clone()

    base = run()
    for _ in range(3):
        again = run()
        assert torch.equal(again[0], base[0]) and torch.equal(again[1], base[1])
    for limit in ("0", "3", "100000"):
        monkeypatch.setenv("DELORA_ICP_MAX_STRIPS", limit)
        losses, grad = run()
        assert float(losses[0, 3]) == float(base[0][0, 3]), limit
        assert torch.allclose(losses[0, :3], base[0][0, :3], rtol=2e-6, atol=0), limit
        assert torch.allclose(grad, base[1], rtol=1e-4, atol=1e-8), limit
    monkeypatch.delenv("DELORA_ICP_MAX_STRIPS")


def test_generic_lists_shuffled_and_po2po(golden, cuda_lib):
    """Arbitrary (shuffled, with out-of-FOV points) lists through delora_grid_build; po2po on."""
    from delora_b200 import ops
    meta, cfg, _, _, t_pred, out = oracle_case("small_16x180", golden)
    h, w = meta["H"], meta["W"]
    hf, vf = fov(cfg)
    g = torch.Generator().manual_seed(11)
    tm = t_pred.view(1, 4, 4)
    src = orc.transform_point_cloud(tm, out["points_2"].t()[None])
    src_n = orc.rotate_point_cloud(tm, out["normals_2"].t()[None])
    tgt, tgt_n = out["points_1"].t()[None], out["normals_1"].t()[None]
    extra = torch.tensor([[0.5, -0.2, 6.0], [0.1, 0.1, -7.0], [-9.0, 1e-3, 0.3]]).t()[None]   # outside the FOV / seam
    tgt = torch.cat((tgt, extra), dim=2)
    tgt_n = torch.cat((tgt_n, torch.zeros_like(extra)), dim=2)
    perm = torch.randperm(tgt.shape[2], generator=g)
    tgt, tgt_n = tgt[:, :, perm].contiguous(), tgt_n[:, :, perm].contiguous()
    src = torch.cat((src, extra * 1.01), dim=2).contiguous()
    src_n = torch.cat((src_n, torch.zeros_like(extra)), dim=2).contiguous()
    lo, aux = orc.icp_losses(src, src_n, tgt, tgt_n, point_to_point_loss=True, nn_method="brute", return_aux=True)
    ns = torch.tensor([src.shape[2]], dtype=torch.int32, device=DEV)
    nt = torch.tensor([tgt.shape[2]], dtype=torch.int32, device=DEV)
    s4, sn4 = ops.pack_lists(src.to(DEV), src_n.to(DEV), ns)
    t4, tn4, cs = ops.grid_build(tgt.to(DEV), tgt_n.to(DEV), nt, h, w, hf, vf)
    losses, _, nn_index, _, _ = ops.icp_fwd_bwd(s4, sn4, ns, None, t4, tn4, cs, h, w, hf, vf, pointwise=True,
                                                flags=ops.LOSS_PO2PO | ops.LOSS_PO2PL | ops.LOSS_PL2PL)
    assert torch.equal(nn_index[0].cpu().long(), aux["nn_index"])
    row = losses[0].cpu()
    for j, key in ((0, "loss_po2po"), (1, "loss_po2pl"), (2, "loss_pl2pl")):
        assert row[j].item() == pytest.approx(float(lo[key]), rel=1e-5), key
    # "linear" normal loss
    lo2 = orc.icp_losses(src, src_n, tgt, tgt_n, normal_loss="linear", nn_method="brute")
    losses2, _, _, _, _ = ops.icp_fwd_bwd(s4, sn4, ns, None, t4, tn4, cs, h, w, hf, vf,
                                          flags=ops.LOSS_PO2PL | ops.LOSS_PL2PL | ops.NORMAL_LINEAR)
    assert losses2[0, 2].item() == pytest.approx(float(lo2["loss_pl2pl"]), rel=1e-5)


def test_nn_far_and_empty_targets(cuda_lib):
    """Guard failures must widen to the exhaustive search: sources far from every target."""
    from delora_b200 import ops, synthetic
    cfg = synthetic.fov_config(h=16, w=180, vfov_deg=(-15.0, 15.0))
    hf, vf = fov(cfg)
    g = torch.Generator().manual_seed(5)
    tgt = (torch.randn(1, 3, 300, generator=g) * torch.tensor([8.0, 8.0, 1.0]).view(1, 3, 1)).contiguous()
    src = (torch.randn(1, 3, 500, generator=g) * torch.tensor([20.0, 20.0, 6.0]).view(1, 3, 1)).contiguous()
    zeros_t, zeros_s = torch.zeros_like(tgt), torch.zeros_like(src)
    ref = torch.from_numpy(orc.nearest_neighbors(tgt[0].t().numpy(), src[0].t().numpy(), "brute"))
    ns = torch.tensor([500], dtype=torch.int32, device=DEV)
    nt = torch.tensor([300], dtype=torch.int32, device=DEV)
    s4, sn4 = ops.pack_lists(src.to(DEV), zeros_s.to(DEV), ns)
    t4, tn4, cs = ops.grid_build(tgt.to(DEV), zeros_t.to(DEV), nt, 16, 180, hf, vf)
    _, _, nn_index, _, _ = ops.icp_fwd_bwd(s4, sn4, ns, None, t4, tn4, cs, 16, 180, hf, vf, pointwise=True)
    assert torch.equal(nn_index[0].cpu().long(), ref)
    # empty target list: every pair is dropped, losses are 0, nothing hangs
    nt0 = torch.tensor([0], dtype=torch.int32, device=DEV)
    t4, tn4, cs = ops.grid_build(tgt.to(DEV), zeros_t.to(DEV), nt0, 16, 180, hf, vf)
    losses, _, nn_index, _, _ = ops.icp_fwd_bwd(s4, sn4, ns, None, t4, tn4, cs, 16, 180, hf, vf, pointwise=True)
    assert bool((nn_index == -1).all()) and float(losses[0, 3]) == 0.0


def test_quat_to_T_forward_backward(cuda_lib):
    from delora_b200 import ops
    z = np.load(os.path.join(GOLDEN, "quaternion.npz"))
    q, t = torch.from_numpy(z["quaternion"]), torch.from_numpy(z["translation"])
    T = ops.quat_to_T(q.to(DEV), t.to(DEV)).cpu()
    assert np.abs(T.numpy() - z["T"]).max() < 5e-7
    qg = q.clone().requires_grad_(True)
    tg = t.clone().requires_grad_(True)
    To = orc.transformation_matrix_quaternion(tg, qg)
    w = torch.randn(16, 4, 4, generator=torch.Generator().manual_seed(3))
    (To * w).sum().backward()
    gq, gt = ops.quat_to_T_bwd(q.to(DEV), w.to(DEV).contiguous())
    assert torch.allclose(gq.cpu(), qg.grad, rtol=1e-4, atol=1e-6)
    assert torch.allclose(gt.cpu(), tg.grad, rtol=1e-6, atol=1e-7)


def test_missing_library_fails_loudly(monkeypatch):
    from delora_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libdelora_b200.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.lib()
