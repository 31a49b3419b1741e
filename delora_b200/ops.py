"""Tensor-level wrappers over the C ABI: one call = one operator over a whole batch.

Every function takes CUDA tensors, allocates its outputs with torch (device memory is the
plumbing torch provides), passes raw pointers + the current stream to libdelora_b200.so and
returns tensors.  Nothing here computes on the host and nothing falls back to torch ops.
"""
import os

import torch

from . import _lib

# NVTX ranges around the operators (SURVEY.md section 5, tracing): DELORA_NVTX=1 names the phases of a step for
# nsys / ncu --nvtx; off by default (no push / pop calls at all on the hot path).
NVTX = os.environ.get("DELORA_NVTX") == "1"


class nvtx_range:
    """`with ops.nvtx_range("normals"):` -- an NVTX range when DELORA_NVTX=1, otherwise nothing."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if NVTX:
            torch.cuda.nvtx.range_push(self.name)
        return self

    def __exit__(self, *exc):
        if NVTX:
            torch.cuda.nvtx.range_pop()
        return False


LOSS_PO2PO, LOSS_PO2PL, LOSS_PL2PL, NORMAL_LINEAR = 1, 2, 4, 8
LOSS_ROW, ICP_PARTIAL = 8, 40

_keys_cache = {}


_last_device = [None]


def _stream():
    """The current stream of the device the operands live on (`_req` records it: with several devices in one process
    torch's *current device* need not be the tensors' device) -- the kernels are launched on that device's stream."""
    dev = _last_device[0]
    return torch.cuda.current_stream(dev).cuda_stream


def _req(t, dtype, name):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.is_contiguous()):
        raise ValueError(f"{name}: expected a contiguous CUDA tensor of dtype {dtype}, got "
                         f"{getattr(t, 'dtype', type(t))} on {getattr(t, 'device', '?')}")
    if _last_device[0] != t.device:
        _last_device[0] = t.device
        if torch.cuda.current_device() != t.device.index:      # the C ABI launches on the CURRENT device
            torch.cuda.set_device(t.device)
    return t.data_ptr()


def _keys(device, b, hw):
    """All-ones uint64 key scratch; delora_project_fwd leaves it all-ones again."""
    k = (device.index, b, hw)
    buf = _keys_cache.get(k)
    if buf is None:
        buf = torch.full((b, hw), -1, dtype=torch.int64, device=device)
        _keys_cache[k] = buf
    return buf


def project(points, n_points, h, w, hfov, vfov, div_mode=0):
    """points [B,C,N] fp32, n_points [B] int32 -> image [B,C+1,H,W], index_map [B,H,W] int32.
    (src/utility/projection.py:48-106)"""
    b, c, n = points.shape
    image = torch.empty((b, c + 1, h, w), dtype=torch.float32, device=points.device)
    index_map = torch.empty((b, h, w), dtype=torch.int32, device=points.device)
    keys = _keys(points.device, b, h * w)
    L = _lib.lib()
    _lib.check(L.delora_project_fwd(_req(points, torch.float32, "points"), _req(n_points, torch.int32, "n_points"),
                                    b, c, n, h, w, float(hfov[0]), float(hfov[1]), float(vfov[0]), float(vfov[1]),
                                    int(div_mode), keys.data_ptr(), image.data_ptr(), index_map.data_ptr(),
                                    _stream()), "delora_project_fwd")
    return image, index_map


def project_uv(points, n_points, h, w, hfov, vfov, div_mode=0):
    """(u, v, range) of every point in the original order: three [B,N] fp32 tensors."""
    b, c, n = points.shape
    u = torch.zeros((b, n), dtype=torch.float32, device=points.device)
    v = torch.zeros_like(u)
    r = torch.zeros_like(u)
    L = _lib.lib()
    _lib.check(L.delora_project_uv(_req(points, torch.float32, "points"), _req(n_points, torch.int32, "n_points"),
                                   b, c, n, h, w, float(hfov[0]), float(hfov[1]), float(vfov[0]), float(vfov[1]),
                                   int(div_mode), u.data_ptr(), v.data_ptr(), r.data_ptr(), _stream()),
               "delora_project_uv")
    return u, v, r


def sort_by_range(rng, n_points):
    """rng [B,N] fp32 -> order [B,N] int32: indices in ascending (range, index) order."""
    b, n = rng.shape
    L = _lib.lib()
    order = torch.empty((b, n), dtype=torch.int32, device=rng.device)
    scratch = torch.empty((int(L.delora_sort_scratch_bytes(b, n)),), dtype=torch.uint8, device=rng.device)
    _lib.check(L.delora_sort_by_range(_req(rng, torch.float32, "range"), _req(n_points, torch.int32, "n_points"),
                                      b, n, order.data_ptr(), scratch.data_ptr(), _stream()), "delora_sort_by_range")
    return order


def normals(image, neighborhood=(7, 11), epsilon_range=0.5, min_neighbors=10, grids=False):
    """image [B,C,H,W] -> normals [B,3,H,W] (src/preprocessing/normal_computation.py:89-122).
    grids=True additionally returns the dense float4 grids (pts_grid, nrm_grid) [B,HW,4]."""
    b, c, h, w = image.shape
    out = torch.empty((b, 3, h, w), dtype=torch.float32, device=image.device)
    pg = ng = None
    if grids:
        pg = torch.empty((b, h * w, 4), dtype=torch.float32, device=image.device)
        ng = torch.empty((b, h * w, 4), dtype=torch.float32, device=image.device)
    L = _lib.lib()
    _lib.check(L.delora_normals_fwd(_req(image, torch.float32, "image"), b, c, h, w, int(neighborhood[0]),
                                    int(neighborhood[1]), float(epsilon_range), int(min_neighbors),
                                    out.data_ptr(), pg.data_ptr() if grids else None,
                                    ng.data_ptr() if grids else None, _stream()), "delora_normals_fwd")
    return (out, pg, ng) if grids else out


def lists_from_images(image, normals_img):
    """-> pts4 [B,HW,4], nrm4 [B,HW,4], cell_start [B,HW+1] int32, counts [B] int32."""
    b, c, h, w = image.shape
    hw = h * w
    dev = image.device
    pts4 = torch.empty((b, hw, 4), dtype=torch.float32, device=dev)
    nrm4 = torch.empty((b, hw, 4), dtype=torch.float32, device=dev)
    cell_start = torch.empty((b, hw + 1), dtype=torch.int32, device=dev)
    counts = torch.empty((b,), dtype=torch.int32, device=dev)
    L = _lib.lib()
    scratch = torch.empty((b * L.delora_scan_blocks(hw),), dtype=torch.int32, device=dev)
    _lib.check(L.delora_lists_from_images(_req(image, torch.float32, "image"),
                                          _req(normals_img, torch.float32, "normals"), b, c, h, w,
                                          pts4.data_ptr(), nrm4.data_ptr(), cell_start.data_ptr(),
                                          counts.data_ptr(), scratch.data_ptr(), _stream()),
               "delora_lists_from_images")
    return pts4, nrm4, cell_start, counts


def grid_build(pts, nrm, n, h, w, hfov, vfov):
    """pts, nrm [B,3,N] channels-first lists, n [B] int32 -> cell-sorted pts4, nrm4 [B,N,4], cell_start."""
    b, _, ns = pts.shape
    hw = h * w
    dev = pts.device
    pts4 = torch.empty((b, ns, 4), dtype=torch.float32, device=dev)
    nrm4 = torch.empty((b, ns, 4), dtype=torch.float32, device=dev)
    cell_start = torch.empty((b, hw + 1), dtype=torch.int32, device=dev)
    cursor = torch.empty((b, hw), dtype=torch.int32, device=dev)
    L = _lib.lib()
    scratch = torch.empty((b * L.delora_scan_blocks(hw),), dtype=torch.int32, device=dev)
    _lib.check(L.delora_grid_build(_req(pts, torch.float32, "pts"),
                                   _req(nrm, torch.float32, "nrm") if nrm is not None else None,
                                   _req(n, torch.int32, "n"), b, ns, h, w, float(hfov[0]), float(hfov[1]),
                                   float(vfov[0]), float(vfov[1]), pts4.data_ptr(), nrm4.data_ptr(),
                                   cell_start.data_ptr(), cursor.data_ptr(), scratch.data_ptr(), _stream()),
               "delora_grid_build")
    return pts4, nrm4, cell_start


def grids_from_projection(points, normal_lists, index_map):
    """points [B,C,N], normal_lists [B,3,N], index_map [B,H,W] int32 -> pts_grid, nrm_grid [B,HW,4]."""
    b, c, n = points.shape
    _, h, w = index_map.shape
    pg = torch.empty((b, h * w, 4), dtype=torch.float32, device=points.device)
    ng = torch.empty((b, h * w, 4), dtype=torch.float32, device=points.device)
    L = _lib.lib()
    _lib.check(L.delora_grids_from_projection(_req(points, torch.float32, "points"),
                                              _req(normal_lists, torch.float32, "normal_lists"),
                                              _req(index_map, torch.int32, "index_map"), b, c, n, h, w,
                                              pg.data_ptr(), ng.data_ptr(), _stream()),
               "delora_grids_from_projection")
    return pg, ng


def pack_lists(pts, nrm, n):
    b, _, ns = pts.shape
    pts4 = torch.empty((b, ns, 4), dtype=torch.float32, device=pts.device)
    nrm4 = torch.empty((b, ns, 4), dtype=torch.float32, device=pts.device)
    L = _lib.lib()
    _lib.check(L.delora_pack_lists(_req(pts, torch.float32, "pts"),
                                   _req(nrm, torch.float32, "nrm") if nrm is not None else None,
                                   _req(n, torch.int32, "n"), b, ns, pts4.data_ptr(), nrm4.data_ptr(), _stream()),
               "delora_pack_lists")
    return pts4, nrm4


def icp_fwd_bwd(src_pts4, src_nrm4, n_src, transform, tgt_pts4, tgt_nrm4, cell_start, h, w, hfov, vfov,
                lambda_po2pl=1.0, flags=LOSS_PO2PL | LOSS_PL2PL, pointwise=False, scratch=None):
    """Fused transform + exact NN + losses + gradient.  transform: [B,12] (3x4 row-major) or None.
    -> losses [B,8], grad_T [B,12], (nn_index [B,Ns] int32, point_dir, normal_dir [B,Ns,4]) or Nones."""
    b, ns, _ = src_pts4.shape
    nt = tgt_pts4.shape[1]
    dev = src_pts4.device
    L = _lib.lib()
    losses = torch.empty((b, LOSS_ROW), dtype=torch.float32, device=dev)
    grad_t = torch.empty((b, 12), dtype=torch.float32, device=dev)
    if scratch is None:
        scratch = icp_scratch(b, ns, dev)
    nn_index = point_dir = normal_dir = None
    if pointwise:
        nn_index = torch.empty((b, ns), dtype=torch.int32, device=dev)
        point_dir = torch.empty((b, ns, 4), dtype=torch.float32, device=dev)
        normal_dir = torch.empty((b, ns, 4), dtype=torch.float32, device=dev)
    _lib.check(L.delora_icp_fwd_bwd(
        _req(src_pts4, torch.float32, "src_pts4"), _req(src_nrm4, torch.float32, "src_nrm4"),
        _req(n_src, torch.int32, "n_src"), ns,
        _req(transform, torch.float32, "transform") if transform is not None else None,
        _req(tgt_pts4, torch.float32, "tgt_pts4"), _req(tgt_nrm4, torch.float32, "tgt_nrm4"),
        _req(cell_start, torch.int32, "cell_start"), nt, b, h, w,
        float(hfov[0]), float(hfov[1]), float(vfov[0]), float(vfov[1]), float(lambda_po2pl), int(flags),
        losses.data_ptr(), grad_t.data_ptr(),
        nn_index.data_ptr() if pointwise else None, point_dir.data_ptr() if pointwise else None,
        normal_dir.data_ptr() if pointwise else None, scratch.data_ptr(), _stream()), "delora_icp_fwd_bwd")
    return losses, grad_t, nn_index, point_dir, normal_dir


def icp_scratch(b, src_stride, device):
    """Zero-initialised scratch for the ICP kernels (they leave its counters at zero)."""
    return torch.zeros((int(_lib.lib().delora_icp_scratch_floats(b, src_stride)),), dtype=torch.float32,
                       device=device)


def icp_dense_fwd_bwd(src_grid, src_ngrid, transform, tgt_grid, tgt_ngrid, h, w, hfov, vfov, lambda_po2pl=1.0,
                      flags=LOSS_PO2PL | LOSS_PL2PL, scratch=None):
    """Dense-grid variant: grids [B,HW,4] from normals(grids=True); transform [B,12]."""
    b = src_grid.shape[0]
    dev = src_grid.device
    losses = torch.empty((b, LOSS_ROW), dtype=torch.float32, device=dev)
    grad_t = torch.empty((b, 12), dtype=torch.float32, device=dev)
    if scratch is None:
        scratch = icp_scratch(b, h * w, dev)
    L = _lib.lib()
    _lib.check(L.delora_icp_dense_fwd_bwd(
        _req(src_grid, torch.float32, "src_grid"), _req(src_ngrid, torch.float32, "src_ngrid"),
        _req(transform, torch.float32, "transform"), _req(tgt_grid, torch.float32, "tgt_grid"),
        _req(tgt_ngrid, torch.float32, "tgt_ngrid"), b, h, w, float(hfov[0]), float(hfov[1]), float(vfov[0]),
        float(vfov[1]), float(lambda_po2pl), int(flags), losses.data_ptr(), grad_t.data_ptr(),
        scratch.data_ptr(), _stream()), "delora_icp_dense_fwd_bwd")
    return losses, grad_t


ICP_STATS = 256      # DELORA_ICP_STATS flag bit


def icp_stats(reset=True):
    """Search statistics of dense ICP calls made with `flags | ICP_STATS` (include/delora_b200.h)."""
    import ctypes
    buf = (ctypes.c_uint32 * 32)()
    _lib.check(_lib.lib().delora_icp_stats(ctypes.cast(buf, ctypes.c_void_p), 1 if reset else 0), "delora_icp_stats")
    v = list(buf)
    names = ("0", "1-2", "3-5", "6-10", "11-20", "21-40", "41-63", "limit")
    return {"warps": v[0], "steps": v[1], "cells_per_lane": v[2], "warps_block_search": v[3], "block_owners": v[4],
            "blocks_bounded": v[5], "blocks_scanned": v[6], "max_blocks_scanned": v[7], "f64_rerank": v[8],
            "max_blocks_bounded": v[9], "owners_over_256_blocks": v[10], "owners_without_candidate": v[11],
            "warps_by_steps": dict(zip(names, v[16:24])), "cells_by_steps": dict(zip(names, v[24:32]))}


def icp_point_grads(point_dir, normal_dir, n_src, losses, upstream):
    """-> grad_pts, grad_nrm [B,3,Ns] channels-first."""
    b, ns, _ = point_dir.shape
    gp = torch.empty((b, 3, ns), dtype=torch.float32, device=point_dir.device)
    gn = torch.empty((b, 3, ns), dtype=torch.float32, device=point_dir.device)
    L = _lib.lib()
    _lib.check(L.delora_icp_point_grads(_req(point_dir, torch.float32, "point_dir"),
                                        _req(normal_dir, torch.float32, "normal_dir"),
                                        _req(n_src, torch.int32, "n_src"), ns, b,
                                        _req(losses, torch.float32, "losses"),
                                        _req(upstream, torch.float32, "upstream"),
                                        gp.data_ptr(), gn.data_ptr(), _stream()), "delora_icp_point_grads")
    return gp, gn


def quat_to_T(quaternion, translation):
    b = quaternion.shape[0]
    t = torch.empty((b, 4, 4), dtype=torch.float32, device=quaternion.device)
    L = _lib.lib()
    _lib.check(L.delora_quat_to_T(_req(quaternion, torch.float32, "quaternion"),
                                  _req(translation, torch.float32, "translation"), b, t.data_ptr(), _stream()),
               "delora_quat_to_T")
    return t


def quat_to_T_bwd(quaternion, grad_t):
    b = quaternion.shape[0]
    gq = torch.empty((b, 4), dtype=torch.float32, device=quaternion.device)
    gt = torch.empty((b, 3), dtype=torch.float32, device=quaternion.device)
    L = _lib.lib()
    _lib.check(L.delora_quat_to_T_bwd(_req(quaternion, torch.float32, "quaternion"),
                                      _req(grad_t, torch.float32, "grad_T"), b, gq.data_ptr(), gt.data_ptr(),
                                      _stream()), "delora_quat_to_T_bwd")
    return gq, gt


# ---------------------------------------------------------------------------------------------
# encoder (tcgen05 implicit-GEMM convolutions, bf16 NHWC with materialised padding)
ACT_NONE, ACT_RELU, ACT_TANH, ACT_TANH_BWD, ACT_RELU_BWD = 0, 1, 2, 3, 4


def padded_nhwc_zeros(b, h, w, c, device):
    """[B, H+2, W+2, C] bf16, all zero (the conv epilogue never touches the zero halo rows)."""
    return torch.zeros((b, h + 2, w + 2, c), dtype=torch.bfloat16, device=device)


def conv_out_size(n, stride):
    """Outputs of the encoder's 3x3/pad 1 and 1x1/pad 0 convolutions along one axis (any n, also odd)."""
    return (n - 1) // stride + 1


def conv2d_fprop(x, weight, hin, win, ksize, stride, act=ACT_NONE, residual=None, out=None, saved=None):
    """x [B,Hin+2,Win+2,Cin] bf16 padded NHWC, weight [Cout,k*k,Cin] bf16 -> y [B,Hout+2,Wout+2,Cout]."""
    b, _, _, cin = x.shape
    cout = weight.shape[0]
    hout, wout = conv_out_size(hin, stride[0]), conv_out_size(win, stride[1])
    if out is None:
        out = padded_nhwc_zeros(b, hout, wout, cout, x.device)
    L = _lib.lib()
    _lib.check(L.delora_conv2d_fprop_bf16(_req(x, torch.bfloat16, "x"), _req(weight, torch.bfloat16, "weight"),
                                          _req(residual, torch.bfloat16, "residual") if residual is not None else None,
                                          _req(saved, torch.bfloat16, "saved") if saved is not None else None,
                                          out.data_ptr(), b, hin, win, cin, cout, ksize, stride[0], stride[1], int(act),
                                          _stream()), "delora_conv2d_fprop_bf16")
    return out


def conv2d_dgrad_eligible(cin, cout, win, stride):
    """Can delora_conv2d_dgrad_bf16 (phase-decomposed data gradient) take this layer?  The library answers: the
    conditions depend on the kernel selection (delora_conv_select_kernel(2) / DELORA_CONV_PAIRS=0 rule out Cin = 64)."""
    return bool(_lib.lib().delora_conv2d_dgrad_supported(int(cin), int(cout), int(win), int(stride[0]), int(stride[1])))


def conv2d_dgrad(dz, w_flip, hin, win, stride, act=ACT_NONE, residual=None, out=None, saved=None,
                 residual_strided=False):
    """dz [B,Hout+2,Wout+2,Cout], w_flip [Cin,9,Cout] -> dx [B,Hin+2,Win+2,Cin] (3x3 conv of `stride`).
    residual_strided: `residual` has dz's spatial size and lands on the pixels (sh*h, sw*w) only."""
    b, _, _, cout = dz.shape
    cin = w_flip.shape[0]
    if out is None:
        out = padded_nhwc_zeros(b, hin, win, cin, dz.device)
    L = _lib.lib()
    _lib.check(L.delora_conv2d_dgrad_bf16(_req(dz, torch.bfloat16, "dz"), _req(w_flip, torch.bfloat16, "w_flip"),
                                          _req(residual, torch.bfloat16, "residual") if residual is not None else None,
                                          _req(saved, torch.bfloat16, "saved") if saved is not None else None,
                                          out.data_ptr(), b, hin, win, cin, cout, stride[0], stride[1], int(act),
                                          1 if residual_strided else 0, _stream()), "delora_conv2d_dgrad_bf16")
    return out


_wgrad_scratch = {}


def _grad_out(out, shape, device):
    if out is None:
        return torch.empty(shape, dtype=torch.float32, device=device)
    if tuple(out.shape) != tuple(shape) or out.dtype != torch.float32 or not out.is_contiguous():
        raise ValueError(f"gradient output must be a contiguous fp32 tensor of shape {tuple(shape)}")
    return out


def conv2d_wgrad(x, dz, hin, win, ksize, stride, cin_true=None, out=None):
    """x [B,Hin+2,Win+2,Cin], dz [B,Hout+2,Wout+2,Cout] (bf16 padded NHWC) -> dW [Cout,Cin_true,k,k] fp32
    (written into `out` when given: a contiguous fp32 tensor of that shape, e.g. a slice of a flat gradient buffer)."""
    b, _, _, cin = x.shape
    cout = dz.shape[3]
    cin_true = cin if cin_true is None else int(cin_true)
    hout, wout = conv_out_size(hin, stride[0]), conv_out_size(win, stride[1])
    L = _lib.lib()
    n = int(L.delora_conv2d_wgrad_scratch_floats(b, hout, wout, cin, cout, ksize))
    key = (x.device.index, n)
    scratch = _wgrad_scratch.get(key)
    if scratch is None:
        scratch = torch.empty((n,), dtype=torch.float32, device=x.device)
        _wgrad_scratch[key] = scratch
    dw = _grad_out(out, (cout, cin_true, ksize, ksize), x.device)
    _lib.check(L.delora_conv2d_wgrad_bf16(_req(x, torch.bfloat16, "x"), _req(dz, torch.bfloat16, "dz"), dw.data_ptr(),
                                          scratch.data_ptr(), b, hin, win, cin, cin_true, cout, ksize, stride[0],
                                          stride[1], _stream()), "delora_conv2d_wgrad_bf16")
    return dw


def zero_upsample(x, h, w, stride, out=None, out_hw=None):
    """x [B,H+2,W+2,C] -> [B,Hout+2,Wout+2,C]: x at the strided positions, zero elsewhere.  (Hout, Wout) is the
    input size of the strided convolution whose output is H x W (default H*sh x W*sw)."""
    b, _, _, c = x.shape
    ho, wo = out_hw if out_hw is not None else (h * stride[0], w * stride[1])
    if out is None:
        out = torch.empty((b, ho + 2, wo + 2, c), dtype=torch.bfloat16, device=x.device)
    L = _lib.lib()
    _lib.check(L.delora_zero_upsample_nhwc_bf16(_req(x, torch.bfloat16, "x"), b, h, w, c, stride[0], stride[1], ho, wo,
                                                out.data_ptr(), _stream()), "delora_zero_upsample_nhwc_bf16")
    return out


def conv_weight_prep(weight, w_fwd, w_flip=None, cin_pad=None):
    """weight [Cout,Cin,k,k] fp32 -> w_fwd [Cout,k*k,Cin_pad] bf16 and (optional) w_flip [Cin,k*k,Cout] bf16, in place."""
    cout, cin, k, _ = weight.shape
    cin_pad = cin if cin_pad is None else int(cin_pad)
    L = _lib.lib()
    _lib.check(L.delora_conv_weight_prep_bf16(_req(weight.detach(), torch.float32, "weight"), cout, cin, k, cin_pad,
                                              w_fwd.data_ptr(), w_flip.data_ptr() if w_flip is not None else None,
                                              _stream()), "delora_conv_weight_prep_bf16")
    return w_fwd, w_flip


def images_to_nhwc(image_1, image_2, cpad=64):
    b, _, h, w = image_1.shape
    x = torch.empty((b, h + 2, w + 2, cpad), dtype=torch.bfloat16, device=image_1.device)
    L = _lib.lib()
    _lib.check(L.delora_images_to_nhwc_bf16(_req(image_1, torch.float32, "image_1"),
                                            _req(image_2, torch.float32, "image_2"), b, h, w, cpad, x.data_ptr(),
                                            _stream()), "delora_images_to_nhwc_bf16")
    return x


def maxpool_w(x, h, w):
    b, _, _, c = x.shape
    y = padded_nhwc_zeros(b, h, w // 2, c, x.device)
    L = _lib.lib()
    _lib.check(L.delora_maxpool_w_nhwc_bf16(_req(x, torch.bfloat16, "x"), b, h, w, c, y.data_ptr(), _stream()),
               "delora_maxpool_w_nhwc_bf16")
    return y


def avgpool(x, h, w):
    """AdaptiveAvgPool2d((1,1)) of a padded NHWC bf16 map -> [B, C] fp32."""
    b, _, _, c = x.shape
    y = torch.empty((b, c), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    _lib.check(L.delora_avgpool_nhwc_bf16(_req(x, torch.bfloat16, "x"), b, h, w, c, y.data_ptr(), _stream()),
               "delora_avgpool_nhwc_bf16")
    return y


def nhwc_to_nchw(x, h, w):
    b, _, _, c = x.shape
    y = torch.empty((b, c, h, w), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    _lib.check(L.delora_nhwc_to_nchw_f32(_req(x, torch.bfloat16, "x"), b, h, w, c, y.data_ptr(), _stream()),
               "delora_nhwc_to_nchw_f32")
    return y


# ---- stem on the 16-channel layout (csrc/conv_stem.cu)
def images_to_nhwc16(image_1, image_2):
    b, _, h, w = image_1.shape
    x = torch.empty((b, h + 2, w + 2, 16), dtype=torch.bfloat16, device=image_1.device)
    L = _lib.lib()
    _lib.check(L.delora_images_to_nhwc16_bf16(_req(image_1, torch.float32, "image_1"),
                                              _req(image_2, torch.float32, "image_2"), b, h, w, x.data_ptr(), _stream()),
               "delora_images_to_nhwc16_bf16")
    return x


def stem_weight_prep(weight, w_stem):
    """weight [64,Cin<=16,3,3] fp32 -> w_stem [3,64,64] bf16 in place."""
    L = _lib.lib()
    _lib.check(L.delora_stem_weight_prep_bf16(_req(weight.detach(), torch.float32, "weight"), weight.shape[1],
                                              w_stem.data_ptr(), _stream()), "delora_stem_weight_prep_bf16")
    return w_stem


def stem_fprop(x16, w_stem, h, w, act, out=None, out_f16=False):
    """x16 [B,H+2,W+2,16], w_stem [3,64,64] -> y [B,H+2,W/2+2,64] (3x3, stride (1,2), activation).
    out_f16: the (bf16-typed) output buffer receives fp16 bit patterns (training: pre-activation for the pool kernels)."""
    b = x16.shape[0]
    if out is None:
        out = padded_nhwc_zeros(b, h, w // 2, 64, x16.device)
    L = _lib.lib()
    _lib.check(L.delora_stem_fprop_bf16(_req(x16, torch.bfloat16, "x16"), _req(w_stem, torch.bfloat16, "w_stem"),
                                        out.data_ptr(), b, h, w, int(act), 1 if out_f16 else 0, _stream()),
               "delora_stem_fprop_bf16")
    return out


def stem_wgrad(x16, dz, h, w, cin_true, out=None):
    """-> dW [64, cin_true, 3, 3] fp32."""
    b = x16.shape[0]
    L = _lib.lib()
    n = int(L.delora_stem_wgrad_scratch_floats(b, h, w))
    key = (x16.device.index, n)
    scratch = _wgrad_scratch.get(key)
    if scratch is None:
        scratch = torch.empty((n,), dtype=torch.float32, device=x16.device)
        _wgrad_scratch[key] = scratch
    dw = _grad_out(out, (64, cin_true, 3, 3), x16.device)
    _lib.check(L.delora_stem_wgrad_bf16(_req(x16, torch.bfloat16, "x16"), _req(dz, torch.bfloat16, "dz"), dw.data_ptr(),
                                        scratch.data_ptr(), b, h, w, int(cin_true), _stream()), "delora_stem_wgrad_bf16")
    return dw


def conv_weight_prep_multi(table, n_layers):
    """table: int64 CUDA tensor [n_layers, 8] (see include/delora_b200.h)."""
    L = _lib.lib()
    _lib.check(L.delora_conv_weight_prep_multi(_req(table, torch.int64, "table"), int(n_layers), _stream()),
               "delora_conv_weight_prep_multi")
