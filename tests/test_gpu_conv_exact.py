"""Per-variant tests of the tcgen05 convolutions (fprop, phase-decomposed dgrad, act' epilogues, wgrad) against a plain
fp64 restatement of the same operator, and a layer-by-layer replay of the encoder at production shapes.

Exact tests draw x, w, dz and the residual from {-1, 0, +1} times one power of two per tensor, and `saved` from
{0, +-0.5, +-1}: every product is exact, every accumulator is an integer multiple of the product unit below 2^24
(exact in fp32 in any summation order), and 1 - s^2 is in {1, 0.75, 0}.  The only rounding left is the final bf16
round-to-nearest-even, so fprop / dgrad outputs must equal `ref_fp64.float().bfloat16()` and wgrad (fp32) must equal
the fp64 reference.  |ref| <= 256 product units on (at least) 99 % of the outputs keeps one missing +-1 term visible
in bf16.

Real-valued tests use bf16 data with full significands and a per-element bound
    |got - ref| <= rel * (|f(ref)| + c S) + c S,   S = conv(|x|, |w|) (+ |residual|), c = n * 2^-23,
with n the number of fp32 additions one product goes through: one accumulator update per 16-deep MMA (ceil(K / 16)),
at most 16 inside an MMA, the residual, the act' product and (wgrad) up to 64 split-K partials; 2^-23 covers a
truncating adder.  rel = 2^-8 (bf16 round-to-nearest) plus 2^-10.987 for tanh.approx.f32 (PTX ISA bound).

The CPU tests (no `gpu` mark) check the fp64 helpers against torch autograd and show that the comparisons reject
mutated references (a dropped column, phase or 64-channel chunk, zero padding at the seam, a shifted tap).
"""
import math
import zlib

import pytest
import torch
import torch.nn.functional as F

F64 = torch.float64
DEV = "cuda"
gpu = pytest.mark.gpu

# kernel variants, as they appear (spaces removed) in the profiler's demangled names
PIXM1 = "conv_rows_tc_kernel<1,true>"
PIXM2 = "conv_rows_tc_kernel<2,true>"
ROWS1 = "conv_rows_tc_kernel<1,false>"
ROWS2 = "conv_rows_tc_kernel<2,false>"
FPROP = "conv_fprop_tc_kernel"
WG2 = "conv_wgrad2_tc_kernel"
WG1 = "conv_wgrad_tc_kernel"
VARIANTS = (PIXM1, PIXM2, ROWS1, ROWS2, FPROP, WG2, WG1)

U23 = 2.0 ** -23
REL_BF16 = 2.0 ** -8
REL_TANH = 2.0 ** -10.987


# ---------------------------------------------------------------------------------------------------------------------
# fp64 reference of the encoder's convolutions: 3x3 with circular padding in W and zero padding in H, or 1x1 without
# padding; stride (sh, sw); output size (n - 1) // s + 1.  Written tap by tap (no autograd), so the CPU tests can hold
# it against torch autograd.
def out_size(n, s):
    return (n - 1) // s + 1


def _taps(k):
    return [(r, q) for r in range(k) for q in range(k)]


def _pad(x, circular=True):
    x = F.pad(x, (1, 1, 0, 0), mode="circular") if circular else F.pad(x, (1, 1, 0, 0))
    return F.pad(x, (0, 0, 1, 1))


def ref_fprop(x, w, stride, k, circular=True):
    """x [B, Ci, H, W], w [Co, Ci, k, k] -> [B, Co, Ho, Wo] (all fp64)."""
    b, _, h, wd = x.shape
    sh, sw = stride
    ho, wo = out_size(h, sh), out_size(wd, sw)
    xp = _pad(x, circular) if k == 3 else x
    out = x.new_zeros((b, w.shape[0], ho, wo))
    for r, q in _taps(k):
        patch = xp[:, :, r:r + sh * (ho - 1) + 1:sh, q:q + sw * (wo - 1) + 1:sw]
        out += torch.einsum("bchw,oc->bohw", patch, w[:, :, r, q])
    return out


def ref_dgrad(dz, w, hw, stride, k, circular=True):
    """Gradient w.r.t. x of ref_fprop for output gradient dz [B, Co, Ho, Wo] -> [B, Ci, H, W]: every tap scatters into
    the padded input; the halo columns fold back onto the seam (circular), the halo rows are dropped (zero padding)."""
    b = dz.shape[0]
    ho, wo = dz.shape[2:]
    h, wd = hw
    sh, sw = stride
    ci = w.shape[1]
    acc = dz.new_zeros((b, ci, h + 2, wd + 2) if k == 3 else (b, ci, h, wd))
    for r, q in _taps(k):
        acc[:, :, r:r + sh * (ho - 1) + 1:sh, q:q + sw * (wo - 1) + 1:sw] += torch.einsum("bohw,oc->bchw", dz,
                                                                                         w[:, :, r, q])
    if k == 1:
        return acc
    dx = acc[:, :, 1:h + 1, 1:wd + 1].clone()
    if circular:
        dx[..., wd - 1] += acc[:, :, 1:h + 1, 0]
        dx[..., 0] += acc[:, :, 1:h + 1, wd + 1]
    return dx


def ref_wgrad(x, dz, stride, k):
    """Gradient w.r.t. w of ref_fprop -> [Co, Ci, k, k]."""
    ho, wo = dz.shape[2:]
    sh, sw = stride
    xp = _pad(x) if k == 3 else x
    dw = x.new_zeros((dz.shape[1], x.shape[1], k, k))
    for r, q in _taps(k):
        patch = xp[:, :, r:r + sh * (ho - 1) + 1:sh, q:q + sw * (wo - 1) + 1:sw]
        dw[:, :, r, q] = torch.einsum("bohw,bchw->oc", dz, patch)
    return dw


def upsample(small, hw, stride):
    """small [B, C, Ho, Wo] at the input pixels (sh * h, sw * w) of a stride-(sh, sw) layer, zero elsewhere: the data
    gradient of the 1x1 strided downsample, i.e. what `residual_strided` adds."""
    out = small.new_zeros(small.shape[:2] + tuple(hw))
    out[:, :, ::stride[0], ::stride[1]] = small
    return out


def act_fn(act):
    return {0: lambda v: v, 1: torch.relu, 2: torch.tanh, 3: lambda v: v, 4: lambda v: v}[act]


def act_prime(act, saved):
    """Factor the epilogue applies in the data-gradient modes (3: tanh' = 1 - s^2, 4: relu' = [s > 0])."""
    if act == 3:
        return 1.0 - saved * saved
    if act == 4:
        return (saved > 0).to(saved.dtype)
    return None


# ---------------------------------------------------------------------------------------------------------------------
# comparisons
def stored(ref, dtype):
    """The fp64 reference rounded like the kernel's store: to fp32, then (bf16 outputs) round-to-nearest-even."""
    return ref.float().to(dtype).double()


def exact_mismatches(got, ref, dtype):
    """Elements where the kernel output (stored as `dtype`) differs from stored(ref, dtype).  NaN (an element never
    written) counts as a mismatch."""
    return int((got.double() != stored(ref, dtype)).sum())


def bound_ratio(got, ref, s, c, rel):
    """max |got - ref| / (rel (|ref| + c S) + c S); inf for NaN, and for any error where the bound is 0."""
    cs = c * s
    bound = rel * (ref.abs() + cs) + cs
    err = (got.double() - ref).abs()
    if bool(torch.isnan(err).any()):
        return math.inf
    if bool(((bound == 0) & (err > 0)).any()):
        return math.inf
    return float((err / bound.clamp_min(1e-300)).max())


def c_of(k_terms, extra=2):
    """fp32 accumulation constant for a dot product of k_terms exact products (see the module docstring)."""
    return (math.ceil(k_terms / 16) + 16 + extra) * U23


# ---------------------------------------------------------------------------------------------------------------------
# which kernel must run (derived from conv_rows_launch / rows_pixm / rows_pick_tile, delora_conv2d_fprop_bf16 and
# delora_conv2d_wgrad_bf16).  sel = delora_conv_select_kernel setting: 0 first-generation kernels for fprop / wgrad,
# 1 default, 2 row-block kernel on single CTAs only.
def rows_variant(cin_k, cout_k, wg, sel):
    """Row-block kernel variant for a launch with cin_k input / cout_k output channels and a job grid wg wide."""
    pairs = sel != 2
    if cin_k % 64 != 0:
        return None
    if cout_k in (64, 128) and wg >= 128 and pairs:
        return PIXM2 if cout_k == 128 else PIXM1
    if cout_k % 128 == 0:
        return ROWS2 if (cout_k % 256 == 0 and pairs) else ROWS1
    return None


def expected_kernel(case, sel):
    if case["op"] == "fprop":
        if case["stride"] == (1, 1) and sel != 0:
            v = rows_variant(case["cin"], case["cout"], case["w"], sel)
            if v is not None:
                return v
        return FPROP
    if case["op"] == "dgrad":
        return dgrad_variant(case["cin"], case["cout"], case["w"], case["stride"], sel)
    k, stride, cout = case["k"], case["stride"], case["cout"]
    if sel != 0 and k == 3 and (cout % 128 == 0 or (cout == 64 and stride == (1, 1))):
        return WG2
    return WG1


def dgrad_variant(cin, cout, win, stride, sel):
    """Variant of delora_conv2d_dgrad_bf16 for a forward layer cin -> cout; None = the call must be rejected."""
    if stride[1] == 2 and win % 2 != 0:
        return None
    wg = (win + stride[1] - 1) // stride[1]
    return rows_variant(cout, cin, wg, sel)


# ---------------------------------------------------------------------------------------------------------------------
# the case table: forward shapes (h, w = input of the forward convolution) and the variant each case must launch
def C(op, b, cin, cout, h, w, k=3, stride=(1, 1), act=0, res=False, strided_res=False, cin_true=None, tag=None):
    return dict(op=op, b=b, cin=cin, cout=cout, h=h, w=w, k=k, stride=stride, act=act, res=res,
                strided_res=strided_res, cin_true=cin_true, tag=tag)


CASES = [
    # pixel-on-M, one CTA (Cout 64, W >= 128): W = 130 / 200 give two segments, the second ragged; H = 1 and 5
    # (R = 1; R = 2 with a partial last row block)
    C("fprop", 1, 64, 64, 1, 130, 3, act=0, tag=PIXM1),
    C("fprop", 2, 64, 64, 5, 200, 3, act=1, res=True, tag=PIXM1),
    C("fprop", 1, 64, 64, 5, 200, 3, act=2, tag=PIXM1),
    C("fprop", 2, 64, 64, 5, 130, 3, act=4, res=True, tag=PIXM1),
    C("fprop", 1, 128, 64, 5, 130, 1, act=0, tag=PIXM1),
    C("fprop", 1, 128, 64, 1, 200, 1, act=3, tag=PIXM1),
    # pixel-on-M, CTA pair (Cout 128): H = 3 -> R = 1, the second pair reaches past the image; H = 7 -> partial block
    C("fprop", 1, 64, 128, 3, 130, 3, act=0, tag=PIXM2),
    C("fprop", 2, 128, 128, 7, 256, 3, act=1, res=True, tag=PIXM2),
    C("fprop", 1, 128, 128, 3, 200, 3, act=4, res=True, tag=PIXM2),
    C("fprop", 1, 256, 128, 7, 130, 1, act=3, tag=PIXM2),
    # channel-on-M, one CTA (Cout 128, W < 128): W = 45, H = 1 is R = 1 with NS % 32 = 16 (second row masked)
    C("fprop", 1, 128, 128, 1, 45, 3, act=0, tag=ROWS1),
    C("fprop", 2, 128, 128, 3, 90, 3, act=1, res=True, tag=ROWS1),
    C("fprop", 1, 64, 128, 2, 90, 3, act=4, tag=ROWS1),
    C("fprop", 1, 256, 128, 5, 45, 1, act=3, tag=ROWS1),
    # channel-on-M, CTA pair (Cout 256 / 512): H = 1 leaves the peer CTA without valid rows
    C("fprop", 1, 256, 256, 1, 23, 3, act=0, tag=ROWS2),
    C("fprop", 2, 256, 512, 3, 45, 3, act=1, res=True, tag=ROWS2),
    C("fprop", 1, 512, 512, 1, 45, 3, act=3, tag=ROWS2),
    C("fprop", 1, 512, 256, 3, 23, 1, act=4, res=True, tag=ROWS2),
    C("fprop", 1, 256, 256, 3, 45, 3, act=2, tag=ROWS2),
    C("fprop", 1, 128, 256, 2, 260, 3, act=0, tag=ROWS2),
    # first-generation kernel: strided 3x3 / 1x1 with odd widths, stride 1 at Cout 64 below 128 columns, act 3 / 4
    C("fprop", 1, 64, 128, 4, 45, 3, (1, 2), act=1, tag=FPROP),
    C("fprop", 1, 64, 128, 4, 90, 3, (1, 2), act=2, tag=FPROP),
    C("fprop", 2, 128, 256, 5, 23, 3, (2, 2), act=0, tag=FPROP),
    C("fprop", 1, 64, 128, 3, 45, 1, (1, 2), act=0, tag=FPROP),
    C("fprop", 1, 256, 512, 5, 23, 1, (2, 2), act=0, tag=FPROP),
    C("fprop", 1, 64, 64, 3, 45, 3, act=3, res=True, tag=FPROP),
    C("fprop", 2, 64, 64, 4, 90, 3, act=4, tag=FPROP),
    # phase-decomposed data gradient (forward Cin -> Cout; the launch writes Cin channels): Cin 64 (pixel-on-M, one
    # CTA), 128 (pixel-on-M pair, or channel-on-M below 128 columns), 256 (channel-on-M pair); strides (1,1), (1,2),
    # (2,2); odd Hin under stride_h = 2; Wg = 130 just above one segment; residual_strided on and off
    C("dgrad", 1, 64, 64, 3, 130, stride=(1, 1), act=3, res=True, tag=PIXM1),
    C("dgrad", 2, 64, 128, 5, 260, stride=(1, 2), act=4, res=True, strided_res=True, tag=PIXM1),
    C("dgrad", 1, 64, 128, 5, 256, stride=(2, 2), act=3, res=True, strided_res=True, tag=PIXM1),
    C("dgrad", 1, 64, 128, 4, 260, stride=(1, 2), act=0, res=True, tag=PIXM1),
    C("dgrad", 1, 128, 256, 5, 260, stride=(2, 2), act=4, res=True, strided_res=True, tag=PIXM2),
    C("dgrad", 2, 128, 128, 3, 130, stride=(1, 1), act=3, res=True, tag=PIXM2),
    C("dgrad", 1, 128, 256, 7, 256, stride=(1, 2), act=0, tag=PIXM2),
    C("dgrad", 1, 128, 256, 5, 90, stride=(2, 2), act=4, res=True, strided_res=True, tag=ROWS1),
    C("dgrad", 1, 256, 512, 5, 90, stride=(2, 2), act=3, res=True, strided_res=True, tag=ROWS2),
    C("dgrad", 2, 256, 512, 4, 46, stride=(1, 2), act=4, res=True, tag=ROWS2),
    C("dgrad", 1, 256, 256, 3, 45, stride=(1, 1), act=0, tag=ROWS2),
    # weight gradient: second-generation mode 0 (Cout % 128 == 0, also strided: even / odd column tile maps) and mode 1
    # (Cout 64, stride 1); first-generation for 1x1, strided Cout 64 and the 8-of-64-channel stem layout
    C("wgrad", 2, 64, 128, 4, 260, 3, (1, 2), tag=WG2),
    C("wgrad", 1, 256, 512, 5, 45, 3, (2, 2), tag=WG2),
    C("wgrad", 1, 128, 128, 3, 130, 3, (1, 1), tag=WG2),
    C("wgrad", 2, 512, 512, 3, 23, 3, (1, 1), tag=WG2),
    C("wgrad", 1, 64, 64, 3, 130, 3, (1, 1), tag=WG2),
    C("wgrad", 2, 64, 64, 5, 45, 3, (1, 1), tag=WG2),
    C("wgrad", 1, 64, 128, 4, 90, 1, (1, 2), tag=WG1),
    C("wgrad", 1, 256, 512, 5, 45, 1, (2, 2), tag=WG1),
    C("wgrad", 1, 64, 64, 4, 90, 3, (1, 2), tag=WG1),
    C("wgrad", 2, 64, 64, 3, 90, 3, (1, 2), cin_true=8, tag=WG1),
]


def case_id(c):
    s = f"{c['op']}-b{c['b']}-{c['cin']}to{c['cout']}-{c['h']}x{c['w']}-k{c['k']}-s{c['stride'][0]}{c['stride'][1]}"
    if c["op"] != "wgrad":
        s += f"-act{c['act']}" + ("-res" if c["res"] else "") + ("-strided" if c["strided_res"] else "")
    if c["cin_true"]:
        s += f"-cin{c['cin_true']}"
    return s


# ---------------------------------------------------------------------------------------------------------------------
# device-side helpers
def to_nhwc(x):
    """[B, C, H, W] (fp64 holding bf16 values) -> padded NHWC bf16 [B, H+2, W+2, C]: circular halo columns, zero rows."""
    return _pad(x).permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def from_nhwc(t, h, w):
    return t[:, 1:h + 1, 1:w + 1].permute(0, 3, 1, 2).double()


NAN16 = 0x7FC0        # bf16 quiet NaN: interior must be overwritten
HALO16 = 0x7F00       # 1.7e38: halo rows must stay untouched
GUARD16 = 0x4B00      # 8388608.0: bytes before / after `out`


def guarded_bf16(shape):
    """-> (flat buffer, out view): `out` a slice of a larger buffer, NaN inside, HALO16 in the halo rows."""
    n = math.prod(shape)
    g = 4 * shape[-1]
    flat = torch.full((n + 2 * g,), GUARD16, dtype=torch.int16, device=DEV)
    out = flat[g:g + n].view(shape)
    out.fill_(NAN16)
    out[:, 0] = HALO16
    out[:, -1] = HALO16
    return flat, g, out.view(torch.bfloat16)


def check_hygiene(flat, g, out, h, w):
    n = out.numel()
    raw = out.view(torch.int16)
    assert bool((flat[:g] == GUARD16).all()) and bool((flat[g + n:] == GUARD16).all()), "write outside `out`"
    assert bool((raw[:, 0] == HALO16).all()) and bool((raw[:, -1] == HALO16).all()), "halo row written"
    assert torch.equal(raw[:, 1:h + 1, 0], raw[:, 1:h + 1, w]), "left halo column is not the circular copy"
    assert torch.equal(raw[:, 1:h + 1, w + 1], raw[:, 1:h + 1, 1]), "right halo column is not the circular copy"


def make(shape, kind, unit, gen):
    """exact: {-1, 0, +1} * unit; real: N(0, 1) * unit rounded to bf16 (full 8-bit significands)."""
    if kind == "exact":
        v = torch.randint(-1, 2, shape, generator=gen, device=DEV).to(F64)
    else:
        v = torch.randn(shape, generator=gen, device=DEV, dtype=F64)
    return (v * unit).to(torch.bfloat16).double()


def make_saved(shape, act, kind, gen):
    if kind == "exact":
        return torch.randint(-2, 3, shape, generator=gen, device=DEV).to(F64) * 0.5
    v = torch.randn(shape, generator=gen, device=DEV, dtype=F64)
    return (torch.tanh(v) if act == 3 else v).to(torch.bfloat16).double()


def launched(fn):
    """Run fn under the profiler -> (result, set of demangled kernel names without spaces)."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.key.replace(" ", "") for e in prof.key_averages()}


def assert_variant(names, variant):
    ran = [v for v in VARIANTS if any(v in n for n in names)]
    assert ran == [variant], (variant, ran)


def run_case(case, sel, kind, seed=0):
    """Run one table case under kernel selection `sel` with `kind` data -> dict(got, ref, S, c, act, ...)."""
    from delora_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(seed * 7919 + zlib.crc32(case_id(case).encode()))
    b, cin, cout, h, w, k, stride, act = (case[n] for n in ("b", "cin", "cout", "h", "w", "k", "stride", "act"))
    ho, wo = out_size(h, stride[0]), out_size(w, stride[1])
    ux, uw, udz = 2.0 ** -2, 2.0 ** -5, 2.0 ** -3
    if kind == "real":
        uw = 1.0 / math.sqrt(cin * k * k)
    variant = expected_kernel(case, sel)
    if case["op"] == "fprop":
        x = make((b, cin, h, w), kind, ux, gen)
        wt = make((cout, cin, k, k), kind, uw, gen)
        res = make((b, cout, ho, wo), kind, ux * uw if kind == "exact" else 1.0, gen) if case["res"] else None
        saved = make_saved((b, cout, ho, wo), act, kind, gen) if act >= 3 else None
        flat, g, out = guarded_bf16((b, ho + 2, wo + 2, cout))
        wk = wt.permute(0, 2, 3, 1).reshape(cout, k * k, cin).contiguous().to(torch.bfloat16)
        _, names = launched(lambda: ops.conv2d_fprop(to_nhwc(x), wk, h, w, k, stride, act,
                                                     to_nhwc(res) if res is not None else None, out=out,
                                                     saved=to_nhwc(saved) if saved is not None else None))
        acc = ref_fprop(x, wt, stride, k)
        s = ref_fprop(x.abs(), wt.abs(), stride, k)
        n_terms, unit, oh, ow = cin * k * k, ux * uw, ho, wo
    elif case["op"] == "dgrad":
        dz = make((b, cout, ho, wo), kind, udz, gen)
        wt = make((cout, cin, 3, 3), kind, uw, gen)
        unit = udz * uw
        res = None
        if case["res"]:
            rshape = (b, cin, ho, wo) if case["strided_res"] else (b, cin, h, w)
            res = make(rshape, kind, unit if kind == "exact" else 1.0, gen)
        saved = make_saved((b, cin, h, w), act, kind, gen) if act >= 3 else None
        flat, g, out = guarded_bf16((b, h + 2, w + 2, cin))
        w_flip = wt.flip(2, 3).permute(1, 2, 3, 0).reshape(cin, 9, cout).contiguous().to(torch.bfloat16)

        def call():
            return ops.conv2d_dgrad(to_nhwc(dz), w_flip, h, w, stride, act, to_nhwc(res) if res is not None else None,
                                    out=out, saved=to_nhwc(saved) if saved is not None else None,
                                    residual_strided=case["strided_res"])
        if variant is None:
            with pytest.raises(RuntimeError):
                call()
            return None
        _, names = launched(call)
        acc = ref_dgrad(dz, wt, (h, w), stride, 3)
        s = ref_dgrad(dz.abs(), wt.abs(), (h, w), stride, 3)
        if res is not None and case["strided_res"]:
            res = upsample(res, (h, w), stride)
        n_terms, oh, ow = cout * 9, h, w
    else:
        cin_true = case["cin_true"] or cin
        x = make((b, cin, h, w), kind, ux, gen)
        dz = make((b, cout, ho, wo), kind, udz, gen)
        n = cout * cin_true * k * k
        flat = torch.full((n + 256,), 1234.5, dtype=torch.float32, device=DEV)
        out = flat[128:128 + n].view(cout, cin_true, k, k)
        out.fill_(float("nan"))
        got, names = launched(lambda: ops.conv2d_wgrad(to_nhwc(x), to_nhwc(dz), h, w, k, stride,
                                                       cin_true=case["cin_true"], out=out))
        assert got.data_ptr() == out.data_ptr()
        assert bool((flat[:128] == 1234.5).all()) and bool((flat[128 + n:] == 1234.5).all()), "write outside `out`"
        assert_variant(names, variant)
        ref = ref_wgrad(x, dz, stride, k)[:, :cin_true]
        s = ref_wgrad(x.abs(), dz.abs(), stride, k)[:, :cin_true]
        k_pix = b * ho * wo
        return dict(got=out, ref=ref, S=s, c=c_of(k_pix, extra=64), rel=2.0 ** -24, units=ref / (ux * udz),
                    dtype=torch.float32)
    assert_variant(names, variant)
    check_hygiene(flat, g, out, oh, ow)
    cout_k = out.shape[-1]
    pre = acc + res if res is not None else acc
    units = pre / unit
    if res is not None:
        s = s + res.abs()
    d = act_prime(act, saved)
    if d is not None:
        pre, s = pre * d, s * d.abs()
    ref = act_fn(act)(pre)
    rel = REL_BF16 + (REL_TANH * (1 + REL_BF16) if act == 2 else 0.0)
    got = from_nhwc(out, oh, ow)
    assert got.shape[1] == cout_k
    return dict(got=got, ref=ref, S=s, c=c_of(n_terms), rel=rel, units=units, act=act, dtype=torch.bfloat16)


def _select(sel):
    from delora_b200 import _lib
    return _lib.lib().delora_conv_select_kernel(sel)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: exact table under the three kernel selections
@gpu
@pytest.mark.parametrize("sel", [1, 0, 2])
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_exact_case(case, sel, cuda_lib):
    prev = _select(sel)
    try:
        r = run_case(case, sel, "exact")
    finally:
        _select(prev)
    if r is None:           # rejected under this selection (checked inside run_case)
        return
    units = r["units"]                    # accumulator (+ residual) in product units, before act'
    assert float((units.abs() <= 256).double().mean()) >= 0.99     # one missing +-1 term stays visible in bf16
    assert bool((units == units.round()).all()) and float(units.abs().max()) < 2 ** 24   # exact in fp32
    if r.get("act") == 2:
        ratio = bound_ratio(r["got"], r["ref"], torch.zeros_like(r["ref"]), 0.0, r["rel"])
        assert ratio <= 1.0, ratio
    else:
        bad = exact_mismatches(r["got"], r["ref"], r["dtype"])
        if bad:
            want = stored(r["ref"], r["dtype"])
            idx = (r["got"].double() != want).nonzero()[:8]
            detail = [(tuple(i.tolist()), float(r["got"][tuple(i)]), float(want[tuple(i)]), float(r["ref"][tuple(i)]),
                       float(units[tuple(i)])) for i in idx]
            pytest.fail(f"{bad} of {r['ref'].numel()} outputs differ from the exact result "
                        f"(index, got, want, fp64 ref, accumulator in product units): {detail}")


@gpu
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_real_valued_case_within_fp32_bound(case, cuda_lib):
    """bf16 data with full significands at encoder scales: per-element bound of the module docstring."""
    prev = _select(1)
    try:
        r = run_case(case, 1, "real", seed=1)
    finally:
        _select(prev)
    ratio = bound_ratio(r["got"], r["ref"], r["S"], r["c"], r["rel"])
    print(f"BOUND_RATIO {case['op']}:{case['tag']} {case_id(case)} {ratio:.4f}")
    assert ratio <= 1.0, ratio


@gpu
def test_dgrad_and_wgrad_are_deterministic(cuda_lib):
    from delora_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(3)
    b, cin, cout, h, w, stride = 2, 64, 128, 6, 260, (1, 2)
    x = to_nhwc(make((b, cin, h, w), "real", 1.0, gen))
    dz = to_nhwc(make((b, cout, h, w // 2), "real", 1.0, gen))
    wf = make((cin, 9, cout), "real", 0.05, gen).to(torch.bfloat16)
    saved = to_nhwc(make_saved((b, cin, h, w), 3, "real", gen))
    dx = [ops.conv2d_dgrad(dz, wf, h, w, stride, ops.ACT_TANH_BWD, saved=saved).clone() for _ in range(2)]
    assert torch.equal(dx[0].view(torch.int16), dx[1].view(torch.int16))
    for (ci, co, hh, ww, k, st) in ((64, 128, 6, 260, 3, (1, 2)), (256, 512, 9, 90, 3, (2, 2)), (64, 64, 8, 130, 3, (1, 1)),
                                    (128, 256, 9, 90, 1, (2, 2))):
        xx = to_nhwc(make((2, ci, hh, ww), "real", 1.0, gen))
        dd = to_nhwc(make((2, co, out_size(hh, st[0]), out_size(ww, st[1])), "real", 1.0, gen))
        dw = [ops.conv2d_wgrad(xx, dd, hh, ww, k, st).clone() for _ in range(2)]
        assert torch.equal(dw[0].view(torch.int32), dw[1].view(torch.int32)), (ci, co, k, st)


@gpu
def test_argument_rejections(cuda_lib):
    from delora_b200 import ops
    z = lambda *s: torch.zeros(s, dtype=torch.bfloat16, device=DEV)       # noqa: E731
    with pytest.raises(RuntimeError, match="even Win"):      # odd Win under stride_w = 2
        ops.conv2d_dgrad(z(1, 6, 25, 256), z(128, 9, 256), 4, 45, (1, 2))
    with pytest.raises(RuntimeError):                         # Cin = 64 below 128 columns per phase
        ops.conv2d_dgrad(z(1, 6, 47, 128), z(64, 9, 128), 4, 90, (1, 2))
    with pytest.raises(RuntimeError, match="need `saved`"):
        ops.conv2d_dgrad(z(1, 6, 132, 64), z(64, 9, 64), 4, 130, (1, 1), ops.ACT_TANH_BWD)
    with pytest.raises(RuntimeError, match="need `saved`"):
        ops.conv2d_fprop(z(1, 6, 132, 64), z(64, 9, 64), 4, 130, 3, (1, 1), ops.ACT_RELU_BWD)


@gpu
@pytest.mark.parametrize("b,h,w,c,act", [(2, 3, 23, 512, 2), (1, 4, 8, 64, 1), (2, 1, 45, 256, 0), (1, 2, 2, 128, 2),
                                         (2, 16, 128, 256, 1)])
def test_avgpool_backward_exact(b, h, w, c, act, cuda_lib):
    """dz = g / (H W) * act'(a) in fp32 (the same two IEEE products), rounded once to bf16: bit for bit."""
    from delora_b200 import ops
    L = ops._lib.lib()
    gen = torch.Generator(device=DEV).manual_seed(h * 131 + w)
    a = torch.randn((b, c, h, w), generator=gen, device=DEV, dtype=F64)
    a = (torch.tanh(a) if act == 2 else a).to(torch.bfloat16).double()
    g = torch.randn((b, c), generator=gen, device=DEV) * 3.0
    flat, off, dz = guarded_bf16((b, h + 2, w + 2, c))
    ops._lib.check(L.delora_avgpool_bwd_nhwc_bf16(g.data_ptr(), to_nhwc(a).data_ptr(), b, h, w, c, act, dz.data_ptr(),
                                                  ops._stream()), "delora_avgpool_bwd_nhwc_bf16")
    torch.cuda.synchronize()
    check_hygiene(flat, off, dz, h, w)
    inv = torch.tensor(1.0, dtype=torch.float32, device=DEV) / torch.tensor(float(h * w), dtype=torch.float32, device=DEV)
    d = {0: torch.ones_like(a), 1: (a > 0).double(), 2: 1.0 - a * a}[act].float()
    want = ((g[:, :, None, None] * inv) * d).to(torch.bfloat16)
    assert torch.equal(from_nhwc(dz, h, w), want.double())


# ---------------------------------------------------------------------------------------------------------------------
# GPU: layer-by-layer replay of the encoder's training step at production shapes
def _tagged(enc, tag):
    hits = [t for k, t in enc._buf.items() if k[2] == tag]
    assert len(hits) == 1, (tag, len(hits))
    return hits[0]


@gpu
@pytest.mark.parametrize("sel", [1, 2])
@pytest.mark.parametrize("activation", ["tanh", "relu"])
@pytest.mark.parametrize("h,w", [(64, 2048), (64, 720), (16, 180)])
def test_encoder_replay_layer_by_layer(h, w, activation, sel, cuda_lib):
    """One pooled_features(...).backward on the tensor-core encoder; then every one of the 20 convolutions is
    recomputed in fp64 from that layer's own bf16 inputs (the encoder's buffers): forward outputs, dz1 (act' mode),
    the data gradient (phase-decomposed or zero-upsample fallback), the downsample's `small`, the weight gradients."""
    from delora_b200 import ops, synthetic
    from delora_b200.models.model import OdometryModel
    from delora_b200.models.tc_encoder import TensorCoreEncoder
    b = 2
    cfg = synthetic.fov_config(h=h, w=w, device=DEV)
    cfg.update({"pre_feature_extraction": False, "resnet_outputs": 1000, "use_dropout": False, "layers": [2, 2, 2, 2],
                "factor_fewer_resnet_channels": 1, "activation_fct": activation, "use_single_mlp_at_output": False})
    torch.manual_seed(0)
    model = OdometryModel(cfg).to(DEV)
    enc = TensorCoreEncoder(model)
    gen = torch.Generator(device=DEV).manual_seed(1)
    img1 = torch.randn(b, 4, h, w, device=DEV, generator=gen) * 5.0
    img2 = torch.randn(b, 4, h, w, device=DEV, generator=gen) * 5.0
    prev = _select(sel)
    try:
        model.zero_grad(set_to_none=True)
        pooled = enc.pooled_features(img1, img2)
        g_pooled = torch.randn(pooled.shape, device=DEV, generator=gen)
        (pooled * g_pooled).sum().backward()
        torch.cuda.synchronize()
    finally:
        _select(prev)
    relu = activation == "relu"
    f = torch.relu if relu else torch.tanh
    dact = (lambda s: (s > 0).double()) if relu else (lambda s: 1.0 - s * s)
    rel_f = REL_BF16 + (0.0 if relu else REL_TANH * (1 + REL_BF16))
    params = enc.trunk_parameters()
    wts = [p.detach().to(torch.bfloat16).double() for p in params]
    ratios = {}

    def check_map(name, buf, hw, ref, s, c, rel, fam):
        assert torch.equal(buf[:, :, 0].view(torch.int16), buf[:, :, hw[1]].view(torch.int16)), name
        assert torch.equal(buf[:, :, hw[1] + 1].view(torch.int16), buf[:, :, 1].view(torch.int16)), name
        assert float(buf[:, 0].abs().max()) == 0.0 and float(buf[:, -1].abs().max()) == 0.0, name
        r = bound_ratio(from_nhwc(buf, *hw), ref, s, c, rel)
        ratios[fam] = max(ratios.get(fam, 0.0), r)
        assert r <= 1.0, (name, r)

    def check_grad(name, got, ref, s, k_pix, fam):
        r = bound_ratio(got, ref, s, c_of(k_pix, extra=64), 2.0 ** -24)
        ratios[fam] = max(ratios.get(fam, 0.0), r)
        assert r <= 1.0, (name, r)

    # geometry of the trunk: stem (1, 2), max pool (1, 2), then the blocks
    hw = (h, out_size(w, 2) // 2)
    geo = []
    for blk in enc.blocks:
        sh, sw = blk["stride"]
        geo.append((hw, (out_size(hw[0], sh), out_size(hw[1], sw))))
        hw = geo[-1][1]
    nb = len(enc.blocks)
    # g_last: the average pool's backward, exact (same fp32 products as the kernel)
    oh, ow = geo[-1][1]
    last = from_nhwc(_tagged(enc, f"t{nb - 1}o"), oh, ow)
    inv = torch.tensor(1.0, dtype=torch.float32, device=DEV) / torch.tensor(float(oh * ow), dtype=torch.float32,
                                                                          device=DEV)
    want = ((g_pooled.float()[:, :, None, None] * inv) * dact(last).float()).to(torch.bfloat16).double()
    assert torch.equal(from_nhwc(_tagged(enc, "g_last"), oh, ow), want)

    dz2_buf = _tagged(enc, "g_last")
    for i in range(nb - 1, -1, -1):
        blk = enc.blocks[i]
        (ch, cw), (oh, ow) = geo[i]
        stride = blk["stride"]
        pidx = enc._block_param_idx[i]
        w1, w2 = wts[pidx[0]], wts[pidx[1]]
        wd = wts[pidx[2]] if blk["has_wd"] else None
        cin = w1.shape[1]
        x = from_nhwc(_tagged(enc, "t_pool" if i == 0 else f"t{i - 1}o"), ch, cw)
        t1 = from_nhwc(_tagged(enc, f"t{i}a"), oh, ow)
        dz2 = from_nhwc(dz2_buf, oh, ow)
        # forward: t1 = f(conv1(x)), [td = conv_d(x)], out = f(conv2(t1) + ident)
        check_map(f"t{i}a", _tagged(enc, f"t{i}a"), (oh, ow), f(ref_fprop(x, w1, stride, 3)),
                  ref_fprop(x.abs(), w1.abs(), stride, 3), c_of(cin * 9), rel_f, "fwd conv1")
        if wd is not None:
            ident = from_nhwc(_tagged(enc, f"t{i}d"), oh, ow)
            check_map(f"t{i}d", _tagged(enc, f"t{i}d"), (oh, ow), ref_fprop(x, wd, stride, 1),
                      ref_fprop(x.abs(), wd.abs(), stride, 1), c_of(cin), REL_BF16, "fwd downsample")
        else:
            ident = x
        cout = w2.shape[0]
        check_map(f"t{i}o", _tagged(enc, f"t{i}o"), (oh, ow), f(ref_fprop(t1, w2, (1, 1), 3) + ident),
                  ref_fprop(t1.abs(), w2.abs(), (1, 1), 3) + ident.abs(), c_of(cout * 9), rel_f, "fwd conv2+res")
        # backward
        check_grad(f"dW2[{i}]", params[pidx[1]].grad, ref_wgrad(t1, dz2, (1, 1), 3),
                   ref_wgrad(t1.abs(), dz2.abs(), (1, 1), 3), b * oh * ow, "wgrad 3x3")
        d1 = dact(t1)
        check_map(f"g{i}a", _tagged(enc, f"g{i}a"), (oh, ow), ref_dgrad(dz2, w2, (oh, ow), (1, 1), 3) * d1,
                  ref_dgrad(dz2.abs(), w2.abs(), (oh, ow), (1, 1), 3) * d1.abs(), c_of(cout * 9), REL_BF16,
                  "dz1 (act')")
        dz1 = from_nhwc(_tagged(enc, f"g{i}a"), oh, ow)
        check_grad(f"dW1[{i}]", params[pidx[0]].grad, ref_wgrad(x, dz1, stride, 3),
                   ref_wgrad(x.abs(), dz1.abs(), stride, 3), b * oh * ow, "wgrad 3x3")
        if wd is not None:
            check_grad(f"dWd[{i}]", params[pidx[2]].grad, ref_wgrad(x, dz2, stride, 1),
                       ref_wgrad(x.abs(), dz2.abs(), stride, 1), b * oh * ow, "wgrad 1x1")
            small_buf = _tagged(enc, f"g{i}ds")
            check_map(f"g{i}ds", small_buf, (oh, ow), torch.einsum("bohw,oc->bchw", dz2, wd[:, :, 0, 0]),
                      torch.einsum("bohw,oc->bchw", dz2.abs(), wd[:, :, 0, 0].abs()), c_of(cout), REL_BF16,
                      "dgrad 1x1 (small)")
            resid = upsample(from_nhwc(small_buf, oh, ow), (ch, cw), stride)
        else:
            resid = dz2
        ref = ref_dgrad(dz1, w1, (ch, cw), stride, 3) + resid
        s = ref_dgrad(dz1.abs(), w1.abs(), (ch, cw), stride, 3) + resid.abs()
        phase = blk["has_wd"] and i > 0 and dgrad_variant(cin, cout, cw, stride, sel) is not None
        fam = "dgrad phase" if phase else ("dgrad fallback" if blk["has_wd"] else "dgrad stride 1")
        if i > 0:
            dx = dact(x)
            dz2_buf = _tagged(enc, f"g{i}x")
            check_map(f"g{i}x", dz2_buf, (ch, cw), ref * dx, s * dx.abs(), c_of(cout * 9), REL_BF16, fam)
        else:
            check_map("g_pool", _tagged(enc, "g_pool"), (ch, cw), ref, s, c_of(cout * 9), REL_BF16, fam)
    print(f"REPLAY_RATIOS {h}x{w} {activation} sel={sel} " +
          " ".join(f"[{k}]={v:.4f}" for k, v in sorted(ratios.items())))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the kernel-selection model, the eligibility query, the fp64 helpers and the teeth of the comparisons
def test_case_table_covers_every_variant():
    """Each case's tag is the variant the dispatch rules give at the default selection, and the table holds every
    variant (fprop / dgrad through every row-block form)."""
    for c in CASES:
        assert expected_kernel(c, 1) == c["tag"], case_id(c)
    tags = {(c["op"], c["tag"]) for c in CASES}
    for v in VARIANTS:
        assert any(t == v for _, t in tags), v
    for v in (PIXM1, PIXM2, ROWS1, ROWS2):
        assert ("dgrad", v) in tags, v
    for stride in ((1, 1), (1, 2), (2, 2)):
        assert any(c["op"] == "dgrad" and c["stride"] == stride for c in CASES)


def test_dgrad_eligibility_matches_the_library():
    """ops.conv2d_dgrad_eligible (what the encoder's backward uses to pick the phase-decomposed data gradient) answers
    like the library's own check under every kernel selection; Cin = 64 needs CTA pairs (not under selection 2)."""
    from delora_b200 import _lib, ops
    L = _lib.lib()
    prev = L.delora_conv_select_kernel(1)
    try:
        for sel in (0, 1, 2):
            L.delora_conv_select_kernel(sel)
            assert L.delora_conv_select_kernel(-1) == sel
            for cin in (64, 128, 256, 512):
                for cout in (64, 128, 256, 512):
                    for win in (45, 46, 90, 180, 255, 256, 260, 512, 1024):
                        for stride in ((1, 1), (1, 2), (2, 2)):
                            want = dgrad_variant(cin, cout, win, stride, sel) is not None
                            got_c = bool(L.delora_conv2d_dgrad_supported(cin, cout, win, stride[0], stride[1]))
                            got_py = bool(ops.conv2d_dgrad_eligible(cin, cout, win, stride))
                            assert got_c == want and got_py == want, (sel, cin, cout, win, stride, got_c, got_py)
    finally:
        L.delora_conv_select_kernel(prev)


def _autograd_conv(x, w, stride, k):
    if k == 3:
        return F.conv2d(F.pad(x, (1, 1, 0, 0), mode="circular"), w, stride=stride, padding=(1, 0))
    return F.conv2d(x, w, stride=stride)


@pytest.mark.parametrize("k,stride,h,w", [(3, (1, 1), 5, 7), (3, (1, 2), 4, 10), (3, (1, 2), 4, 9), (3, (2, 2), 5, 9),
                                          (3, (2, 2), 6, 8), (1, (1, 2), 4, 9), (1, (2, 2), 5, 6), (3, (1, 1), 1, 1)])
def test_reference_helpers_match_autograd(k, stride, h, w):
    g = torch.Generator().manual_seed(h * 10 + w)
    b, ci, co = 2, 3, 4
    x = torch.randn((b, ci, h, w), generator=g, dtype=F64, requires_grad=True)
    wt = torch.randn((co, ci, k, k), generator=g, dtype=F64, requires_grad=True)
    y = _autograd_conv(x, wt, stride, k)
    assert torch.allclose(ref_fprop(x.detach(), wt.detach(), stride, k), y, rtol=1e-12, atol=1e-12)
    dz = torch.randn(y.shape, generator=g, dtype=F64)
    gx, gw = torch.autograd.grad(y, (x, wt), dz, retain_graph=True)
    assert torch.allclose(ref_dgrad(dz, wt.detach(), (h, w), stride, k), gx, rtol=1e-12, atol=1e-12)
    assert torch.allclose(ref_wgrad(x.detach(), dz, stride, k), gw, rtol=1e-12, atol=1e-12)
    if k == 3 and stride != (1, 1):
        # residual_strided: the block's input gradient = dgrad(conv1) + the 1x1 strided downsample's gradient, which is
        # `small` = dz_d . Wd placed on the pixels (sh h, sw w)
        wd = torch.randn((co, ci, 1, 1), generator=g, dtype=F64, requires_grad=True)
        yd = _autograd_conv(x, wd, stride, 1)
        dzd = torch.randn(yd.shape, generator=g, dtype=F64)
        gx2, = torch.autograd.grad((y * dz).sum() + (yd * dzd).sum(), x)
        small = torch.einsum("bohw,oc->bchw", dzd, wd.detach()[:, :, 0, 0])
        assert torch.allclose(ref_dgrad(dz, wt.detach(), (h, w), stride, k) + upsample(small, (h, w), stride), gx2,
                              rtol=1e-12, atol=1e-12)


def _exact_setup(op, stride, h, w, cin=128, cout=128, seed=0):
    g = torch.Generator().manual_seed(seed)
    t = lambda *s: torch.randint(-1, 2, s, generator=g).to(F64)      # noqa: E731
    wt = t(cout, cin, 3, 3) * 2.0 ** -5
    if op == "fprop":
        x = t(2, cin, h, w) * 2.0 ** -2
        return x, wt, ref_fprop(x, wt, stride, 3)
    ho, wo = out_size(h, stride[0]), out_size(w, stride[1])
    dz = t(2, cout, ho, wo) * 2.0 ** -3
    return dz, wt, ref_dgrad(dz, wt, (h, w), stride, 3)


@pytest.mark.parametrize("op,stride", [("fprop", (1, 1)), ("fprop", (1, 2)), ("dgrad", (1, 2)), ("dgrad", (2, 2))])
def test_comparisons_reject_mutated_references(op, stride):
    """Outputs a subtly wrong kernel would produce -- the last column not written, one dgrad phase missing, one
    64-channel chunk of the reduction missing, zero padding at the circular seam, one tap applied one column off --
    fail both the exact comparison and the real-valued bound, while the correct result passes both."""
    h, w = 5, 12
    inp, wt, ref = _exact_setup(op, stride, h, w)
    fn = ref_fprop if op == "fprop" else (lambda a, b_, s, k, circular=True: ref_dgrad(a, b_, (h, w), s, k, circular))
    s = fn(inp.abs(), wt.abs(), stride, 3)
    c = c_of(inp.shape[1] * 9)
    good = ref.float().to(torch.bfloat16)
    assert exact_mismatches(good, ref, torch.bfloat16) == 0 and bound_ratio(good, ref, s, c, REL_BF16) <= 1.0
    mutants = {}
    m = ref.clone()
    m[..., -1] = 0.0
    mutants["last column dropped"] = m
    if op == "dgrad":
        m = ref.clone()
        m[:, :, stride[0] - 1::stride[0], 1::2] = 0.0
        mutants["one phase dropped"] = m
    chunk = inp.clone()
    chunk[:, 64:128] = 0.0
    mutants["64-channel chunk dropped"] = fn(chunk, wt, stride, 3)
    mutants["zero padding at the seam"] = fn(inp, wt, stride, 3, circular=False)
    shifted = wt.clone()
    shifted[:, :, 1, 2] += shifted[:, :, 1, 1]
    shifted[:, :, 1, 1] = 0.0
    mutants["one tap shifted"] = fn(inp, shifted, stride, 3)
    for name, mref in mutants.items():
        got = mref.float().to(torch.bfloat16)
        assert exact_mismatches(got, ref, torch.bfloat16) > 0, name
        assert bound_ratio(got, ref, s, c, REL_BF16) > 1.0, name
