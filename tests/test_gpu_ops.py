"""Per-operator parity of the CUDA kernels (through the C ABI) against the CPU oracle and the
golden vectors recorded from the reference.  fp32 tolerance: max|d| / max|ref| <= 1e-4
(BASELINE north_star); most ops are far below that and are checked tighter."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import common
from oracle import texture_diffuser_ref as O

pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def OP():
    common.package()
    from dgtd_b200.twig.ops.functions import texture_diffusion_func
    return texture_diffusion_func


def dev(a):
    return torch.as_tensor(np.asarray(a)).float().cuda().contiguous()


def t64(a):
    return torch.as_tensor(np.asarray(a)).double()


def check(got, ref, tol=TOL):
    got = got.detach().float().cpu().double()
    ref = ref.double()
    assert tuple(got.shape) == tuple(ref.shape), (got.shape, ref.shape)
    assert torch.isfinite(got).all()
    err = float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
    assert err <= tol, f"rel err {err:.3e} > {tol}"
    return err


def test_library_loads_and_counts_launches(OP):
    from dgtd_b200.twig.ops import capi
    n0 = capi.launch_count()
    OP.surface_normals(torch.rand(1, 1, 8, 8).cuda())
    assert capi.launch_count() == n0 + 1


def test_surface_normals(OP, golden_ops):
    check(OP.surface_normals(dev(golden_ops["normals_in"])), t64(golden_ops["normals_out"]), 1e-6)


def test_fft_highpass_small_nonsquare(OP, golden_ops):
    check(OP.fft_highpass(dev(golden_ops["fft_in"])), t64(golden_ops["fft_out"]), 1e-5)


@pytest.mark.parametrize("S", [384, 352])
def test_fft_highpass_image_size(OP, S):
    x, _ = common.synthetic_inputs(2, S)
    check(OP.fft_highpass(x.cuda()), O.fft_highpass(x.double()), 1e-5)


def test_regressor_and_conv1x1(OP, golden_ops):
    w = dev(golden_ops["reg_w"]).reshape(24 * 49, 3).contiguous()
    got = OP.conv1x1_nchw(dev(golden_ops["reg_in"]), w, dev(golden_ops["reg_b"]), sigmoid=True)
    check(got, t64(golden_ops["reg_out"]), 1e-6)


@pytest.mark.parametrize("tag", ["mp24", "mp1"])
def test_message_passing_forward_backward(OP, golden_ops, tag):
    x = dev(golden_ops[f"{tag}_x"]).requires_grad_(True)
    w = dev(golden_ops[f"{tag}_w"]).requires_grad_(True)
    y = OP.message_passing_core(x, w, 4, 1e-5)
    check(y, t64(golden_ops[f"{tag}_core"]), 1e-5)
    y.backward(dev(golden_ops[f"{tag}_gout"]))
    check(x.grad, t64(golden_ops[f"{tag}_gx"]), 1e-5)
    check(w.grad, t64(golden_ops[f"{tag}_gw"]), 2e-5)


def test_message_passing_is_linear_and_mass_conserving(OP):
    """Size-independent properties: linear in x; interior of a constant field stays constant
    (weights are random-walk normalised), 32x32 plane = on-chip limit."""
    g = torch.Generator().manual_seed(3)
    x1, x2 = torch.randn(1, 4, 32, 32, generator=g).cuda(), torch.randn(1, 4, 32, 32, generator=g).cuda()
    w = torch.rand(1, 4 * 49, 32, 32, generator=g).cuda()
    a = OP.message_passing_core(x1, w, 3)
    b = OP.message_passing_core(x2, w, 3)
    ab = OP.message_passing_core(2.0 * x1 - 0.5 * x2, w, 3)
    assert float((ab - (2.0 * a - 0.5 * b)).abs().max()) < 1e-4
    ones = OP.message_passing_core(torch.ones_like(x1), w, 3)
    assert float((ones[:, :, 9:-9, 9:-9] - 1.0).abs().max()) < 1e-4


@pytest.mark.parametrize("n,h,w,c,T", [(1, 40, 70, 64, 1), (2, 17, 33, 64, 3), (1, 64, 64, 256, 2)])
def test_message_passing_tiled_large_map_variant(OP, n, h, w, c, T):
    """Halo-tiled TMA kernel (shared weights, NHWC) == the reference operator semantics."""
    g = torch.Generator().manual_seed(21)
    x = torch.randn(n, c, h, w, generator=g)
    wgt = torch.rand(n, 49, h, w, generator=g)
    ref = O.message_passing_core(x.double(), wgt.double(), 7, T)
    got = OP.message_passing_tiled(x.permute(0, 2, 3, 1).contiguous().cuda(), wgt.cuda(), T)
    check(got.permute(0, 3, 1, 2), ref, 1e-5)


@pytest.mark.parametrize("n,h,w,c,T", [(1, 40, 70, 32, 1), (2, 17, 33, 64, 3), (1, 48, 48, 96, 2)])
def test_message_passing_regress_generates_the_models_weights_on_chip(OP, n, h, w, c, T):
    """W2 mode of the microbench: per-channel weights sigmoid(Wr g + br) generated inside the kernel ==
    ShapePropWeightRegressor (cod.py:1051-1060) + MessagePassing core (cod.py:1190-1205) of the oracle.
    Regressor scaled so that the weights are far from the uniform 0.5 (SURVEY.md 8c)."""
    g = torch.Generator().manual_seed(31)
    x = torch.randn(n, c, h, w, generator=g)
    guide = torch.randn(n, 3, h, w, generator=g)
    reg_w = torch.randn(c * 49, 3, 1, 1, generator=g) * 0.8
    reg_b = torch.randn(c * 49, generator=g)
    wgt = O.regress_weights(guide.double(), reg_w.double(), reg_b.double())
    ref = O.message_passing_core(x.double(), wgt, 7, T)
    xc = x.permute(0, 2, 3, 1).contiguous().cuda()
    got = OP.message_passing_regress(xc, guide.cuda(), reg_w.cuda(), reg_b.cuda(), T)
    check(got.permute(0, 3, 1, 2), ref, 1e-5)
    # tanh.approx sigmoid (one MUFU op per weight): stated tolerance 2e-3 of max|ref|
    fast = OP.message_passing_regress(xc, guide.cuda(), reg_w.cuda(), reg_b.cuda(), T, fast_sigmoid=True)
    check(fast.permute(0, 3, 1, 2), ref, 2e-3)
    # bf16 storage / fp32 accumulate: one bf16 rounding per iteration
    xb = x.to(torch.bfloat16)
    refb = O.message_passing_core(xb.double(), wgt, 7, T)
    gotb = OP.message_passing_regress(xb.permute(0, 2, 3, 1).contiguous().cuda(), guide.cuda(), reg_w.cuda(),
                                      reg_b.cuda(), T, fast_sigmoid=True)
    check(gotb.float().permute(0, 3, 1, 2), refb, 4e-3 * T + 2e-3)


# 32 of the 256 channels (the operator is independent per channel): every residue mod 8 and every 64-channel
# chunk occurs, so each lane / register slot / TMA channel box of the kernels is sampled; keeps the float64
# oracle at seconds per crop
CH_SUBSET = torch.tensor([8 * i + (i % 8) for i in range(32)])


def _crop_reference(x_nhwc, wgt, T, y0, y1, x0, x1):
    """float64 oracle of rows [y0,y1) x cols [x0,x1) of a big map: the oracle runs on the crop + 3T halo (clamped
    to the map, so true borders keep the operator's zero padding) and only the crop proper is returned."""
    H, W = x_nhwc.shape[1:3]
    r = 3 * T
    ya, yb, xa, xb = max(0, y0 - r), min(H, y1 + r), max(0, x0 - r), min(W, x1 + r)
    xs = x_nhwc[:, ya:yb, xa:xb][..., CH_SUBSET].permute(0, 3, 1, 2).double().cpu()
    ws = wgt[:, :, ya:yb, xa:xb].double().cpu()
    ref = O.message_passing_core(xs, ws, 7, T)
    return ref[:, :, y0 - ya:y1 - ya, x0 - xa:x1 - xa]


CROPS_1024 = [(0, 160, 0, 160), (0, 160, 864, 1024), (864, 1024, 0, 160), (864, 1024, 864, 1024),     # corners
              (0, 160, 430, 590), (500, 660, 864, 1024), (437, 597, 443, 603), (120, 280, 504, 664)]  # edges, interior


@pytest.mark.parametrize("storage,T", [("fp32", 1), ("fp32", 4), ("bf16", 1), ("bf16", 4)])
def test_message_passing_tiled_at_microbench_size(OP, storage, T):
    """BASELINE configs[3] at FULL size (1024 x 1024 x 256; 8192 tiles, TMA boxes on every border): 8 crops of
    160 x 160 (4 corners, 2 edges, 2 interior, none tile-aligned in the interior) against the float64 oracle on the
    crop + 3T halo.  fp32 storage <= 1e-5; bf16 storage: one bf16 rounding per step (stated 6e-3 * T: tensor-pipe kernel, weights operand in bf16)."""
    g = torch.Generator().manual_seed(77)
    H = W = 1024
    C = 256
    x = torch.randn(1, H, W, C, generator=g)
    wgt = torch.rand(1, 49, H, W, generator=g)
    if storage == "bf16":
        x = x.to(torch.bfloat16)
    got = OP.message_passing_tiled(x.cuda(), wgt.cuda(), T)
    assert got.dtype == x.dtype and torch.isfinite(got).all()
    tol = 1e-5 if storage == "fp32" else 6e-3 * T
    worst = 0.0
    for (y0, y1, x0, x1) in CROPS_1024:
        ref = _crop_reference(x.float(), wgt, T, y0, y1, x0, x1)
        worst = max(worst, check(got[:, y0:y1, x0:x1][..., CH_SUBSET.cuda()].permute(0, 3, 1, 2), ref, tol))
    print(f"mp_tiled 1024^2 x 256 {storage} T={T}: worst crop rel err {worst:.3e}")


@pytest.mark.parametrize("storage,T", [("fp32", 1), ("bf16", 2)])
def test_message_passing_regress_at_microbench_size(OP, storage, T):
    """W2 (weights generated on chip) at 1024 x 1024 x 256: 3 crops of 96 x 96 against the float64 oracle."""
    g = torch.Generator().manual_seed(78)
    H = W = 1024
    C = 256
    x = torch.randn(1, H, W, C, generator=g)
    guide = torch.randn(1, 3, H, W, generator=g)
    reg_w = torch.randn(C * 49, 3, 1, 1, generator=g) * 0.8
    reg_b = torch.randn(C * 49, generator=g)
    if storage == "bf16":
        x = x.to(torch.bfloat16)
    got = OP.message_passing_regress(x.cuda(), guide.cuda(), reg_w.cuda(), reg_b.cuda(), T)
    r = 3 * T
    for (y0, y1, x0, x1) in [(0, 96, 0, 96), (928, 1024, 500, 596), (461, 557, 470, 566)]:
        ya, yb, xa, xb = max(0, y0 - r), min(H, y1 + r), max(0, x0 - r), min(W, x1 + r)
        rows = (CH_SUBSET[:, None] * 49 + torch.arange(49)[None, :]).reshape(-1)
        wts = O.regress_weights(guide[:, :, ya:yb, xa:xb].double(), reg_w[rows].double(), reg_b[rows].double())
        ref = O.message_passing_core(x[:, ya:yb, xa:xb][..., CH_SUBSET].permute(0, 3, 1, 2).double(), wts, 7, T)
        ref = ref[:, :, y0 - ya:y1 - ya, x0 - xa:x1 - xa]
        check(got[:, y0:y1, x0:x1][..., CH_SUBSET.cuda()].permute(0, 3, 1, 2), ref, 1e-5 if storage == "fp32" else 4e-3 * T)


@pytest.mark.parametrize("n,h,w,c,T", [(1, 40, 70, 256, 1), (2, 17, 33, 256, 3), (1, 64, 64, 512, 2), (1, 8, 16, 256, 1),
                                       (1, 5, 3, 256, 2), (3, 23, 16, 256, 1), (2, 200, 264, 256, 2)])
def test_message_passing_tensor_core_banded_gemm(OP, n, h, w, c, T):
    """mp_tc.cu: the step as Y[128 px, C] = A[128, 336] . X[336, C] on tcgen05 (bf16 storage).  Ragged maps (tiles
    clipped by TMA on both axes), maps smaller than one tile, two channel passes (C = 512), several images, T > 1.
    The last case has 850 tiles (> 148 CTAs: every CTA walks several tiles, the A ring is rewritten in flight).
    Stated tolerance 6e-3 * T of max|ref|: one bf16 rounding of the stored result per step (2^-9 of the element)
    plus the bf16 rounding of the normalised weights in the A operand (zero-mean, ~1e-3 of max|ref| at 4.5 sigma)."""
    g = torch.Generator().manual_seed(23)
    x = torch.randn(n, c, h, w, generator=g).to(torch.bfloat16)
    wgt = torch.rand(n, 49, h, w, generator=g)
    ref = O.message_passing_core(x.double(), wgt.double(), 7, T)
    xc = x.permute(0, 2, 3, 1).contiguous().cuda()
    got = OP.message_passing_tiled(xc, wgt.cuda(), T, impl="tc")
    assert got.dtype == torch.bfloat16
    err = check(got.float().permute(0, 3, 1, 2), ref, 6e-3 * T)
    simt = OP.message_passing_tiled(xc, wgt.cuda(), T, impl="simt") if c % 128 == 0 else None
    if simt is not None:      # the CUDA-core kernel of the same operator (fp32 weights): two independently bf16-rounded results
        d = float((got.float() - simt.float()).abs().max() / ref.abs().max())
        print(f"tc vs oracle {err:.2e}; vs SIMT kernel {d:.2e}")
        assert d <= 1e-2 * T


@pytest.mark.parametrize("n,h,w,c,T", [(1, 40, 72, 256, 1), (2, 17, 36, 256, 3), (1, 64, 64, 512, 2), (1, 8, 16, 256, 1),
                                       (1, 5, 4, 256, 2), (2, 200, 264, 256, 2)])
def test_message_passing_tensor_core_fp32_storage(OP, n, h, w, c, T):
    """mp_tc_f32.cu: fp32 storage on the tensor pipe as three bf16 products (A_hi X_hi + A_hi X_lo + A_lo X_hi,
    16 significant bits per operand): <= 1e-5 of max|ref| against the float64 oracle -- the bar of the CUDA-core
    kernel.  Ragged heights, maps smaller than a tile, two channel blocks, several images, 850 tiles, T > 1."""
    g = torch.Generator().manual_seed(29)
    x = torch.randn(n, c, h, w, generator=g)
    wgt = torch.rand(n, 49, h, w, generator=g)
    ref = O.message_passing_core(x.double(), wgt.double(), 7, T)
    xc = x.permute(0, 2, 3, 1).contiguous().cuda()
    got = OP.message_passing_tiled(xc, wgt.cuda(), T, impl="tc")
    assert got.dtype == torch.float32
    err = check(got.permute(0, 3, 1, 2), ref, 1e-5)
    simt = OP.message_passing_tiled(xc, wgt.cuda(), T, impl="simt")
    print(f"tc[fp32] vs oracle {err:.2e}; SIMT kernel vs oracle {common.rel_err(simt.permute(0, 3, 1, 2), ref):.2e}")


def test_message_passing_tensor_core_constant_map(OP):
    """Interior pixels of a constant map stay constant (weights sum to sum/(sum+eps)); borders lose exactly the
    weight of the taps that fall outside (zero padding, no renormalisation: cod.py:1204)."""
    h, w, c = 32, 48, 256
    x = torch.full((1, h, w, c), 1.5, dtype=torch.bfloat16).cuda()
    g = torch.Generator().manual_seed(24)
    wgt = torch.rand(1, 49, h, w, generator=g)
    got = OP.message_passing_tiled(x, wgt.cuda(), 1, impl="tc").float()
    assert float((got[:, 3:-3, 3:-3] - 1.5).abs().max()) <= 1.5 * 2 ** -8
    wn = wgt / (wgt.sum(1, keepdim=True) + 1e-5)
    inside = wn[:, [ky * 7 + kx for ky in range(3, 7) for kx in range(3, 7)]].sum(1)     # taps in-bounds at the (0,0) corner
    assert abs(float(got[0, 0, 0, 0]) - 1.5 * float(inside[0, 0, 0])) <= 1.5 * 2 ** -7


def test_message_passing_tiled_bf16_storage(OP):
    """bf16 storage / fp32 accumulate: exact on bf16-representable inputs up to the output rounding."""
    g = torch.Generator().manual_seed(22)
    n, h, w, c = 1, 24, 40, 128
    x = torch.randn(n, c, h, w, generator=g).to(torch.bfloat16)
    wgt = torch.rand(n, 49, h, w, generator=g)
    ref = O.message_passing_core(x.double(), wgt.double(), 7, 1)
    got = OP.message_passing_tiled(x.permute(0, 2, 3, 1).contiguous().cuda(), wgt.cuda(), 1)
    assert got.dtype == torch.bfloat16
    check(got.float().permute(0, 3, 1, 2), ref, 6e-3)


def test_message_passing_module_bilinear_upsample(OP, golden_ops):
    tag = "mp24"
    core = OP.message_passing_core(dev(golden_ops[f"{tag}_x"]), dev(golden_ops[f"{tag}_w"]), 4)
    y = OP.conv1x1_nchw(core, dev(golden_ops[f"{tag}_convw"]).reshape(3, 24).contiguous(),
                        dev(golden_ops[f"{tag}_convb"]))
    check(OP.resize_nchw(y, (48, 48), True), t64(golden_ops[f"{tag}_full"]), 1e-5)


def test_resize_nearest_and_bilinear_down(OP):
    x = torch.randn(2, 3, 48, 36)
    check(OP.resize_nchw(x.cuda(), (12, 12), False), O.nearest_grid(x.double(), 12), 1e-7)
    check(OP.resize_nchw(x.cuda(), (12, 12), True), O.bilinear_resize(x.double(), (12, 12)), 1e-5)
    check(OP.resize_nchw(x.cuda(), (96, 80), True), O.bilinear_resize(x.double(), (96, 80)), 1e-5)


def test_layer_norm_both_formats(OP, golden_ops):
    g = golden_ops
    check(OP.layer_norm(dev(g["ln_channels_first_in"]), dev(g["ln_channels_first_w"]),
                        dev(g["ln_channels_first_b"]), 1e-6, True), t64(g["ln_channels_first_out"]), 1e-5)
    check(OP.layer_norm(dev(g["ln_channels_last_in"]), dev(g["ln_channels_last_w"]),
                        dev(g["ln_channels_last_b"]), 1e-6, False), t64(g["ln_channels_last_out"]), 1e-5)


@pytest.mark.parametrize("S,B", [(48, 2), (384, 1)])
def test_diffusion_front(OP, S, B):
    """Fused nearest/regressor/normalise/depth-taps/4 iterations/1x1 conv vs the staged oracle."""
    g = torch.Generator().manual_seed(5)
    emb1 = torch.rand(B, 3, S, S, generator=g)
    depth = torch.rand(B, 1, S, S, generator=g)
    reg_w = torch.randn(24 * 49, 3, 1, 1, generator=g) * 0.8
    reg_b = torch.randn(24 * 49, generator=g)
    enc_w, enc_b = torch.randn(24, 1, 1, 1, generator=g), torch.randn(24, generator=g)
    cw, cb = torch.randn(3, 24, 1, 1, generator=g) * 0.3, torch.randn(3, generator=g)
    d = lambda v: v.double()
    wts = O.regress_weights(O.nearest_grid(d(emb1), 12), d(reg_w), d(reg_b))
    x0 = O.depth_to_grid(d(depth), d(enc_w), d(enc_b), 12)
    core = O.message_passing_core(x0, wts)
    ref = F.conv2d(core, d(cw), d(cb))
    got, states, wn = OP.diffusion_front(emb1.cuda(), depth.cuda(), reg_w.reshape(-1, 3).cuda().contiguous(),
                                         reg_b.cuda(), enc_w.reshape(-1).cuda().contiguous(), enc_b.cuda(),
                                         cw.reshape(3, 24).cuda().contiguous(), cb.cuda(), save_wn=True)
    check(got, ref, 1e-5)
    check(states[:, 0], x0, 1e-5)
    check(states[:, 4], core, 1e-5)
    wt = wts.reshape(B, 24, 49, 144)
    check(wn, wt / (wt.sum(2, keepdim=True) + 1e-5), 1e-5)


def test_stem_with_upsampled_grid(OP):
    g = torch.Generator().manual_seed(6)
    B, S, C = 2, 96, 128
    image, grid = torch.randn(B, 3, S, S, generator=g), torch.randn(B, 3, 12, 12, generator=g)
    w, b = torch.randn(C, 3, 4, 4, generator=g) * 0.2, torch.randn(C, generator=g) * 0.1
    lw, lb = 1 + 0.2 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    x = O.bilinear_resize(grid.double(), (S, S)) + image.double()
    ref = O.layer_norm_channels_first(F.conv2d(x, w.double(), b.double(), stride=4), lw.double(), lb.double())
    got = OP.stem(image.cuda(), grid.cuda(), w.reshape(C, 48).cuda().contiguous(), b.cuda(), lw.cuda(), lb.cuda())
    check(got.permute(0, 3, 1, 2), ref, 1e-5)
    got0 = OP.stem(image.cuda(), None, w.reshape(C, 48).cuda().contiguous(), b.cuda(), lw.cuda(), lb.cuda())
    ref0 = O.layer_norm_channels_first(F.conv2d(image.double(), w.double(), b.double(), stride=4), lw.double(), lb.double())
    check(got0.permute(0, 3, 1, 2), ref0, 1e-5)


@pytest.mark.parametrize("h,w", [(12, 12), (11, 10)])
def test_downsample_ln_patchify_linear(OP, h, w):
    from dgtd_b200.twig.ops.capi import F32
    g = torch.Generator().manual_seed(7)
    B, C = 2, 64
    x = torch.randn(B, C, h, w, generator=g) * 2 + 0.5
    lw, lb = 1 + 0.2 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    cw, cb = torch.randn(2 * C, C, 2, 2, generator=g) * 0.1, torch.randn(2 * C, generator=g) * 0.1
    ref = F.conv2d(O.layer_norm_channels_first(x.double(), lw.double(), lb.double()), cw.double(), cb.double(), stride=2)
    a = OP.ln_patchify(x.permute(0, 2, 3, 1).contiguous().cuda(), lw.cuda(), lb.cuda(), F32)
    wp = cw.permute(0, 2, 3, 1).reshape(2 * C, 4 * C).contiguous().cuda()
    y = OP.linear(a, wp, cb.cuda()).view(B, h // 2, w // 2, 2 * C)
    check(y.permute(0, 3, 1, 2), ref, 1e-5)


@pytest.mark.parametrize("C,h,w", [(32, 10, 12), (128, 9, 17), (512, 6, 5), (1024, 4, 4)])
def test_dwconv7_ln(OP, C, h, w):
    from dgtd_b200.twig.ops.capi import F32
    g = torch.Generator().manual_seed(8)
    B = 2
    x = torch.randn(B, C, h, w, generator=g)
    dw, db = torch.randn(C, 1, 7, 7, generator=g) * 0.2, torch.randn(C, generator=g) * 0.1
    lw, lb = 1 + 0.2 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    y = F.conv2d(x.double(), dw.double(), db.double(), padding=3, groups=C).permute(0, 2, 3, 1)
    ref = O.layer_norm_channels_last(y, lw.double(), lb.double())
    got = OP.dwconv7_ln(x.permute(0, 2, 3, 1).contiguous().cuda(), dw.reshape(C, 49).cuda().contiguous(),
                        db.cuda(), lw.cuda(), lb.cuda(), F32)
    check(got, ref, 1e-5)


@pytest.mark.parametrize("C,h,w,B", [(128, 96, 96, 1), (128, 20, 28, 2), (256, 48, 48, 1), (512, 24, 24, 2),
                                     (512, 22, 22, 1), (1024, 12, 12, 3), (1024, 11, 11, 2)])
def test_dwconv7_ln_tma_variant(OP, C, h, w, B):
    from dgtd_b200.twig.ops.capi import F32
    g = torch.Generator().manual_seed(18)
    x = torch.randn(B, C, h, w, generator=g)
    dw, db = torch.randn(C, 1, 7, 7, generator=g) * 0.2, torch.randn(C, generator=g) * 0.1
    lw, lb = 1 + 0.2 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    y = F.conv2d(x.double(), dw.double(), db.double(), padding=3, groups=C).permute(0, 2, 3, 1)
    ref = O.layer_norm_channels_last(y, lw.double(), lb.double())
    xn = x.permute(0, 2, 3, 1).contiguous().cuda()
    ws = torch.empty(xn.numel(), device="cuda")
    got = OP.dwconv7_ln_tma(xn, dw.reshape(C, 49).t().contiguous().cuda(), db.cuda(), lw.cuda(), lb.cuda(), F32, ws)
    check(got, ref, 1e-5)


@pytest.mark.parametrize("M,N,K,act", [(300, 128, 64, 0), (257, 24, 128, 1), (128, 320, 216, 2), (1000, 512, 2048, 1)])
def test_linear_fp32_exact_path(OP, M, N, K, act):
    g = torch.Generator().manual_seed(9)
    a, w, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    ref = a.double() @ w.double().t() + b.double()
    ref = O.gelu_erf(ref) if act == 1 else (ref.clamp_min(0) if act == 2 else ref)
    check(OP.linear(a.cuda(), w.cuda(), b.cuda(), act=act), ref, 1e-5)


def test_linear_residual_fp32(OP):
    g = torch.Generator().manual_seed(10)
    B, rows, N, K = 3, 50, 64, 256
    M = B * rows
    a, w = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / 16
    b, gam = torch.randn(N, generator=g), torch.randn(N, generator=g)
    keep = torch.tensor([0.0, 1.25, 1.25])
    res = torch.randn(M, N, generator=g)
    ref = res.double() + keep.double().repeat_interleave(rows)[:, None] * (gam.double() * (a.double() @ w.double().t() + b.double()))
    r = res.clone().cuda()
    OP.linear_residual_(a.cuda(), w.cuda(), b.cuda(), gam.cuda(), keep.cuda(), rows, r)
    check(r, ref, 1e-5)


def test_convnext_block_fp32_vs_reference_golden(golden_ops):
    TD = common.package()
    blk = TD.convnext_Block(32, drop_path=0.2, layer_scale_init_value=1.0)
    sd = {k[len("blk_p_"):]: torch.as_tensor(v).float() for k, v in golden_ops.items() if k.startswith("blk_p_")}
    blk.load_state_dict(sd)
    blk = blk.cuda().eval()
    TD.set_precision(blk, "fp32")
    with torch.no_grad():
        y = blk(dev(golden_ops["blk_in"]))
    assert y.shape == (2, 32, 10, 12)
    check(y, t64(golden_ops["blk_out"]), 2e-5)


def test_fusion_sum(OP):
    """ShapePropEncoder head (cod.py:1171-1176) with the 1x1 fusion conv folded into the level projections, as
    `_head` calls it: z_i = lv_i Wf_i^T per level, then bias + sum_i bilinear_up(z_i) against the un-folded
    conv2d(cat(bilinear_up(lv_i)), Wf, bf)."""
    g = torch.Generator().manual_seed(11)
    B, C = 2, 24
    hw = [(24, 20), (12, 10), (6, 5), (3, 3)]
    lv = [torch.randn(B, C, h, w, generator=g) for h, w in hw]
    wf, bf = torch.randn(C, 4 * C, 1, 1, generator=g) * 0.2, torch.randn(C, generator=g)
    cat = torch.cat([O.bilinear_resize(v.double(), hw[0]) for v in lv], 1)
    ref = F.conv2d(cat, wf.double(), bf.double())
    wf2 = wf.reshape(C, 4 * C).double()
    z = [(v.double().permute(0, 2, 3, 1).reshape(-1, C) @ wf2[:, i * C:(i + 1) * C].T).float().contiguous().cuda()
         for i, v in enumerate(lv)]
    nhwc, nchw, pad = OP.fusion_sum(z, hw, bf.cuda(), B, want_nhwc=True, want_nchw=True, pad_to=32)
    check(nchw, ref, 1e-5)
    check(nhwc.permute(0, 3, 1, 2), ref, 1e-5)
    check(pad[..., :C].float().permute(0, 3, 1, 2), ref, 1e-2)   # bf16 storage
    assert float(pad[..., C:].float().abs().max()) == 0.0


def test_decoder_convs_and_folded_injection(golden_ops):
    """ShapePropDecoder through the implicit-GEMM convs; injection through the folded 4x4 conv
    (ratios 2, 4, 8) must equal conv + F.interpolate(bilinear) of the reference."""
    TD = common.package()
    from dgtd_b200.twig.model.texture_diffuser import _decode_tokens
    from dgtd_b200.twig.ops.functions import texture_diffusion_func as OPS
    dec = TD.ShapePropDecoder(40, 24)
    dec.load_state_dict({k[len("dec_p_"):]: torch.as_tensor(v).float() for k, v in golden_ops.items()
                         if k.startswith("dec_p_")})
    dec = dec.cuda().eval()
    emb = dev(golden_ops["dec_in"])
    with torch.no_grad():
        y = dec(emb)
        check(y, t64(golden_ops["dec_out"]), 1e-5)
        nhwc = OPS.nchw_to_nhwc(emb)
        for n in (16, 8, 4, 2):
            tok = _decode_tokens([dec], nhwc, (n, n))[0]
            ref = t64(golden_ops[f"dec_tokens{n}"]) if n < 16 else t64(golden_ops["dec_out"]).flatten(2).permute(0, 2, 1)
            check(tok, ref, 1e-5)
        # non-integer ratio falls back to conv + NHWC bilinear resize
        tok = _decode_tokens([dec], nhwc, (5, 7))[0]
        ref = O.prompt_to_tokens(t64(golden_ops["dec_out"]), (5, 7))
        check(tok, ref, 1e-5)


def test_layout_and_cast_round_trip(OP):
    x = torch.randn(2, 24, 7, 9).cuda()
    nhwc = OP.nchw_to_nhwc(x, ld=32)
    assert nhwc.shape == (2, 7, 9, 32) and float(nhwc[..., 24:].abs().max()) == 0.0
    assert torch.equal(OP.nhwc_to_nchw(nhwc, C=24), x)
    b = OP.cast(x, torch.bfloat16)
    assert torch.equal(b, x.to(torch.bfloat16))
    assert torch.equal(OP.cast(b, torch.float32), b.float())


def test_errors_are_python_exceptions(OP):
    with pytest.raises(RuntimeError, match="multiples of 4"):
        OP.fft_highpass(torch.randn(1, 1, 10, 10).cuda())
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        OP.surface_normals(torch.rand(1, 1, 4, 4))
    with pytest.raises(RuntimeError, match="must be 1 or"):
        OP.message_passing_core(torch.randn(1, 4, 8, 8).cuda(), torch.rand(1, 2 * 49, 8, 8).cuda(), 2)


def test_diffusion_stage_modules_are_differentiable(golden_ops):
    """MessagePassing (core + 1x1 conv + bilinear up) and ShapePropWeightRegressor through the
    CUDA autograd Functions vs float64 autograd of the oracle: gradients w.r.t. the depth state,
    the guide image, the regressor and the 24->3 conv (backward obligations a4/a6)."""
    TD = common.package()
    g = torch.Generator().manual_seed(31)
    n, c, h, w = 2, 24, 12, 12
    xx = torch.rand(n, 3, h, w, generator=g)
    x0 = torch.randn(n, c, h, w, generator=g)
    reg = TD.ShapePropWeightRegressor(3, c)
    mp = TD.MessagePassing(c, img_size=48)
    with torch.no_grad():
        reg.reg.weight.normal_(0, 1.0, generator=g); reg.reg.bias.normal_(0, 1.0, generator=g)
        mp.conv.weight.normal_(0, 0.5, generator=g); mp.conv.bias.normal_(0, 0.5, generator=g)
    gout = torch.randn(n, 3, 48, 48, generator=g)
    # oracle (float64 autograd)
    P = {k: v.detach().double().requires_grad_(True) for k, v in
         dict(rw=reg.reg.weight, rb=reg.reg.bias, cw=mp.conv.weight, cb=mp.conv.bias).items()}
    xx64, x064 = xx.double().requires_grad_(True), x0.double().requires_grad_(True)
    ref = O.message_passing(x064, O.regress_weights(xx64, P["rw"], P["rb"]), P["cw"], P["cb"], (48, 48))
    refg = torch.autograd.grad(ref, [x064, xx64, P["rw"], P["rb"], P["cw"], P["cb"]], gout.double())
    # CUDA modules
    reg, mp = reg.cuda(), mp.cuda()
    xx_d, x0_d = xx.cuda().requires_grad_(True), x0.cuda().requires_grad_(True)
    out = mp(x0_d, reg(xx_d))
    check(out, ref.detach(), 1e-5)
    out.backward(gout.cuda())
    got = [x0_d.grad, xx_d.grad, reg.reg.weight.grad, reg.reg.bias.grad, mp.conv.weight.grad, mp.conv.bias.grad]
    for a, b, name in zip(got, refg, ["x0", "guide", "reg.w", "reg.b", "conv.w", "conv.b"]):
        assert a is not None, name
        check(a, b, 5e-5)


def test_bilinear_resize_adjoint_identity():
    """<R x, y> == <x, R^T y> for up- and down-sampling (exact adjoint of F.interpolate)."""
    common.package()
    from dgtd_b200.twig.ops.functions import texture_diffusion_func as OPS
    g = torch.Generator().manual_seed(32)
    for (h, w, oh, ow) in [(12, 12, 384, 384), (12, 10, 37, 51), (48, 36, 12, 12)]:
        x = torch.randn(2, 3, h, w, generator=g).cuda().requires_grad_(True)
        y = torch.randn(2, 3, oh, ow, generator=g).cuda()
        r = OPS.resize_bilinear_nchw_autograd(x, (oh, ow))
        lhs = float((r.detach().double() * y.double()).sum())
        r.backward(y)
        rhs = float((x.detach().double() * x.grad.double()).sum())
        assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs)), (h, w, oh, ow, lhs, rhs)


# ---- randomized shape sweeps (hypothesis), oracle = float64 torch on the same inputs ---------------
from hypothesis import given, settings, strategies as st, HealthCheck

_sweep = settings(max_examples=12, deadline=None, derandomize=True,
                  suppress_health_check=[HealthCheck.function_scoped_fixture])


@_sweep
@given(n=st.integers(1, 3), c=st.integers(1, 5), h=st.integers(1, 20), w=st.integers(1, 20),
       shared=st.booleans(), T=st.integers(0, 5))
def test_sweep_message_passing_core(OP, n, c, h, w, shared, T):
    g = torch.Generator().manual_seed(1000 * n + 100 * c + 10 * h + w)
    x = torch.randn(n, c, h, w, generator=g)
    wgt = torch.rand(n, (1 if shared else c) * 49, h, w, generator=g)
    ref = O.message_passing_core(x.double(), wgt.double(), 7, T)
    check(OP.message_passing_core(x.cuda(), wgt.cuda(), T), ref, 1e-5)


@_sweep
@given(M=st.integers(1, 700), N4=st.integers(1, 40), K4=st.integers(1, 40), act=st.sampled_from([0, 1, 2]))
def test_sweep_linear_fp32(OP, M, N4, K4, act):
    N, K = 4 * N4, 4 * K4
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    a, w, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    ref = a.double() @ w.double().t() + b.double()
    ref = O.gelu_erf(ref) if act == 1 else (ref.clamp_min(0) if act == 2 else ref)
    check(OP.linear(a.cuda(), w.cuda(), b.cuda(), act=act), ref, 1e-5)


@_sweep
@given(planes=st.integers(1, 4), h=st.integers(1, 30), w=st.integers(1, 30), oh=st.integers(1, 40), ow=st.integers(1, 40))
def test_sweep_bilinear_resize(OP, planes, h, w, oh, ow):
    x = torch.randn(1, planes, h, w, generator=torch.Generator().manual_seed(h * 31 + w))
    check(OP.resize_nchw(x.cuda(), (oh, ow), True), O.bilinear_resize(x.double(), (oh, ow)), 2e-5)


@_sweep
@given(B=st.integers(1, 2), h4=st.integers(3, 12), w4=st.integers(3, 12))
def test_sweep_fft_highpass_sizes(OP, B, h4, w4):
    """H, W multiples of 4 (the only constraint of the projector form); non-square, tiny, line = 0 .. n/2."""
    H, W = 4 * h4, 4 * w4
    x = torch.randn(B, 3, H, W, generator=torch.Generator().manual_seed(H * 100 + W))
    check(OP.fft_highpass(x.cuda()), O.fft_highpass(x.double()), 2e-5)


def test_fft_highpass_properties_at_full_size(OP):
    """Size-independent properties at 384^2, B=8: output >= 0; the operator |x - P x| kills what P keeps
    (a pure low-frequency image maps to ~0) and leaves a pure high-frequency image unchanged in magnitude."""
    S = 384
    yy, xx = torch.meshgrid(torch.arange(S, dtype=torch.float64), torch.arange(S, dtype=torch.float64), indexing="ij")
    low = torch.cos(2 * torch.pi * 5 * yy / S) * torch.cos(2 * torch.pi * 40 * xx / S)       # |k| < 105: removed band
    high = torch.cos(2 * torch.pi * 150 * yy / S) * torch.cos(2 * torch.pi * 120 * xx / S)   # outside the band
    mixed = torch.cos(2 * torch.pi * 5 * yy / S) * torch.cos(2 * torch.pi * 150 * xx / S)    # one axis outside: kept
    x = torch.stack([low, high, mixed]).float()[None].repeat(8, 1, 1, 1).cuda()
    y = OP.fft_highpass(x)
    assert float(y.min()) >= 0.0
    assert float(y[:, 0].abs().max()) < 1e-4
    assert float((y[:, 1] - x[:, 1].abs()).abs().max()) < 1e-4
    assert float((y[:, 2] - x[:, 2].abs()).abs().max()) < 1e-4


@pytest.mark.parametrize("B,H,W", [(2, 384, 384), (1, 96, 160), (3, 352, 352)])
def test_fft_highpass_tensor_core_variant_is_fp32_accurate(OP, B, H, W):
    """Projector products on tcgen05 with the two-term bf16 split, each product as one K-concatenated GEMM: within
    2e-5 of the float64 oracle (relative to max|ref|), i.e. the same bar as the exact CUDA-core variant up to the
    split's 2^-16 terms."""
    g = torch.Generator().manual_seed(H + W)
    x = torch.randn(B, 3, H, W, generator=g)
    ref = O.fft_highpass(x.double(), 0.3)
    got = OP.fft_highpass(x.cuda(), 0.3, tensor_cores=True)
    assert check(got, ref, 2e-5) <= 2e-5
    exact = OP.fft_highpass(x.cuda(), 0.3)
    check(exact, ref, 1e-5)


def test_standalone_layernorm_is_differentiable_and_dwconv_forward_runs():
    """VERDICT r1 boundary holes: the custom `LayerNorm` called on its own builds a graph (both data formats), and
    `pvt.DWConv.forward(x, H, W)` is callable like the reference's (cod.py:1520-1531)."""
    TD = common.package()
    from dgtd_b200.twig.model import pvt
    g = torch.Generator().manual_seed(41)
    for fmt, shape in (("channels_last", (2, 5, 7, 64)), ("channels_first", (2, 64, 5, 7))):
        ln = TD.LayerNorm(64, eps=1e-6, data_format=fmt).cuda()
        with torch.no_grad():
            ln.weight.copy_(1.0 + 0.3 * torch.randn(64, generator=g))
            ln.bias.copy_(0.3 * torch.randn(64, generator=g))
        x = torch.randn(shape, generator=g)
        go = torch.randn(shape, generator=g)
        xg = x.cuda().requires_grad_(True)
        y = ln(xg)
        y.backward(go.cuda())
        x64 = x.double().requires_grad_(True)
        w64, b64 = ln.weight.detach().double().cpu().requires_grad_(True), ln.bias.detach().double().cpu().requires_grad_(True)
        if fmt == "channels_last":
            r = F.layer_norm(x64, (64,), w64, b64, 1e-6)
        else:
            u = x64.mean(1, keepdim=True)
            v = (x64 - u).pow(2).mean(1, keepdim=True)
            r = w64[:, None, None] * ((x64 - u) / torch.sqrt(v + 1e-6)) + b64[:, None, None]
        r.backward(go.double())
        check(y, r.detach(), 1e-5)
        check(xg.grad, x64.grad, 1e-4)
        check(ln.weight.grad, w64.grad, 1e-4)
        check(ln.bias.grad, b64.grad, 1e-4)
    dw = pvt.DWConv(64).cuda()
    x = torch.randn(2, 6 * 10, 64, generator=g)
    got = dw(x.cuda(), 6, 10)
    ref = F.conv2d(x.double().transpose(1, 2).reshape(2, 64, 6, 10), dw.dwconv.weight.detach().double().cpu(),
                   dw.dwconv.bias.detach().double().cpu(), padding=1, groups=64).flatten(2).transpose(1, 2)
    check(got, ref, 1e-5)
