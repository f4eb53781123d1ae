"""GPU parity at the layer shapes BASELINE configs 4 / 5 actually run (VERDICT r01 weak #1): every code path of the
conv engine that the 256x256 BigGAN-Deep step selects -- multi-K-block generic tiles, the halo-row kernel's resident and
ring filter paths, the 64-channel weight-gradient kernel, split-K / per-image weight gradients, small-map 1x1 layers
with many channel tiles -- against plain fp32 torch on the CPU.  Tolerances as in test_gpu_parity.py: one bf16 rounding of the output (8e-3 max-norm),
fp32 accumulation of bf16 products for weight gradients (2e-3).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from test_gpu_parity import _cuda, bfr, rel_err, to_nhwc  # noqa: E402


# (B, H, W, Cin, Cout, k): which kernel / path it selects at these sizes
BENCH_SHAPES = [
    (32, 4, 4, 2048, 512, 1),     # 1x1 2048->512 @4x4, B=32: 32 K blocks, 4 pixel tiles x 4 channel tiles (8-GPU operating point)
    (4, 4, 4, 512, 2048, 1),      # 1x1 512->2048 @4x4: 8 channel tiles of 256
    (2, 16, 16, 512, 512, 3),     # 3x3 512->512 @16x16: generic per-tap kernel, 72 K iterations, direct-store epilogue
    (1, 128, 128, 128, 128, 3),   # 3x3 128->128 @128x128: halo-row kernel, filter ring (2 K blocks)
    (1, 256, 256, 64, 64, 3),     # 3x3 64->64 @256x256: halo-row kernel, resident taps + wgrad3x3_c64
    (2, 64, 64, 256, 256, 3),     # 3x3 256->256 @64x64: generic kernel at the roofline shape
    (2, 128, 128, 64, 256, 1),    # write-dominated 1x1 (TMA-store epilogue, two staging tiles per team)
    (1, 256, 256, 128, 64, 1),    # read-dominated 1x1 at 256x256
    (2, 64, 64, 512, 64, 1),      # attention-adjacent 1x1 (theta / phi)
]


@pytest.mark.parametrize("B,H,W,Cin,Cout,k", BENCH_SHAPES)
def test_conv_fwd_bwd_at_bench_shapes(B, H, W, Cin, Cout, k):
    from sgb200 import autograd_ops as A
    dev = _cuda()
    g = torch.Generator().manual_seed(B * 1000 + Cin + Cout + k)
    x = bfr(torch.randn(B, Cin, H, W, generator=g))
    w = torch.randn(Cout, Cin, k, k, generator=g) * (1.0 / np.sqrt(Cin * k * k))
    b = torch.randn(Cout, generator=g)
    dy = bfr(torch.randn(B, Cout, H, W, generator=g))
    xr, wr, br = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    yr = F.conv2d(xr, bfr(wr.detach()) + (wr - wr.detach()), br, padding=k // 2)
    yr.backward(dy)
    xd = to_nhwc(x, dev).requires_grad_(True)
    wd, bd = w.to(dev).requires_grad_(True), b.to(dev).requires_grad_(True)
    y = A.ConvFn.apply(xd, wd, bd, None, {"KH": k, "KW": k, "pad": k // 2})
    y.backward(to_nhwc(dy, dev))
    assert rel_err(y, yr) < 8e-3
    assert rel_err(xd.grad, xr.grad) < 8e-3
    assert rel_err(wd.grad, wr.grad) < 2e-3
    assert rel_err(bd.grad, br.grad) < 2e-3


def test_per_image_wgrad_at_attention_size():
    """Per-image weight gradient at N = 4096 pixels (attention dK / dV of BASELINE config 4): dphi[b] = dS[b]^T theta[b]
    with theta [B, 64, 64x64], dS [B, M = 1024, 64x64]."""
    from sgb200 import kernels as K
    dev = _cuda()
    g = torch.Generator().manual_seed(5)
    B, c8, M, S = 2, 64, 1024, 64
    theta = bfr(torch.randn(B, c8, S, S, generator=g))
    dS = bfr(torch.randn(B, M, S, S, generator=g) * 0.1)
    got = K.conv_wgrad(to_nhwc(theta, dev), to_nhwc(dS, dev), 1, 1, 0, 0, per_image=True)     # [B][M][1][c8]
    ref = torch.einsum("bmn,bcn->bmc", dS.flatten(2).double(), theta.flatten(2).double())
    assert rel_err(got.view(B, M, c8), ref) < 2e-3


# ------------------------------------------------------------------------------------------------ full model at 256x256
def _digest_errors(net, g, prefix):
    """Checks a gradient against tests/golden/make_golden.py::grad_digest: full tensors where stored, else norm + seeded
    +-1 projections.  Returns (worst relative error over full tensors, worst norm ratio error, worst projection error in
    units of the reference norm)."""
    gmax = max(float(g[prefix + "norm/" + n]) for n, _ in net.named_parameters())
    worst_full, worst_norm, worst_proj = (0.0, ""), (0.0, ""), (0.0, "")
    for i, (n, p) in enumerate(net.named_parameters()):
        got = p.grad.detach().double().cpu().flatten()
        rn = float(g[prefix + "norm/" + n])
        floor = rn + 1e-3 * gmax
        r = torch.randint(0, 2, (8, got.numel()), generator=torch.Generator().manual_seed(1000 + i)).double() * 2 - 1
        pe = float(((r @ got) - torch.from_numpy(g[prefix + "proj/" + n])).abs().max()) / floor
        worst_proj = max(worst_proj, (pe, n))
        worst_norm = max(worst_norm, (abs(float(got.norm()) - rn) / floor, n))
        if prefix + "full/" + n in g.files:
            ref = torch.from_numpy(g[prefix + "full/" + n]).double().flatten()
            worst_full = max(worst_full, (float((got - ref).norm()) / floor, n))
    return worst_full, worst_norm, worst_proj


def _digest_median(net, g, prefix):
    gmax = max(float(g[prefix + "norm/" + n]) for n, _ in net.named_parameters())
    errs = []
    for n, p in net.named_parameters():
        if prefix + "full/" + n in g.files:
            ref = torch.from_numpy(g[prefix + "full/" + n]).double().flatten()
            errs.append(float((p.grad.detach().double().cpu().flatten() - ref).norm() / (ref.norm() + 1e-3 * gmax)))
    return float(np.median(errs))


def test_biggan_deep_256_d_and_g_phase_vs_reference_golden(golden_dir):
    """BASELINE config 4's topology at its resolution -- 256x256, g_depth = d_depth = 2, attention at 64x64 (N = 4096,
    M = 1024), six up / down-sampling stages -- with conv_dim 16, against the reference's own CPU numbers
    (tests/golden/deep256_c16_attn_d2.npz).  Weights and inputs are regenerated from the seeds the generator script used
    (the parameter L1 checksums prove both sides hold the same values).  Tolerances: relative L2 4e-2 on discriminator
    features / logits and 1e-1 on discriminator-phase gradients, as for the 32x32 goldens.  The generated IMAGE passes
    through 12 blocks = 49 (conditional) batch norms with bf16 storage in between: rounding the fp32 oracle to bf16 at the
    same points on the CPU (tests/diag_bf16_emulation.py machinery) gives 0.061 relative L2 against this golden, the CUDA
    path measures 0.069 -- stated bound 1e-1.  Generator-phase gradients (B = 16) travel back through D and G's 49-deep
    batch-norm chain with bf16 storage: the same CPU emulation gives median 0.047 and worst-tensor 0.48 (a cBN gain weight
    at 8x8 whose gradient is a heavily cancelling sum) -- stated bounds: median <= 0.08, worst <= 0.75, projections <= 1.5
    reference norms."""
    import importlib
    import os
    from sgb200 import config as C
    from sgb200.utils import losses
    from test_gpu_parity import l2_err
    dev = _cuda()
    g = np.load(os.path.join(golden_dir, "deep256_c16_attn_d2.npz"))
    deep = importlib.import_module("sgb200.models.big_resnet_deep_legacy")
    torch.manual_seed(1234)
    M = C.make_modules(True, True, "cBN", "big_resnet_deep_legacy")
    MODEL = C._Section(info_type="N/A", g_info_injection="N/A")
    G = deep.Generator(z_dim=16, g_shared_dim=16, img_size=256, g_conv_dim=16, apply_attn=True, attn_g_loc=[4], g_cond_mtd="cBN",
                       num_classes=5, g_init="ortho", g_depth=2, mixed_precision=False, MODULES=M, MODEL=MODEL)
    D = deep.Discriminator(img_size=256, d_conv_dim=16, apply_d_sn=True, apply_attn=True, attn_d_loc=[2], d_cond_mtd="PD",
                           aux_cls_type="W/O", d_embed_dim="N/A", normalize_d_embed=False, num_classes=5, d_init="ortho",
                           d_depth=2, mixed_precision=False, MODULES=M, MODEL=MODEL)
    from sgb200.utils import ops
    with torch.no_grad():
        for mod in list(G.modules()) + list(D.modules()):
            if isinstance(mod, ops.SelfAttention):
                mod.sigma.fill_(0.37)
    l1g = sum(float(p.detach().double().abs().sum()) for p in G.parameters())
    l1d = sum(float(p.detach().double().abs().sum()) for p in D.parameters())
    assert abs(l1g - float(g["param_l1_G"])) < 1e-6 * l1g and abs(l1d - float(g["param_l1_D"])) < 1e-6 * l1d
    gi = torch.Generator().manual_seed(77)
    z = torch.randn(16, 16, generator=gi)
    yf = torch.randint(0, 5, (16,), generator=gi)
    real = torch.rand(16, 3, 256, 256, generator=gi) * 2 - 1
    yr = torch.randint(0, 5, (16,), generator=gi)
    assert torch.equal(yf, torch.from_numpy(g["y_fake"])) and torch.equal(yr, torch.from_numpy(g["y_real"]))   # index path: bit exact
    assert abs(float(real.double().sum()) - float(g["real_sum"])) < 1e-6
    G, D = G.to(dev).train(), D.to(dev).train()
    z, yf, real, yr = z.to(dev), yf.to(dev), real.to(dev), yr.to(dev)
    for p in G.parameters():
        p.requires_grad_(False)
    fake = G(z, yf)
    assert fake.shape == (16, 3, 256, 256)
    assert l2_err(fake[:, :, ::8, ::8], torch.from_numpy(g["fake_sub8"])) < 1e-1
    real_d, fake_d = D(real, yr), D(fake.detach(), yf)
    assert l2_err(real_d["h"], torch.from_numpy(g["h_real"])) < 4e-2
    assert l2_err(real_d["adv_output"], torch.from_numpy(g["adv_real"])) < 4e-2
    assert l2_err(fake_d["adv_output"], torch.from_numpy(g["adv_fake"])) < 4e-2
    d_loss = losses.d_wasserstein(real_d["adv_output"], fake_d["adv_output"])
    d_loss.backward()
    assert abs(float(d_loss) - float(g["d_loss"])) < 5e-2 * max(1.0, abs(float(g["d_loss"])))
    wf, wn, wp = _digest_errors(D, g, "Dgrad/")
    assert wf[0] < 1e-1 and wn[0] < 1e-1 and wp[0] < 3e-1, (wf, wn, wp)
    for n, b in D.named_buffers():
        if "weight_u" in n:
            assert rel_err(b, torch.from_numpy(g["D1/" + n])) < 1e-2, n
    for n, b in G.named_buffers():
        if "weight_u" in n or "running_" in n:
            assert rel_err(b, torch.from_numpy(g["G1/" + n])) < 1e-2, n
    D.zero_grad(set_to_none=True)
    for p in G.parameters():
        p.requires_grad_(True)
    for p in D.parameters():
        p.requires_grad_(False)
    fake2 = G(z, yf)
    assert l2_err(fake2[:, :, ::8, ::8], torch.from_numpy(g["fake2_sub8"])) < 1e-1
    g_loss = losses.g_wasserstein(D(fake2, yf)["adv_output"])
    g_loss.backward()
    assert abs(float(g_loss) - float(g["g_loss"])) < 5e-2 * abs(float(g["g_loss"]))
    wf, wn, wp = _digest_errors(G, g, "Ggrad/")
    assert wf[0] < 0.75 and wn[0] < 0.75 and wp[0] < 1.5, (wf, wn, wp)
    assert _digest_median(G, g, "Ggrad/") < 0.08


# ------------------------------------------------------------------------------------------------ multi-rank numerics
def test_two_ranks_reproduce_one_rank_on_the_global_batch():
    """2 ranks x 4 images with sync-BN groups + the arena gradient all-reduce == 1 rank x 8 images: D-phase and G-phase
    gradients (relative L2 <= 1e-1, the single-GPU gradient tolerance; typically ~1e-2), losses, BN running statistics
    (1e-2).  Needs two GPUs (skipped on a one-GPU box; bench.py runs the same check at every N > 1 and reports it)."""
    import json
    import os
    import subprocess
    import sys
    _cuda()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29500 + os.getpid() % 1000
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(root, "tests", "multirank_gpu_check.py")],
                       capture_output=True, text=True, timeout=600)
    lines = [l for l in r.stdout.splitlines() if l.startswith("MULTIRANK_CHECK ")]
    assert r.returncode == 0 and lines, r.stdout[-2000:] + r.stderr[-2000:]
    out = json.loads(lines[-1][len("MULTIRANK_CHECK "):])
    assert out["ok"], out


# ------------------------------------------------------------------------------------------------ DCGAN (BASELINE config 1)
def test_dcgan_layers_conv_transpose_and_strided_conv():
    """ConvTranspose2d / Conv2d with kernel 4, stride 2, padding 1 (src/models/deep_conv.py:20,140) through the stride-1
    engine identities of csrc/resample.cu, forward and every gradient, against torch on the CPU."""
    from sgb200.utils import ops
    dev = _cuda()
    g = torch.Generator().manual_seed(21)
    # transposed convolution 64 -> 32, 8x8 -> 16x16
    x = bfr(torch.randn(3, 64, 8, 8, generator=g))
    ct = ops.deconv2d(64, 32, 4, 2, 1)
    with torch.no_grad():
        ct.weight.copy_(torch.randn(64, 32, 4, 4, generator=g) * 0.05)
        ct.bias.copy_(torch.randn(32, generator=g) * 0.1)
    dy = bfr(torch.randn(3, 32, 16, 16, generator=g))
    xr = x.clone().requires_grad_(True)
    wr, br = ct.weight.detach().clone().requires_grad_(True), ct.bias.detach().clone().requires_grad_(True)
    yr = F.conv_transpose2d(xr, bfr(wr.detach()) + (wr - wr.detach()), br, stride=2, padding=1)
    yr.backward(dy)
    ct = ct.to(dev)
    xd = to_nhwc(x, dev).requires_grad_(True)
    y = ct(xd)
    y.backward(to_nhwc(dy, dev))
    assert rel_err(y, yr) < 8e-3 and rel_err(xd.grad, xr.grad) < 8e-3
    assert rel_err(ct.weight.grad, wr.grad) < 2e-3 and rel_err(ct.bias.grad, br.grad) < 2e-3
    # strided convolution 32 -> 48, 16x16 -> 8x8
    x = bfr(torch.randn(3, 32, 16, 16, generator=g))
    cv = ops.conv2d(32, 48, 4, 2, 1)
    with torch.no_grad():
        cv.weight.copy_(torch.randn(48, 32, 4, 4, generator=g) * 0.05)
        cv.bias.copy_(torch.randn(48, generator=g) * 0.1)
    dy = bfr(torch.randn(3, 48, 8, 8, generator=g))
    xr = x.clone().requires_grad_(True)
    wr, br = cv.weight.detach().clone().requires_grad_(True), cv.bias.detach().clone().requires_grad_(True)
    yr = F.conv2d(xr, bfr(wr.detach()) + (wr - wr.detach()), br, stride=2, padding=1)
    yr.backward(dy)
    cv = cv.to(dev)
    xd = to_nhwc(x, dev).requires_grad_(True)
    y = cv(xd)
    assert y.shape == yr.shape
    y.backward(to_nhwc(dy, dev))
    assert rel_err(y, yr) < 8e-3 and rel_err(xd.grad, xr.grad) < 8e-3
    assert rel_err(cv.weight.grad, wr.grad) < 2e-3 and rel_err(cv.bias.grad, br.grad) < 2e-3


def test_dcgan_config1_d_and_g_phase_vs_reference_golden(golden_dir):
    """BASELINE config 1 as a product path: models.deep_conv on the kernel set against the reference's DCGAN golden
    (tests/golden/dcgan32.npz; weights regenerated from the seed on both sides).  Tolerances of the 32x32 goldens: images /
    logits 4e-2 relative L2, losses 5e-2, BatchNorm running statistics 1e-2, discriminator-phase gradient norms 1e-1."""
    import json
    import os
    from oracle import studiogan_oracle as O
    from sgb200 import config as C
    from sgb200.models import deep_conv
    from sgb200.utils import losses
    from test_gpu_parity import l2_err
    dev = _cuda()
    g = np.load(os.path.join(golden_dir, "dcgan32.npz"))
    M = C.make_modules(False, False, "W/O", "deep_conv")
    MODEL = C._Section(info_type="N/A", g_info_injection="N/A")
    G = deep_conv.Generator(z_dim=16, g_shared_dim="N/A", img_size=32, g_conv_dim="N/A", apply_attn=False, attn_g_loc=[], g_cond_mtd="W/O",
                            num_classes=10, g_init="ortho", g_depth="N/A", mixed_precision=False, MODULES=M, MODEL=MODEL)
    D = deep_conv.Discriminator(img_size=32, d_conv_dim="N/A", apply_d_sn=False, apply_attn=False, attn_d_loc=[], d_cond_mtd="W/O",
                                aux_cls_type="W/O", d_embed_dim="N/A", normalize_d_embed=False, num_classes=10, d_init="ortho",
                                d_depth="N/A", mixed_precision=False, MODULES=M, MODEL=MODEL)
    G.load_state_dict(O.seeded_state(json.loads(str(g["keys_g"])), 101), strict=True)
    D.load_state_dict(O.seeded_state(json.loads(str(g["keys_d"])), 202), strict=True)
    G, D = G.to(dev).train(), D.to(dev).train()
    z, y, real = torch.from_numpy(g["z"]).to(dev), torch.from_numpy(g["y"]).to(dev), torch.from_numpy(g["real"]).to(dev)
    for p in G.parameters():
        p.requires_grad_(False)
    fake = G(z, y)
    assert l2_err(fake, torch.from_numpy(g["fake"])) < 4e-2
    rd, fd = D(real, y), D(fake.detach(), y)
    assert l2_err(rd["adv_output"], torch.from_numpy(g["adv_real"])) < 4e-2
    assert l2_err(fd["adv_output"], torch.from_numpy(g["adv_fake"])) < 4e-2
    d_loss = losses.d_vanilla(rd["adv_output"], fd["adv_output"])
    d_loss.backward()
    assert abs(float(d_loss) - float(g["d_loss"])) < 5e-2 * abs(float(g["d_loss"]))
    gmax = max(float(g[k]) for k in g.files if k.startswith("Dgnorm/"))
    for n, p in D.named_parameters():
        assert abs(float(p.grad.norm()) - float(g["Dgnorm/" + n])) < 1e-1 * float(g["Dgnorm/" + n]) + 2e-3 * gmax, n
    for n, b in list(G.named_buffers()) + list(D.named_buffers()):
        key = ("G1/" if any(b is bb for bb in G.buffers()) else "D1/") + n
        if "running_" in n:
            assert rel_err(b, torch.from_numpy(g[key])) < 1e-2, key
    D.zero_grad(set_to_none=True)
    for p in G.parameters():
        p.requires_grad_(True)
    for p in D.parameters():
        p.requires_grad_(False)
    fake2 = G(z, y)
    assert l2_err(fake2, torch.from_numpy(g["fake2"])) < 4e-2
    g_loss = losses.g_vanilla(D(fake2, y)["adv_output"])
    g_loss.backward()
    assert abs(float(g_loss) - float(g["g_loss"])) < 5e-2 * abs(float(g["g_loss"]))
    gmax = max(float(g[k]) for k in g.files if k.startswith("Ggnorm/"))
    for n, p in G.named_parameters():
        assert abs(float(p.grad.norm()) - float(g["Ggnorm/" + n])) < 0.3 * float(g["Ggnorm/" + n]) + 1e-2 * gmax, n


# ------------------------------------------------------------------------------------------------ augmentations
def test_diffaug_and_cr_kernels_match_reference_golden(golden_dir):
    """sgb_diffaug_fwd / bwd and sgb_cr_aug against the reference's DiffAugment / CR outputs and input gradients
    (tests/golden/augment.npz), with the parameters drawn by the product in the reference's RNG order on the host generator
    (the device path uses the same draw on the CUDA generator).  fp32 element-wise arithmetic: 1e-5."""
    import os
    from sgb200.utils import cr, diffaug
    dev = _cuda()
    g = np.load(os.path.join(golden_dir, "augment.npz"))
    for tag in ("a", "b"):
        x = torch.from_numpy(g["x_" + tag])
        ct = torch.from_numpy(g["ct_" + tag])
        B, _, H, W = x.shape
        for pname, policy in (("full", "color,translation,cutout"), ("color", "color"), ("geo", "translation,cutout")):
            torch.manual_seed(4242)
            params = diffaug.draw_params(B, H, W, policy, "cpu")
            xd = x.to(dev).requires_grad_(True)
            y = diffaug.apply_diffaug(xd, policy, params=params.to(dev))
            np.testing.assert_allclose(y.detach().cpu().numpy(), g["diffaug_%s_%s" % (pname, tag)], rtol=1e-5, atol=1e-5)
            y.backward(ct.to(dev))
            np.testing.assert_allclose(xd.grad.cpu().numpy(), g["diffaug_%s_%s_dx" % (pname, tag)], rtol=1e-5, atol=1e-5)
        torch.manual_seed(777)
        f, tx, ty = cr.draw_params(B, H, W, "cpu")
        y = cr.apply_cr_aug(x.to(dev), params=(f.to(dev), tx.to(dev), ty.to(dev)))
        np.testing.assert_array_equal(y.cpu().numpy(), g["cr_" + tag])
    # the device draw + kernel path end to end (statistical sanity: translation / cutout leave ~ the expected share of zeros)
    xd = torch.randn(64, 3, 32, 32, device=dev).abs() + 1.0
    y = diffaug.apply_diffaug(xd, "translation,cutout")
    zero_share = float((y == 0).float().mean())
    assert 0.15 < zero_share < 0.5, zero_share


def test_worker_step_with_diffaug_bcr_zcr_and_lecam():
    """WORKER.train_discriminator / train_generator with AUG.apply_diffaug (DiffAugment on every discriminator input,
    gradient through it in the generator phase), LOSS.apply_bcr + apply_zcr (consistency terms, src/worker.py:339-366,603-605)
    and LOSS.apply_lecam (:394-407) on a small BigGAN-Deep: the step runs on the CUDA path, the discriminator loss contains
    the extra terms (it differs from the plain hinge loss of the same logits), the LeCam EMAs move, parameters move, nothing
    is NaN."""
    from sgb200 import config as C
    from sgb200.models import model as M
    from sgb200.worker import WORKER
    dev = _cuda()
    cfgs = C.Configurations(None)
    cfgs.DATA.img_size, cfgs.DATA.num_classes = 32, 10
    m = cfgs.MODEL
    m.backbone, m.g_cond_mtd, m.d_cond_mtd, m.apply_g_sn, m.apply_d_sn = "big_resnet_deep_legacy", "cBN", "PD", True, True
    m.z_dim, m.g_shared_dim, m.g_conv_dim, m.d_conv_dim, m.g_depth, m.d_depth = 32, 32, 16, 16, 1, 1
    m.apply_g_ema = False
    L_ = cfgs.LOSS
    L_.adv_loss = "hinge"
    L_.apply_bcr, L_.real_lambda, L_.fake_lambda = True, 10.0, 10.0
    L_.apply_zcr, L_.radius, L_.g_lambda, L_.d_lambda = True, 0.05, 0.5, 5.0
    L_.apply_lecam, L_.lecam_lambda, L_.lecam_ema_start_iter, L_.lecam_ema_decay = True, 0.3, 2, 0.9
    cfgs.AUG.apply_diffaug, cfgs.AUG.diffaug_type, cfgs.AUG.bcr_aug_type = True, "diffaug", "bcr"
    o = cfgs.OPTIMIZATION
    o.batch_size, o.d_updates_per_step, o.g_updates_per_step, o.acml_steps = 16, 2, 1, 1
    cfgs.define_modules()
    cfgs.define_losses()
    cfgs.define_augments()
    torch.manual_seed(0)
    Gen, _, _, Dis, Gen_ema, _, _, ema = M.load_generator_discriminator(cfgs.DATA, o, cfgs.MODEL, cfgs.STYLEGAN, cfgs.MODULES,
                                                                        cfgs.RUN, dev, None)
    cfgs.define_optimizer(Gen, Dis)

    class Loader:
        def __iter__(self):
            return self

        def __next__(self):
            g = torch.Generator().manual_seed(1)
            return torch.rand(32, 3, 32, 32, generator=g) * 2 - 1, torch.randint(0, 10, (32,), generator=g)
    w = WORKER(cfgs=cfgs, run_name="t", Gen=Gen, Gen_mapping=None, Gen_synthesis=None, Dis=Dis, Gen_ema=Gen_ema, Gen_ema_mapping=None,
               Gen_ema_synthesis=None, ema=ema, eval_model=None, train_dataloader=Loader(), eval_dataloader=None, global_rank=0,
               local_rank=dev, mu=None, sigma=None, real_feats=None, logger=None)
    assert w.lecam_ema.D_real == 7777
    d0 = [p.detach().clone() for p in Dis.parameters()]
    g0 = [p.detach().clone() for p in Gen.parameters()]
    for step in range(1, 4):             # step 1: EMA = current (before start_iter); step 2: decayed; step 3: regulariser active
        _, d_loss = w.train_discriminator(step)
        g_loss = w.train_generator(step)
        assert torch.isfinite(d_loss).all() and torch.isfinite(g_loss).all()
    assert w.lecam_ema.D_real != 7777 and abs(w.lecam_ema.D_real) < 1e3          # the EMA has been fed with mean logits
    assert all(torch.isfinite(p).all() for p in list(Dis.parameters()) + list(Gen.parameters()))
    assert any(float((p.detach() - q).abs().max()) > 0 for p, q in zip(Dis.parameters(), d0))
    assert any(float((p.detach() - q).abs().max()) > 0 for p, q in zip(Gen.parameters(), g0))


# (B, H, W, Cin, Cout, k): epilogue paths that write / read ReLU bit planes
BIT_SHAPES = [
    (2, 64, 64, 128, 64, 1),      # generic kernel, TMA-store epilogue, one 64-channel chunk
    (2, 32, 32, 64, 256, 1),      # ... four chunks, two teams
    (1, 256, 256, 64, 64, 3),     # halo-row kernel: staging-tile row + direct-store row
    (1, 128, 128, 128, 128, 3),   # halo-row kernel, two chunks
    (2, 16, 16, 256, 256, 3),     # generic kernel, direct-store epilogue (K > TMA-store limit)
    (3, 20, 20, 64, 128, 1),      # ragged pixel tiles (clipped rows)
]


@pytest.mark.parametrize("B,H,W,Cin,Cout,k", BIT_SHAPES)
def test_relu_bit_planes_written_and_consumed(B, H, W, Cin, Cout, k):
    """A relu epilogue's bit planes equal (y > 0) packed little-endian per 64-channel word, and an input-gradient launch
    masked by those bits equals the launch masked by the bf16 tensor, bit for bit."""
    from sgb200 import kernels as K
    dev = _cuda()
    g = torch.Generator().manual_seed(Cin * 7 + Cout + k)
    x = to_nhwc(bfr(torch.randn(B, Cin, H, W, generator=g)), dev)
    w = (torch.randn(Cout, Cin, k, k, generator=g) / np.sqrt(Cin * k * k)).to(dev)
    b = torch.randn(Cout, generator=g).to(dev)
    wf, wd = K.weight_pack(w, None, Cout, Cin, k * k, True, True)
    y = K.conv_fprop(x, wf, Cout, k, k, k // 2, k // 2, bias=b, relu=True, want_relu_bits=True)
    y_plain = K.conv_fprop(x, wf, Cout, k, k, k // 2, k // 2, bias=b, relu=True)
    bits = y._sgb_relu_bits
    assert torch.equal(y, y_plain)
    pos = (y.permute(0, 2, 3, 1).float() > 0).cpu().numpy()                       # [B, H, W, C]
    expect = np.packbits(pos, axis=-1, bitorder="little")
    got = bits.cpu().numpy()
    # a positive accumulator below the smallest bf16 rounds to zero in y but keeps its bit: allow only that direction
    diff = np.unpackbits(got ^ expect, axis=-1, bitorder="little").astype(bool)
    assert diff.mean() < 1e-6 and not (diff & pos).any()
    # consumer: dgrad of a layer whose INPUT was y (mask has Cout_of_dgrad = Cout channels)
    dz = to_nhwc(bfr(torch.randn(B, Cin, H, W, generator=g)), dev)
    wt = (torch.randn(Cin, Cout, k, k, generator=g) / np.sqrt(Cout * k * k)).to(dev)   # next layer: Cout -> Cin
    _, wtd = K.weight_pack(wt, None, Cin, Cout, k * k, True, True)
    dx_ref = K.conv_fprop(dz, wtd, Cout, k, k, k - 1 - k // 2, k - 1 - k // 2, mask=y)
    dx_bits = K.conv_fprop(dz, wtd, Cout, k, k, k - 1 - k // 2, k - 1 - k // 2, mask_bits=bits)
    if diff.any():
        keep = torch.from_numpy(~diff).to(dev).permute(0, 3, 1, 2)
        assert torch.equal(dx_ref * keep, dx_bits * keep)
    else:
        assert torch.equal(dx_ref, dx_bits)
    # with a half-resolution residual on top (fused discriminator block entry)
    if H % 2 == 0 and k == 1:
        r = to_nhwc(bfr(torch.randn(B, Cout, H // 2, W // 2, generator=g)), dev)
        a = K.conv_fprop(dz, wtd, Cout, 1, 1, 0, 0, mask=y, residual=r, res_up2=True, res_scale=0.25)
        c = K.conv_fprop(dz, wtd, Cout, 1, 1, 0, 0, mask_bits=bits, residual=r, res_up2=True, res_scale=0.25)
        assert diff.any() or torch.equal(a, c)


def test_pool2_bwd_with_bit_planes_and_d_block_uses_them():
    from sgb200 import kernels as K
    dev = _cuda()
    g = torch.Generator().manual_seed(3)
    B, C, H, W = 2, 128, 32, 32
    x = to_nhwc(bfr(torch.randn(B, 64, H, W, generator=g)), dev)
    w = (torch.randn(C, 64, 1, 1, generator=g) / 8).to(dev)
    wf, _ = K.weight_pack(w, None, C, 64, 1, True, False)
    y = K.conv_fprop(x, wf, C, 1, 1, 0, 0, relu=True, want_relu_bits=True)
    dy = to_nhwc(bfr(torch.randn(B, C, H // 2, W // 2, generator=g)), dev)
    assert torch.equal(K.pool2_bwd(dy, 0, relu_src=y), K.pool2_bwd(dy, 0, relu_bits=y._sgb_relu_bits))
    # the discriminator block hands bit planes from producer to consumer (no silent fallback to the bf16 masks)
    import importlib
    from sgb200 import config as Cfg
    deep = importlib.import_module("sgb200.models.big_resnet_deep_legacy")
    M = Cfg.make_modules(True, True, "cBN", "big_resnet_deep_legacy")
    MODEL = Cfg._Section(info_type="N/A", g_info_injection="N/A")
    torch.manual_seed(0)
    D = deep.Discriminator(img_size=32, d_conv_dim=64, apply_d_sn=True, apply_attn=False, attn_d_loc=[1], d_cond_mtd="PD",
                           aux_cls_type="W/O", d_embed_dim="N/A", normalize_d_embed=False, num_classes=5, d_init="ortho",
                           d_depth=1, mixed_precision=False, MODULES=M, MODEL=MODEL).to(dev).train()
    img = (torch.rand(4, 3, 32, 32, generator=g) * 2 - 1).to(dev).requires_grad_(True)
    lab = torch.randint(0, 5, (4,), generator=g).to(dev)
    K.BITS_STATS.update(written=0, used=0)
    D(img, lab)["adv_output"].sum().backward()
    assert K.BITS_STATS["written"] > 0 and K.BITS_STATS["used"] >= K.BITS_STATS["written"] - 1, K.BITS_STATS   # (the head reads the last tensor itself)


@pytest.mark.parametrize("B,S,c8,c2", [(2, 64, 64, 256), (3, 16, 48, 192), (1, 32, 16, 64)])
def test_attention_softmax_inside_the_gemm_epilogues(B, S, c8, c2):
    """P = softmax(theta . phi^T) written by the score GEMM's second pass (statistics pass + apply pass) and
    dS = P * (do . g^T - rowsum(do * o)) written by the dP GEMM, against fp32 torch on the same bf16 operands
    (src/utils/ops.py:93-97 and its autograd)."""
    from sgb200 import kernels as K
    dev = _cuda()
    g_ = torch.Generator().manual_seed(S + c8)
    N, M = S * S, (S // 2) * (S // 2)
    theta = bfr(torch.randn(B, c8, S, S, generator=g_) * 0.7)
    phi = bfr(torch.randn(B, c8, S // 2, S // 2, generator=g_) * 0.7)
    gv = bfr(torch.randn(B, c2, S // 2, S // 2, generator=g_))
    do = bfr(torch.randn(B, c2, S, S, generator=g_))
    th, ph, gd, dod = (to_nhwc(t, dev) for t in (theta, phi, gv, do))
    P, stats = K.conv_fprop(th, ph, M, 1, 1, 0, 0, w_mode=1, sm_mode=1)
    K.conv_fprop(th, ph, M, 1, 1, 0, 0, w_mode=1, sm_mode=2, sm_stats=stats, out=P)
    q = theta.reshape(B, c8, N).transpose(1, 2)                      # [B, N, c8]
    k = phi.reshape(B, c8, M)                                        # [B, c8, M]
    Pr = torch.softmax(torch.bmm(q, k), -1)                          # [B, N, M]
    Pg = P.permute(0, 2, 3, 1).reshape(B, N, M).float().cpu()
    assert float((Pg - Pr).abs().max()) < 8e-3 * float(Pr.max()) + 1e-6
    assert float((Pg.sum(-1) - 1).abs().max()) < 2e-2
    # same result as the two-kernel path (score GEMM rounded to bf16, then the row-softmax kernel) up to that rounding
    S2 = K.conv_fprop(th, ph, M, 1, 1, 0, 0, w_mode=1)
    K.softmax_rows(S2, M, out=S2)
    assert rel_err(P, S2.float().cpu()) < 2e-2
    # backward
    o = K.conv_fprop(P, gd, c2, 1, 1, 0, 0, w_mode=2)
    dS = K.conv_fprop(dod, gd, M, 1, 1, 0, 0, w_mode=1, sm_mode=3, sm_delta=K.rowdot(dod, o), sm_p=P)
    v = gv.reshape(B, c2, M)                                          # [B, c2, M]
    dP = torch.bmm(do.reshape(B, c2, N).transpose(1, 2), v)          # [B, N, M]
    Pb = Pg                                                          # the bf16 P the kernels used
    dSr = Pb * (dP - (Pb * dP).sum(-1, keepdim=True))
    dSg = dS.permute(0, 2, 3, 1).reshape(B, N, M).float().cpu()
    assert float((dSg - dSr).norm() / dSr.norm()) < 1.5e-2


@pytest.mark.parametrize("mtd,sn", [("PD", True), ("W/O", True), ("PD", False)])
def test_discriminator_head_kernels_match_the_eager_head(mtd, sn):
    """sgb_dhead_fwd / sgb_dhead_bwd (+ the spectral-norm chain rule) against the same head written as tensor arithmetic
    (src/models/big_resnet_deep_legacy.py:346-349,366-368): logits, feature gradient and parameter gradients."""
    import copy
    import importlib
    from sgb200 import config as Cfg
    from sgb200.utils import ops
    dev = _cuda()
    deep = importlib.import_module("sgb200.models.big_resnet_deep_legacy")
    M = Cfg.make_modules(True, sn, "cBN", "big_resnet_deep_legacy")
    MODEL = Cfg._Section(info_type="N/A", g_info_injection="N/A")
    torch.manual_seed(3)
    D1 = deep.Discriminator(img_size=32, d_conv_dim=16, apply_d_sn=sn, apply_attn=False, attn_d_loc=[1], d_cond_mtd=mtd,
                            aux_cls_type="W/O", d_embed_dim="N/A", normalize_d_embed=False, num_classes=7, d_init="ortho",
                            d_depth=1, mixed_precision=False, MODULES=M, MODEL=MODEL).to(dev).train()
    D2 = copy.deepcopy(D1)
    for m in D2.modules():
        if hasattr(m, "_sn"):
            m._sn.module, m._sn.ws = m, None
    g = torch.Generator().manual_seed(1)
    C = D1.linear1.in_features
    h0 = (torch.rand(6, C, generator=g) * 3).to(dev)
    lab = torch.randint(0, 7, (6,), generator=g).to(dev)
    res = []
    for D, fused in ((D1, True), (D2, False)):
        ops.DHEAD_FUSED = fused
        try:
            h = h0.clone().requires_grad_(True)
            adv = ops.discriminator_head(D, h, lab)["adv_output"]
            (adv * torch.arange(1, 7, device=dev).float()).sum().backward()
        finally:
            ops.DHEAD_FUSED = True
        pg = {n: p.grad.clone() for n, p in D.named_parameters() if p.grad is not None}
        res.append((adv.detach(), h.grad.clone(), pg))
    (a1, dh1, g1), (a2, dh2, g2) = res
    assert rel_err(a1, a2.cpu()) < 1e-5 and rel_err(dh1, dh2.cpu()) < 1e-5
    assert set(g1) == set(g2) and len(g1) >= (3 if mtd == "PD" else 2)
    for n in g1:
        assert rel_err(g1[n], g2[n].cpu()) < 1e-4, n
    if sn:   # both heads ran one power iteration from the same state
        assert rel_err(D1.linear1.weight_u, D2.linear1.weight_u.cpu()) < 1e-6


def test_batched_cbn_affine_gemm_matches_per_layer_linears():
    """Gradient-free generator passes compute every cBN gain(y) / bias(y) with one GEMM over the contiguous packs
    (snbatch.cbn_affine_all); the image must equal the per-layer path (grad-enabled pass of an identical copy)."""
    import copy
    import importlib
    from sgb200 import config as Cfg
    from sgb200 import kernels as K
    dev = _cuda()
    deep = importlib.import_module("sgb200.models.big_resnet_deep_legacy")
    M = Cfg.make_modules(True, True, "cBN", "big_resnet_deep_legacy")
    MODEL = Cfg._Section(info_type="N/A", g_info_injection="N/A")
    torch.manual_seed(11)
    G1 = deep.Generator(z_dim=24, g_shared_dim=16, img_size=32, g_conv_dim=16, apply_attn=False, attn_g_loc=[2], g_cond_mtd="cBN",
                        num_classes=9, g_init="ortho", g_depth=2, mixed_precision=False, MODULES=M, MODEL=MODEL).to(dev).train()
    G2 = copy.deepcopy(G1)
    for net in (G2,):
        for m in net.modules():
            if hasattr(m, "_sn"):
                m._sn.module, m._sn.ws = m, None
        net._snb.net, net._snb.mods = net, None
    g = torch.Generator().manual_seed(2)
    z = torch.randn(5, 24, generator=g).to(dev)
    y = torch.randint(0, 9, (5,), generator=g).to(dev)
    calls = []
    orig = K.conv_fprop
    K.conv_fprop = lambda *a, **k: (calls.append(a[2]), orig(*a, **k))[1]
    try:
        with torch.no_grad():
            img1 = G1(z, y)
        n1 = len(calls)
        calls.clear()
        img2 = G2(z, y)
        n2 = len(calls)
    finally:
        K.conv_fprop = orig
    assert G1._snb.cbn is not None and n1 < n2 - 10, (n1, n2)            # dozens of tiny GEMMs became one
    # images: a 12-block generator with batch statistics over 5 samples amplifies the fp32 summation-order differences of the two
    # GEMM tilings (and of the atomics in the statistics kernels) to the 1e-2 level -- a sanity bound only; the maps themselves
    # are compared exactly below
    assert rel_err(img1, img2.detach().float().cpu()) < 5e-2
    for (n, b1), (_, b2) in zip(G1.named_buffers(), G2.named_buffers()):
        if n.endswith("weight_u"):
            assert rel_err(b1, b2.cpu()) < 1e-4, n
    # every gain(y) / bias(y) column slice of the batched GEMM against the layer's own GEMM
    from sgb200 import autograd_ops as A
    from sgb200.utils import ops
    with torch.no_grad():
        G1._snb.run()
        yv = A.ToBF16Fn.call(torch.cat([G1.shared(y), z], 1))
        assert G1._snb.cbn_affine_all(yv)
        checked = 0
        for m in G1.modules():
            if isinstance(m, ops.ConditionalBatchNorm2d):
                for lin in (m.gain, m.bias):
                    ref = lin(yv, out_fp32=True).reshape(z.shape[0], -1)
                    assert lin._pre_out.shape == ref.shape and rel_err(lin._pre_out, ref.float().cpu()) < 1e-5
                    checked += 1
        G1._snb.clear()
    assert checked >= 16
