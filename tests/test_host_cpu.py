"""CPU-side checks of the host layer: C-ABI surface, ctypes signatures, module/state_dict compatibility and seeded
initialisation parity with the reference (golden G0/D0 tensors come from the real StudioGAN modules)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from sgb200 import _lib as L
from sgb200 import config as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "sgb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    decls = {}
    for m in re.finditer(r"\b(int|int64_t)\s+(sgb_\w+)\s*\(([^;{]*)\)\s*;", src):
        args = m.group(3).strip()
        n = 0 if args in ("", "void") else len(args.split(","))
        decls[m.group(2)] = n
    return decls


def test_header_and_ctypes_table_agree():
    decls = _declared()
    assert len(decls) >= 28
    assert set(decls) == set(L.SIGNATURES), set(decls) ^ set(L.SIGNATURES)
    for name, n in decls.items():
        assert len(L.SIGNATURES[name][1]) == n, name


def test_library_exports_every_declared_symbol():
    if not os.path.exists(L.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(L.LIB_PATH)
    for name in _declared():
        assert hasattr(lib, name), name
    assert lib.sgb_abi_version() == 1          # pure host call, no GPU needed


def test_struct_layout_matches_header():
    # field order / count of the two descriptor structs (a mismatch would silently corrupt kernel arguments)
    src = open(os.path.join(ROOT, "include", "sgb200.h")).read()
    for sname, cls in (("sgb_conv_desc", L.ConvDesc), ("sgb_wgrad_desc", L.WgradDesc)):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (sname, sname), src, flags=re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        names = []
        for stmt in body.split(";"):
            stmt = stmt.strip()
            if not stmt:
                continue
            for part in stmt.split(","):
                names.append(re.findall(r"(\w+)\s*$", part.strip())[0])
        assert names == [f[0] for f in cls._fields_], (sname, names)


def _build(tag_cfg):
    import importlib
    deep = importlib.import_module("sgb200.models." + tag_cfg.get("backbone", "big_resnet_deep_legacy"))
    M = C.make_modules(True, True, "cBN", tag_cfg.get("backbone", "big_resnet_deep_legacy"))
    MODEL = C._Section(info_type="N/A", g_info_injection="N/A")
    torch.manual_seed(1234)
    G = deep.Generator(z_dim=16, g_shared_dim=16, img_size=32, g_conv_dim=tag_cfg["conv_dim"], apply_attn=tag_cfg["attn"],
                       attn_g_loc=[2], g_cond_mtd="cBN", num_classes=5, g_init="ortho", g_depth=tag_cfg["depth"],
                       mixed_precision=False, MODULES=M, MODEL=MODEL)
    D = deep.Discriminator(img_size=32, d_conv_dim=tag_cfg["conv_dim"], apply_d_sn=True, apply_attn=tag_cfg["attn"],
                           attn_d_loc=[1], d_cond_mtd="PD", aux_cls_type="W/O", d_embed_dim="N/A", normalize_d_embed=False,
                           num_classes=5, d_init="ortho", d_depth=tag_cfg["depth"], mixed_precision=False, MODULES=M, MODEL=MODEL)
    return G, D


@pytest.mark.parametrize("tag,cfg", [("deep32_c8", dict(conv_dim=8, depth=1, attn=False)),
                                     ("deep32_c16_attn_d2", dict(conv_dim=16, depth=2, attn=True)),
                                     ("deepsg32_c8", dict(conv_dim=8, depth=1, attn=False, backbone="big_resnet_deep_studiogan"))])
def test_state_dict_keys_and_seeded_init_match_reference(golden_dir, tag, cfg):
    g = np.load(os.path.join(golden_dir, tag + ".npz"))
    G, D = _build(cfg)
    for net, prefix in ((G, "G0/"), (D, "D0/")):
        sd = net.state_dict()
        ref_keys = [k[len(prefix):] for k in g.files if k.startswith(prefix)]
        assert list(sd.keys()) == ref_keys                     # same keys in the same registration order
        for k in ref_keys:
            ref = g[prefix + k]
            assert tuple(sd[k].shape) == tuple(ref.shape), k
            if k.endswith("sigma"):
                continue                                        # the golden script overwrote the attention gate
            np.testing.assert_array_equal(sd[k].numpy(), ref, err_msg=k)   # identical RNG consumption -> bit-identical init


def test_reference_checkpoint_loads_strictly(golden_dir):
    g = np.load(os.path.join(golden_dir, "deep32_c16_attn_d2.npz"))
    G, D = _build(dict(conv_dim=16, depth=2, attn=True))
    for net, prefix in ((G, "G1/"), (D, "D1/")):
        sd = {k[3:]: torch.from_numpy(g[k].copy()) for k in g.files if k.startswith(prefix[0] + "0/")}
        sd.update({k[len(prefix):]: torch.from_numpy(g[k].copy()) for k in g.files if k.startswith(prefix)})
        net.load_state_dict(sd, strict=True)


def test_yaml_configs_drop_in(golden_dir):
    # unmodified copies of the reference's src/configs files
    ref_cfgs = os.path.join(golden_dir, "reference_configs")
    for rel in ["ImageNet/BigGAN-Deep-256.yaml", "CIFAR10/BigGAN.yaml", "CIFAR10/SNGAN.yaml", "CIFAR10/WGAN-GP.yaml",
                "CIFAR10/BigGAN-Deep.yaml"]:
        cfg = C.Configurations(os.path.join(ref_cfgs, rel))
        assert callable(cfg.MODULES.g_conv2d) and callable(cfg.LOSS.d_loss)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(L, "_lib", None)
    monkeypatch.setattr(L, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU / PyTorch fallback"):
        L.load()


def test_bn_tangent_formulas_and_reverse_over_forward_identity():
    """(1) The oracle's closed forms for the tangent of a training-mode batch norm and its (x, a, gamma) derivatives (what the
    sgb_bn_tangent_* kernels compute) equal torch autograd's JVP / double backward in fp64.
    (2) dP/dtheta of the gradient penalty obtained by reverse-over-forward (utils/gp.py) equals the reference's
    double-backward formulation (src/utils/losses.py:268-316) on a conv -> BN -> ReLU -> conv -> sum -> linear discriminator."""
    import torch.nn.functional as F
    from oracle import studiogan_oracle as O
    torch.manual_seed(0)
    dd = torch.float64
    x = torch.randn(4, 3, 5, 5, dtype=dd, requires_grad=True)
    a = torch.randn(4, 3, 5, 5, dtype=dd, requires_grad=True)
    c = torch.randn(4, 3, 5, 5, dtype=dd)
    gamma = (torch.rand(3, dtype=dd) + 0.5).requires_grad_(True)
    beta = torch.zeros(3, dtype=dd)
    eps = 1e-4
    bn = lambda t: F.batch_norm(t, None, None, gamma, beta, True, 0.1, eps)                      # noqa: E731
    _, jvp = torch.autograd.functional.jvp(bn, x, a)
    t = O.bn_tangent(x, a, gamma, eps)
    assert float((t - jvp).abs().max()) < 1e-10                                                 # closed form == torch's JVP
    gx, ga, gg = torch.autograd.grad((t * c).sum(), (x, a, gamma))                              # autograd through the closed form
    dx, da, dgamma = O.bn_tangent_backward(x.detach(), a.detach(), c, gamma.detach(), eps)
    assert float((dx - gx).abs().max()) < 1e-9 and float((da - ga).abs().max()) < 1e-9 and float((dgamma - gg).abs().max()) < 1e-9

    w1 = (torch.randn(6, 3, 3, 3, dtype=dd) * 0.3).requires_grad_(True)
    w2 = (torch.randn(4, 6, 3, 3, dtype=dd) * 0.3).requires_grad_(True)
    g1 = (torch.rand(6, dtype=dd) + 0.5).requires_grad_(True)
    b1 = torch.zeros(6, dtype=dd, requires_grad=True)
    wl = torch.randn(1, 4, dtype=dd, requires_grad=True)
    params = (w1, w2, g1, wl)

    def disc(img):
        h = F.conv2d(img, w1, padding=1)
        h = F.relu(F.batch_norm(h, None, None, g1, b1, True, 0.1, eps))
        h = F.conv2d(h, w2, padding=1)
        return F.linear(F.relu(h).sum((2, 3)), wl).squeeze(1)

    real, fake = torch.randn(4, 3, 6, 6, dtype=dd), torch.randn(4, 3, 6, 6, dtype=dd)
    alpha = torch.rand(4, 1, dtype=dd)
    gp = O.grad_penalty(disc, real, fake, alpha)
    ref = torch.autograd.grad(gp, params)
    # reverse over forward, exactly as utils/gp.py: g (no graph) -> seed v -> tangent pass -> backward
    a4 = alpha.view(4, 1, 1, 1)
    x_hat = (a4 * real + (1 - a4) * fake).requires_grad_(True)
    (g,) = torch.autograd.grad(disc(x_hat).sum(), x_hat)
    n = g.flatten(1).norm(dim=1)
    assert abs(float(((n - 1) ** 2).mean()) - float(gp)) < 1e-10
    v = (2 * (n - 1) / (4 * n)).view(4, 1, 1, 1) * g
    h = F.conv2d(x_hat, w1, padding=1)
    th = F.conv2d(v, w1, padding=1)
    y = F.relu(F.batch_norm(h, None, None, g1, b1, True, 0.1, eps))
    ty = O.bn_tangent(h, th, g1, eps) * (y > 0)
    h2, th2 = F.conv2d(y, w2, padding=1), F.conv2d(ty, w2, padding=1)
    t_adv = F.linear((th2 * (h2 > 0)).sum((2, 3)), wl).squeeze(1)
    got = torch.autograd.grad(t_adv.sum(), params)
    for r_, g_ in zip(ref, got):
        assert float((r_ - g_).abs().max()) < 1e-8 * (1 + float(r_.abs().max()))


def test_standing_statistics_choreography():
    """apply_standing_statistics (src/utils/misc.py:301-333): statistics reset, `standing_step` train-mode passes with
    batch sizes in [1, standing_max_batch], generator left in eval mode."""
    import torch.nn as nn
    from sgb200.utils import misc

    class G(nn.Module):
        def __init__(self):
            super().__init__()
            self.bn = nn.BatchNorm2d(4)
            self.sizes = []

        def forward(self, z, label, eval=False):
            assert self.training and not eval and not torch.is_grad_enabled()
            self.sizes.append(z.shape[0])
            return self.bn(torch.randn(z.shape[0], 4, 2, 2) + 3.0)
    g = G()
    g.bn.running_mean.fill_(7.0)
    cfgs = C.Configurations(None)
    cfgs.RUN.distributed_data_parallel = False
    misc.apply_standing_statistics(g, standing_max_batch=6, standing_step=5, DATA=cfgs.DATA, MODEL=cfgs.MODEL, LOSS=cfgs.LOSS,
                                   OPTIMIZATION=cfgs.OPTIMIZATION, RUN=cfgs.RUN, device="cpu")
    assert len(g.sizes) == 5 and all(1 <= s <= 6 for s in g.sizes)
    assert not g.training and int(g.bn.num_batches_tracked) == 5
    assert 0.5 < float(g.bn.running_mean.mean()) < 3.5            # reset to 0, then moved towards the batch mean 3


def test_conditioning_losses_match_reference(golden_dir):
    """AC / 2C / D2D-CE losses (src/utils/losses.py:38-165): values and input gradients vs the reference's own classes."""
    from sgb200.utils import losses
    g = np.load(os.path.join(golden_dir, "cond_losses.npz"))
    label = torch.from_numpy(g["label"])
    logits = torch.from_numpy(g["logits"]).requires_grad_(True)
    ce = losses.CrossEntropyLoss()(cls_output=logits, label=label)
    ce.backward()
    np.testing.assert_allclose(ce.item(), g["ce"], rtol=1e-6)
    np.testing.assert_allclose(logits.grad.numpy(), g["ce_dlogits"], rtol=1e-5, atol=1e-7)
    for name, mod in (("c2", losses.ConditionalContrastiveLoss(num_classes=4, temperature=0.5)),
                      ("d2dce", losses.Data2DataCrossEntropyLoss(num_classes=4, temperature=0.5, m_p=0.98))):
        embed = torch.from_numpy(g[name + "_embed"]).requires_grad_(True)
        proxy = torch.from_numpy(g[name + "_proxy"]).requires_grad_(True)
        loss = mod(embed=embed, proxy=proxy, label=label, h=None, adv_output=None)     # extra head keys are ignored (**_)
        loss.backward()
        np.testing.assert_allclose(loss.item(), g[name], rtol=1e-5)
        np.testing.assert_allclose(embed.grad.numpy(), g[name + "_dembed"], rtol=1e-4, atol=1e-7)
        np.testing.assert_allclose(proxy.grad.numpy(), g[name + "_dproxy"], rtol=1e-4, atol=1e-7)


def test_checkpoint_round_trip_in_reference_format(tmp_path, golden_dir):
    """utils/ckpt.py writes the reference's file names / dict keys (src/worker.py:940-985, src/utils/ckpt.py:28-141) and
    reads them back strictly; the previous file of the same (model, when) is replaced."""
    import types
    from sgb200.utils import ckpt
    G, D = _build(dict(conv_dim=8, depth=1, attn=False))
    G2, D2 = _build(dict(conv_dim=8, depth=1, attn=False))
    with torch.no_grad():
        for p in list(G2.parameters()) + list(D2.parameters()):
            p.add_(1.0)
    g_opt = torch.optim.Adam(G.parameters(), lr=2e-4, betas=(0.0, 0.999), eps=1e-6)
    d_opt = torch.optim.Adam(D.parameters(), lr=2e-4, betas=(0.0, 0.999), eps=1e-6)
    for p in D.parameters():
        p.grad = torch.ones_like(p)
    d_opt.step()
    w = types.SimpleNamespace(Gen=G, Dis=D, Gen_ema=G2, run_name="unit", best_step=3, best_fid=12.5,
                              OPTIMIZATION=types.SimpleNamespace(g_optimizer=g_opt, d_optimizer=d_opt),
                              RUN=types.SimpleNamespace(seed=7, ckpt_dir=str(tmp_path)))
    ckpt.save(w, step=10, is_best=False)
    paths = ckpt.save(w, step=20, is_best=False)
    names = sorted(os.listdir(tmp_path))
    assert names == ["model=D-current-weights-step=20.pth", "model=G-current-weights-step=20.pth",
                     "model=G_ema-current-weights-step=20.pth"] and len(paths) == 3
    d_file = torch.load(os.path.join(tmp_path, names[0]), weights_only=False)
    assert set(d_file) == {"state_dict", "optimizer", "seed", "run_name", "step", "epoch", "topk", "aa_p", "best_step", "best_fid",
                           "best_fid_ckpt", "lecam_emas"}
    G3, D3 = _build(dict(conv_dim=8, depth=1, attn=False))
    G4, _ = _build(dict(conv_dim=8, depth=1, attn=False))
    d_opt3 = torch.optim.Adam(D3.parameters(), lr=1.0)
    g_opt3 = torch.optim.Adam(G3.parameters(), lr=1.0)
    ema = types.SimpleNamespace(source=None, target=None)
    misc_ = ckpt.load_StudioGAN_ckpts(str(tmp_path), False, G3, D3, g_opt3, d_opt3, True, G4, ema)
    assert misc_[:3] == (7, "unit", 20) and misc_[6:8] == (3, 12.5) and ema.source is G3 and ema.target is G4
    for a, b in zip(D.state_dict().values(), D3.state_dict().values()):
        assert torch.equal(a, b)
    for a, b in zip(G2.state_dict().values(), G4.state_dict().values()):
        assert torch.equal(a, b)
    assert d_opt3.state_dict()["param_groups"][0]["lr"] == 2e-4 and len(d_opt3.state_dict()["state"]) == len(list(D3.parameters()))


def test_sampler_rng_order_matches_reference_bit_for_bit(golden_dir):
    """sample_zy (src/utils/sample.py:69-90): labels first, then z, on the same generator -- every branch reproduces the
    reference's draws exactly (tests/golden/sampler.npz, from the unmodified reference)."""
    import numpy as np
    from sgb200.utils import sample
    g = np.load(os.path.join(golden_dir, "sampler.npz"))
    for name, kw in (("gauss", dict(z_prior="gaussian", truncation_factor=-1.0, y_sampler="totally_random", radius="N/A")),
                     ("uniform", dict(z_prior="uniform", truncation_factor=-1.0, y_sampler="totally_random", radius="N/A")),
                     ("eps", dict(z_prior="gaussian", truncation_factor=-1.0, y_sampler="totally_random", radius=0.5)),
                     ("trunc", dict(z_prior="gaussian", truncation_factor=0.7, y_sampler="totally_random", radius="N/A")),
                     ("some", dict(z_prior="gaussian", truncation_factor=-1.0, y_sampler="acending_some", radius="N/A")),
                     ("all", dict(z_prior="gaussian", truncation_factor=-1.0, y_sampler="acending_all", radius="N/A")),
                     ("fixed", dict(z_prior="gaussian", truncation_factor=-1.0, y_sampler=3, radius="N/A"))):
        torch.manual_seed(2718)
        np.random.seed(31)
        zs, y, zs_eps = sample.sample_zy(batch_size=16, z_dim=12, num_classes=7, device="cpu", **kw)
        assert np.array_equal(y.numpy(), g[name + "_y"]), name            # integer path: bit exact
        assert np.array_equal(zs.numpy(), g[name + "_z"]), name           # same generator, same order: bit exact
        if name + "_zeps" in g.files:
            assert np.array_equal(zs_eps.numpy(), g[name + "_zeps"]), name


def test_dcgan_state_dict_keys_match_reference(golden_dir):
    """models.deep_conv (BASELINE config 1): state_dict keys and shapes of generator / discriminator equal the reference's
    (recorded in tests/golden/dcgan32.npz by the generator script), so reference DCGAN checkpoints load strictly."""
    import json
    import numpy as np
    from sgb200 import config as C
    from sgb200.models import deep_conv
    g = np.load(os.path.join(golden_dir, "dcgan32.npz"))
    M = C.make_modules(False, False, "W/O", "deep_conv")
    MODEL = C._Section(info_type="N/A", g_info_injection="N/A")
    G = deep_conv.Generator(z_dim=16, g_shared_dim="N/A", img_size=32, g_conv_dim="N/A", apply_attn=False, attn_g_loc=[], g_cond_mtd="W/O",
                            num_classes=10, g_init="ortho", g_depth="N/A", mixed_precision=False, MODULES=M, MODEL=MODEL)
    D = deep_conv.Discriminator(img_size=32, d_conv_dim="N/A", apply_d_sn=False, apply_attn=False, attn_d_loc=[], d_cond_mtd="W/O",
                                aux_cls_type="W/O", d_embed_dim="N/A", normalize_d_embed=False, num_classes=10, d_init="ortho",
                                d_depth="N/A", mixed_precision=False, MODULES=M, MODEL=MODEL)
    assert [[k, list(v.shape)] for k, v in G.state_dict().items()] == json.loads(str(g["keys_g"]))
    assert [[k, list(v.shape)] for k, v in D.state_dict().items()] == json.loads(str(g["keys_d"]))


def test_uint8_dataset_matches_reference_transform_chain(tmp_path):
    """data_util.Dataset_ (src/data_util.py:59-142): an .npz / HDF5-style uint8 NHWC store; ``__getitem__`` equals the
    reference's ToTensor + Normalize(0.5, 0.5) chain bit for bit, the batched ``gather`` returns the stored bytes."""
    import numpy as np
    from sgb200 import data_util
    rs = np.random.RandomState(0)
    imgs = rs.randint(0, 256, size=(10, 6, 5, 3)).astype(np.uint8)
    labels = rs.randint(0, 4, size=10)
    path = str(tmp_path / "toy.npz")
    np.savez(path, imgs=imgs, labels=labels)
    ds = data_util.Dataset_("toy", None, True, hdf5_path=path, random_flip=False)
    assert len(ds) == 10
    x, y = ds[3]
    ref = (torch.from_numpy(imgs[3]).permute(2, 0, 1).float().div(255) - 0.5) / 0.5
    assert torch.equal(x, ref) and y == int(labels[3])
    out_i, out_l = torch.empty((4, 6, 5, 3), dtype=torch.uint8), torch.empty(4, dtype=torch.int64)
    ds.gather([7, 0, 2, 2], out_i, out_l)
    assert np.array_equal(out_i.numpy(), imgs[[7, 0, 2, 2]]) and out_l.tolist() == labels[[7, 0, 2, 2]].tolist()


def test_spectral_norm_table_orders_cbn_packs_contiguously_and_counts_pack_units():
    """Host logic of snbatch: the conditional-BN gain / bias linears lead the layer table so that their bf16 packs form ONE
    [rows][K] matrix (snbatch.cbn_affine_all: all cBN affine maps of a gradient-free pass as one GEMM), every layer keeps its
    own u / v slices, and tile_start counts the pack kernel's work units (include/sgb200.h, sgb_sn_layer)."""
    from sgb200 import snbatch
    from sgb200.utils import ops
    G, D = _build(dict(conv_dim=16, depth=2, attn=True))
    for net in (G, D):
        sb = net._snb
        sb._build(torch.device("cpu"))
        t = np.frombuffer(sb.table.numpy().tobytes(), dtype=snbatch.LAYER_DTYPE)
        assert len(t) == len(sb.mods) and len({id(m) for m in sb.mods}) == len(sb.mods)
        # work units: cumulative, taps * ceil(Cout/32) * ceil(Cin/32) per layer (no layer of these networks has more than 9 taps)
        units = 0
        for e in t:
            assert int(e["tile_start"]) == units
            units += int(e["taps"]) * ((int(e["Cout"]) + 31) // 32) * ((int(e["Cin"]) + 31) // 32)
        assert sb.max_blocks[2] == units
        # packs: 128-byte aligned, non-overlapping, in table order
        end = 0
        for (of, od, nf, shf, shd, su, sv), e in zip(sb.slices, t):
            assert of % 64 == 0 and of >= end and nf == int(e["Cout_p"]) * int(e["taps"]) * int(e["Cin_p"])
            end = of + nf
    cbn_lin = [m for mod in G.modules() if isinstance(mod, ops.ConditionalBatchNorm2d) for m in (mod.gain, mod.bias)]
    n, rows, Kp, of0, spans = G._snb.cbn
    assert n == len(cbn_lin) >= 16 and set(map(id, G._snb.mods[:n])) == set(map(id, cbn_lin))
    assert all(getattr(m, "_cbn_affine", False) for m in G._snb.mods[:n]) and not any(getattr(m, "_cbn_affine", False) for m in G._snb.mods[n:])
    r = 0
    for m, (r0, c), sl in zip(G._snb.mods[:n], spans, G._snb.slices):
        assert r0 == r and c == m.out_features and sl[0] == of0 + r0 * Kp and m.in_features <= Kp
        r += (c + 7) // 8 * 8
    assert r == rows
    assert D._snb.cbn is None                                   # no conditional batch norm in the discriminator
