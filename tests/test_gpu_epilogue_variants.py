"""One launch per fused-epilogue variant the conv engine dispatches: every compile-time instantiation of the generic kernel
(conv_fprop_kernel<F>) and of the halo-row kernel (conv3x3_rows_kernel<F>), their run-time versions (F = -1) through the
staged-store and the direct-store paths.  Each case is built through kernels.conv_fprop with the operands that select its
variant and compared with fp32 torch on the same bf16 operands: one bf16 rounding of the output (8e-3 max-norm relative),
bit planes and masked outputs exactly.  Where CUPTI is available the instantiation that ran is read from the kernel name.
"""
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from test_gpu_parity import _cuda, bfr, rel_err, to_nhwc  # noqa: E402

# F bits (csrc/conv_epilogue.cuh): 1 bias, 2 ReLU, 4 residual, 8 residual after the mask, 16 mask, 32 Cout % 64 == 0,
# 64 mask as bit plane, 128 / 256 residual / mask through the aux ring, 512 ReLU bit plane out, 1024 / 2048 / 4096 softmax.
GEN, ROWS = "conv_fprop_kernel", "conv3x3_rows_kernel"
_G = dict(B=2, H=16, W=16, Cin=64, Cout=128, k=1)       # generic kernel, one 128-wide channel tile, staged stores
_R = dict(B=1, H=8, W=128, Cin=64, Cout=64, k=3)        # halo-row kernel: row 0 staged, row 1 direct stores (C = 64)
CONV_CASES = [
    # (kernel, F, shape, epilogue operands)
    (GEN, 32, _G, {}),                                                       # plain (dgrad / GEMM)
    (GEN, 33, _G, dict(bias=True)),                                          # generator conv
    (GEN, 35, _G, dict(bias=True, relu=True)),                               # discriminator conv
    (GEN, 547, _G, dict(bias=True, relu=True, bits=True)),                   # ... writing the ReLU bit plane
    (GEN, 164, _G, dict(res="full")),                                        # residual through the aux ring
    (GEN, 165, _G, dict(bias=True, res="full")),                             # block output + skip
    (GEN, 167, _G, dict(bias=True, relu=True, res="full")),                  # ... with the next block's ReLU
    (GEN, 679, _G, dict(bias=True, relu=True, res="full", bits=True)),       # ... writing the ReLU bit plane
    (GEN, 112, _G, dict(mask="bits")),                                       # dgrad through a ReLU (bit plane)
    (GEN, 244, _G, dict(mask="bits", res="up2")),                            # fused block entry (bit plane + pooled skip)
    (GEN, 304, _G, dict(mask="bf16")),                                       # dgrad through a ReLU (bf16 mask tile)
    (GEN, 308, _G, dict(mask="bf16", res="up2")),                            # fused block entry (bf16 mask tile)
    (GEN, -1, _G, dict(mask="bf16", res="full", res_after=True)),            # run-time flags, staged stores (post-mask residual)
    (GEN, -1, dict(_G, Cout=96), dict(bias=True, relu=True)),                # run-time flags, staged stores, ragged channel tile
    (GEN, -1, _G, dict(bias=True, fp32=True)),                               # direct stores: fp32 output
    (GEN, -1, dict(_G, Cout=64, k=3), dict(bias=True, relu=True, stride=2)),  # direct stores: stride 2 (out_sub)
    (GEN, -1, dict(_G, Cout=24, k=3), dict(bias=True, relu=True, res="full")),  # direct stores: 24-channel tile
    (GEN, -1, dict(_G, Cout=3), dict(bias=True, relu=True, res="full", mask="bf16")),  # direct stores: scalar tail (Cout = 3)
    (GEN, -1, dict(_G, Cin=128, k=3), dict(bias=True, relu=True, bits=True)),  # direct stores: K = 1152 above the staging limit
    (ROWS, 32, _R, {}),
    (ROWS, 33, _R, dict(bias=True)),
    (ROWS, 35, _R, dict(bias=True, relu=True)),
    (ROWS, 547, _R, dict(bias=True, relu=True, bits=True)),
    (ROWS, 48, _R, dict(mask="bf16")),
    (ROWS, 112, _R, dict(mask="bits")),
    (ROWS, -1, _R, dict(bias=True, res="full")),                             # run-time flags on both rows
]


def _case_id(c):
    kern, f, shape, ops = c
    return "%s-%d-%s" % ("rows" if kern == ROWS else "gen", f, "-".join(sorted(ops)) or "plain")


_CUPTI = []


def _cupti_available():
    """True when torch.profiler records device kernels on this machine (checked once on a torch kernel)."""
    if not _CUPTI:
        from torch.profiler import ProfilerActivity, profile
        try:
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                torch.ones(16, device="cuda").mul_(2)
                torch.cuda.synchronize()
            _CUPTI.append(any(e.device_type == torch.autograd.DeviceType.CUDA for e in prof.events()))
        except Exception:
            _CUPTI.append(False)
    return _CUPTI[0]


def _run_checking_variant(launch, kern, f):
    """launch() under torch.profiler; asserts that exactly the instantiation kern<f> ran (when CUPTI is available)."""
    if not _cupti_available():
        return launch()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = launch()
        torch.cuda.synchronize()
    ran = {m.group(0) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
           for m in [re.search(r"(conv_fprop_kernel|conv3x3_rows_kernel)<-?\d+>", e.name)] if m}
    assert ran == {"%s<%d>" % (kern, f)}, ran
    return out


def conv_case(c, dev):
    """(launch, ref, ctx) of one conv case: launch() -> y (its ReLU bit plane as y._sgb_relu_bits), ref: fp32 torch."""
    from sgb200 import kernels as K
    kern, f, shape, ops = c
    B, H, W, Cin, Cout, k = (shape[n] for n in ("B", "H", "W", "Cin", "Cout", "k"))
    stride = ops.get("stride", 1)
    g = torch.Generator().manual_seed(1000 * (f + 2) + Cin + Cout + k + 7 * len(ops))
    x = bfr(torch.randn(B, Cin, H, W, generator=g))
    w = torch.randn(Cout, Cin, k, k, generator=g) / np.sqrt(Cin * k * k)
    b = torch.randn(Cout, generator=g)
    up2 = ops.get("res") == "up2"
    r = bfr(torch.randn(B, Cout, H // 2, W // 2, generator=g)) if up2 else bfr(torch.randn(B, Cout, H, W, generator=g))
    rs = 0.25 if up2 else 1.0
    m = bfr(torch.randn(B, Cout, H, W, generator=g))
    wf, _ = K.weight_pack(w.to(dev), None, Cout, Cin, k * k, True, False)
    kw = dict(bias=b.to(dev) if ops.get("bias") else None, relu=bool(ops.get("relu")), stride=stride,
              out_fp32=bool(ops.get("fp32")), want_relu_bits=bool(ops.get("bits")))
    if ops.get("res"):
        kw.update(residual=to_nhwc(r, dev), res_up2=up2, res_scale=rs, res_after_mask=bool(ops.get("res_after")))
    if ops.get("mask") == "bf16":
        kw["mask"] = to_nhwc(m, dev)
    elif ops.get("mask") == "bits":
        planes = np.packbits((m > 0).permute(0, 2, 3, 1).numpy(), axis=-1, bitorder="little")
        kw["mask_bits"] = torch.from_numpy(planes).to(dev)
    xd = to_nhwc(x, dev)

    def launch(**over):
        return K.conv_fprop(xd, wf, Cout, k, k, k // 2, k // 2, **dict(kw, **over))

    y = F.conv2d(x, bfr(w), padding=k // 2)
    if ops.get("bias"):
        y = y + b[None, :, None, None]
    rr = r.repeat_interleave(2, 2).repeat_interleave(2, 3) if up2 else r
    if ops.get("res") and not ops.get("res_after"):
        y = y + rs * rr
    if ops.get("relu"):
        y = torch.relu(y)
    if ops.get("mask"):
        y = torch.where(m > 0, y, torch.zeros(()))
    if ops.get("res") and ops.get("res_after"):
        y = y + rs * rr
    if stride == 2:
        y = y[:, :, ::2, ::2]
    return launch, y, dict(m=m, kw=kw)


@pytest.mark.parametrize("case", CONV_CASES, ids=[_case_id(c) for c in CONV_CASES])
def test_conv_epilogue_variant(case):
    kern, f, shape, ops = case
    dev = _cuda()
    launch, ref, ctx = conv_case(case, dev)
    y = _run_checking_variant(launch, kern, f)
    assert y.dtype == (torch.float32 if ops.get("fp32") else torch.bfloat16)
    assert rel_err(y, ref) < 8e-3
    yc = y.float().cpu()
    if ops.get("mask") and not ops.get("res_after"):
        assert (yc[ctx["m"] <= 0] == 0).all()                      # masked outputs are exact zeros
    if ops.get("mask") == "bits":                                  # the bit plane masks exactly like the bf16 tensor
        assert torch.equal(y, launch(mask=to_nhwc(ctx["m"], dev), mask_bits=None))
    if ops.get("bits"):
        pos = (y.permute(0, 2, 3, 1).float() > 0).cpu().numpy()
        got = y._sgb_relu_bits.cpu().numpy()
        diff = np.unpackbits(got ^ np.packbits(pos, axis=-1, bitorder="little"), axis=-1, bitorder="little").astype(bool)
        # a positive accumulator below the smallest bf16 rounds to zero in y but keeps its bit: allow only that direction
        assert diff.mean() < 1e-6 and not (diff & pos).any()


SM_CASES = [1056, 2080, 4128]     # softmax statistics, softmax apply, softmax backward (P through the aux ring)


def softmax_case(f, dev):
    """(launch, ref) of one attention-softmax epilogue launch: theta [B, c8, S, S], keys / values at S / 2."""
    from sgb200 import kernels as K
    B, S, c8, c2 = 2, 32, 64, 128
    N, M = S * S, (S // 2) * (S // 2)
    g = torch.Generator().manual_seed(f)
    theta = bfr(torch.randn(B, c8, S, S, generator=g) * 0.7)
    phi = bfr(torch.randn(B, c8, S // 2, S // 2, generator=g) * 0.7)
    th, ph = to_nhwc(theta, dev), to_nhwc(phi, dev)
    s = torch.bmm(theta.reshape(B, c8, N).transpose(1, 2), phi.reshape(B, c8, M))      # [B, N, M] scores
    if f == 1056:
        def launch():
            return K.conv_fprop(th, ph, M, 1, 1, 0, 0, w_mode=1, sm_mode=1)[1]
        return launch, s
    P, stats = K.conv_fprop(th, ph, M, 1, 1, 0, 0, w_mode=1, sm_mode=1)
    if f == 2080:
        def launch():
            return K.conv_fprop(th, ph, M, 1, 1, 0, 0, w_mode=1, sm_mode=2, sm_stats=stats, out=P)
        return launch, torch.softmax(s, -1)
    K.conv_fprop(th, ph, M, 1, 1, 0, 0, w_mode=1, sm_mode=2, sm_stats=stats, out=P)
    gv = bfr(torch.randn(B, c2, S // 2, S // 2, generator=g))
    do = bfr(torch.randn(B, c2, S, S, generator=g))
    delta = torch.randn(B * N, generator=g) * 0.1
    gd, dod, dd = to_nhwc(gv, dev), to_nhwc(do, dev), delta.to(dev)

    def launch():
        return K.conv_fprop(dod, gd, M, 1, 1, 0, 0, w_mode=1, sm_mode=3, sm_delta=dd, sm_p=P)
    Pb = P.permute(0, 2, 3, 1).reshape(B, N, M).float().cpu()
    dP = torch.bmm(do.reshape(B, c2, N).transpose(1, 2), gv.reshape(B, c2, M))
    return launch, Pb * (dP - delta.reshape(B, N, 1))


@pytest.mark.parametrize("f", SM_CASES)
def test_softmax_epilogue_variant(f):
    dev = _cuda()
    launch, ref = softmax_case(f, dev)
    out = _run_checking_variant(launch, GEN, f)
    B, N, M = ref.shape
    if f == 1056:                      # per-row (max, sum exp) partials, merged as the apply pass merges them
        st = out.reshape(B * N, -1, 2).double().cpu()
        m = st[..., 0].max(-1).values
        l = (st[..., 1] * torch.exp(st[..., 0] - m[:, None])).sum(-1)
        r = ref.reshape(B * N, M).double()
        assert float((m - r.max(-1).values).abs().max()) < 8e-3 * float(r.abs().max())
        assert rel_err(l, torch.exp(r - r.max(-1, keepdim=True).values).sum(-1)) < 8e-3
    else:
        assert rel_err(out.permute(0, 2, 3, 1).reshape(B, N, M), ref) < 8e-3
