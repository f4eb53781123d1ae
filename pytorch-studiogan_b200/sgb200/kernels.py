"""Tensor-level wrappers over the C ABI (no autograd here; see autograd_ops.py).

Activation convention: a torch tensor of logical shape [B, C, H, W], dtype bfloat16, whose memory is NHWC
(stride(1) == 1).  Channel slices ``x[:, a:b]`` stay valid (channel stride > C).  Everything runs on the
current CUDA stream of the tensor's device.
"""
import ctypes

import torch

from . import _lib as L

# ReLU masks of the discriminators travel to the backward as bit planes (1/16 of the bf16 bytes) wherever the layer allows
# them (conv_fprop want_relu_bits); BITS_STATS counts the planes written and consumed.
BITS_STATS = {"written": 0, "used": 0}

bf16 = torch.bfloat16


def empty_nhwc(B, C, H, W, device, dtype=bf16):
    return torch.empty((B, H, W, C), device=device, dtype=dtype).permute(0, 3, 1, 2)


def zeros_nhwc(B, C, H, W, device, dtype=bf16):
    return torch.zeros((B, H, W, C), device=device, dtype=dtype).permute(0, 3, 1, 2)


def geom(x):
    """(B, C, H, W, channel_stride) of an NHWC-in-memory activation; raises on any other layout."""
    B, C, H, W = x.shape
    sb, sc, sh, sw = x.stride()
    if C > 1 and sc != 1:
        raise RuntimeError("sgb200: activation is not NHWC in memory (strides %s)" % (x.stride(),))
    cs = sw if W > 1 else (sh if H > 1 else sb)
    if W > 1 and H > 1 and sh != W * cs:
        raise RuntimeError("sgb200: unexpected row stride %s" % (x.stride(),))
    if B > 1 and sb != H * W * cs:
        raise RuntimeError("sgb200: unexpected batch stride %s" % (x.stride(),))
    return B, C, H, W, cs


def as_nhwc(x):
    """Return x if it already is NHWC-in-memory bf16, otherwise re-layout through the library (rare guard path)."""
    try:
        if x.dtype == bf16:
            geom(x)
            return x
    except RuntimeError:
        pass
    B, C, H, W = x.shape
    out = empty_nhwc(B, C, H, W, x.device)
    out.copy_(x)  # layout guard only; never hit on the model paths (asserted in tests)
    return out


def _s():
    return L.stream_ptr()


# ---------------------------------------------------------------------------------------------- conv engine
def conv_fprop(x, w, Cout, KH, KW, pad_h, pad_w, bias=None, residual=None, res_up2=False, res_after_mask=False,
               mask=None, relu=False, alpha=1.0, alpha_ptr=None, out=None, out_fp32=False, w_mode=0, same_size=True, stride=1,
               res_scale=1.0, mask_bits=None, want_relu_bits=False, sm_mode=0, sm_stats=None, sm_delta=None, sm_p=None):
    """y = epilogue(conv(x, w)); see sgb_conv_fprop. ``w`` is a packed bf16 weight (layout by w_mode).
    want_relu_bits (with relu): also write the (y > 0) bit planes, returned as ``y._sgb_relu_bits`` (uint8 [B, H, W, Cout / 8]);
    mask_bits: such a tensor, used instead of ``mask`` by the input-gradient launch of the layer that consumed y.
    same_size=False: output grid = Hin + 2*pad - K + 1 ("valid"-style); stride=2 stores its even positions only.
    res_scale: multiplier of the residual (0.25 with res_up2 = average-pool backward added in the epilogue)."""
    B, Cin, Hin, Win, xcs = geom(x)
    H, W = (Hin, Win) if same_size else (Hin + 2 * pad_h - KH + 1, Win + 2 * pad_w - KW + 1)
    Ho, Wo = ((H + 1) // 2, (W + 1) // 2) if stride == 2 else (H, W)
    if out is None:
        out = empty_nhwc(B, Cout, Ho, Wo, x.device, torch.float32 if out_fp32 else bf16)
    _, _, _, _, ycs = geom(out)
    d = L.ConvDesc()
    d.B, d.H, d.W, d.Cin, d.Cout = B, H, W, Cin, Cout
    if not same_size:
        d.Hin, d.Win = Hin, Win
    d.out_sub = 2 if stride == 2 else 0
    d.KH, d.KW, d.pad_h, d.pad_w = KH, KW, pad_h, pad_w
    d.x, d.x_cstride = x.data_ptr(), xcs
    d.w, d.w_mode = w.data_ptr(), w_mode
    d.alpha = alpha
    d.alpha_ptr = alpha_ptr.data_ptr() if alpha_ptr is not None else None
    d.bias = bias.data_ptr() if bias is not None else None
    if residual is not None:
        d.residual, d.res_cstride = residual.data_ptr(), geom(residual)[4]
    d.res_up2 = 1 if res_up2 else 0
    d.res_scale = float(res_scale)
    d.res_after_mask = 1 if res_after_mask else 0
    if mask_bits is not None:
        assert mask_bits.dtype == torch.uint8 and mask_bits.numel() == B * H * W * Cout // 8 and Cout % 64 == 0
        d.mask_bits, mask = mask_bits.data_ptr(), None
        BITS_STATS["used"] += 1
    if mask is not None:
        d.mask, d.mask_cstride = mask.data_ptr(), geom(mask)[4]
    d.relu = 1 if relu else 0
    bits = None
    if want_relu_bits and relu and Cout % 64 == 0 and stride == 1 and out.dtype == bf16 and ycs % 8 == 0:
        bits = torch.empty((B, H, W, Cout // 8), device=x.device, dtype=torch.uint8)
        d.relu_bits = bits.data_ptr()
        out._sgb_relu_bits = bits
        BITS_STATS["written"] += 1
    d.y, d.y_cstride, d.y_fp32 = out.data_ptr(), ycs, 1 if out.dtype == torch.float32 else 0
    if sm_mode:
        d.sm_mode = sm_mode
        if sm_mode in (1, 2):
            if sm_stats is None:
                parts = L.load().sgb_conv_softmax_parts(ctypes.byref(d))
                sm_stats = torch.empty(B * H * W * parts * 2, device=x.device, dtype=torch.float32)
            d.sm_stats = sm_stats.data_ptr()
        else:
            d.sm_delta, d.sm_p, d.sm_p_cstride = sm_delta.data_ptr(), sm_p.data_ptr(), geom(sm_p)[4]
    # algorithmic bytes: every operand tensor once (the residual at its own resolution), weights once
    nb = 2.0 * B * Hin * Win * Cin + out.element_size() * float(B * Ho * Wo * Cout) + 2.0 * Cout * Cin * KH * KW * (B if w_mode else 1)
    if residual is not None:
        nb += 2.0 * B * H * W * Cout / (4 if res_up2 else 1)
    if mask is not None:
        nb += 2.0 * B * H * W * Cout
    if mask_bits is not None:
        nb += B * H * W * Cout / 8.0
    if bits is not None:
        nb += B * H * W * Cout / 8.0
    if sm_mode == 1:
        nb -= out.element_size() * float(B * Ho * Wo * Cout)        # the statistics pass stores no tile
    if sm_mode == 3:
        nb += 2.0 * B * H * W * Cout
    # accounting kind = the kernel the library dispatches (csrc/umma_conv3x3.cu conv3x3_rows_eligible): the halo-row kernel, the
    # generic kernel on a k x k filter (tensor bound) or on a 1x1 filter (HBM bound at these channel counts)
    rows = (KH == 3 and KW == 3 and pad_h == 1 and pad_w == 1 and w_mode == 0 and same_size and stride == 1 and W % 128 == 0
            and H % 2 == 0 and Cin % 64 == 0 and Cin <= 128 and Cout % 8 == 0)
    kind = "conv3x3_rows" if rows else ("conv_fprop_1x1" if KH * KW == 1 else "conv_fprop_kxk")
    L.call("sgb_conv_fprop", ctypes.byref(d), _s(), tag="%s %dx%d %d->%d @%dx%d m%d" % (kind, KH, KW, Cin, Cout, H, W, w_mode),
           flops=2.0 * B * H * W * Cout * Cin * KH * KW, nbytes=nb)
    if sm_mode == 1:
        return out, sm_stats
    return out


def dhead_fwd(h, w1, sigma1, b1, E, sigmaE, labels):
    """adv [B] of the discriminator head (see sgb_dhead_fwd); h fp32 [B, C] contiguous."""
    B, C = h.shape
    adv = torch.empty(B, device=h.device, dtype=torch.float32)
    L.call("sgb_dhead_fwd", L.ptr(h), L.ptr(w1), L.ptr(sigma1), L.ptr(b1), L.ptr(E), L.ptr(sigmaE), L.ptr(labels), B, C, L.ptr(adv), _s())
    return adv


def dhead_bwd(dadv, h, w1, sigma1, E, sigmaE, labels, need_dh=True, need_w=True):
    """(dh [B, C] | None, gw1 [1, C] | None, gE [n_cls, C] | None, db1 [1] | None): gradients of the EFFECTIVE head weights."""
    B, C = h.shape
    dh = torch.empty_like(h) if need_dh else None
    gw1 = torch.empty((1, C), device=h.device, dtype=torch.float32) if need_w else None
    db1 = torch.empty(1, device=h.device, dtype=torch.float32) if need_w else None
    gE = torch.zeros_like(E) if (need_w and E is not None) else None
    L.call("sgb_dhead_bwd", L.ptr(dadv), L.ptr(h), L.ptr(w1), L.ptr(sigma1), L.ptr(E), L.ptr(sigmaE), L.ptr(labels), B, C,
           L.ptr(dh), L.ptr(gw1), L.ptr(gE), L.ptr(db1), _s())
    return dh, gw1, gE, db1


def rowdot(x, y):
    """fp32 [B*H*W]: sum over channels of x * y (bf16 NHWC tensors of equal shape)."""
    B, C, H, W, xs = geom(x)
    out = torch.empty(B * H * W, device=x.device, dtype=torch.float32)
    L.call("sgb_rowdot", L.ptr(x), xs, L.ptr(y), geom(y)[4], B * H * W, C, L.ptr(out), _s(), nbytes=_nb(x, y))
    return out


def conv_wgrad(x, dy, KH, KW, pad_h, pad_w, dw=None, accumulate=False, per_image=False, want_dbias=False, dbias_acc=None):
    """fp32 weight gradient in the fprop-pack layout [Cout][KH*KW][Cin] (or [B][...] when per_image).
    want_dbias: returns (dw, dbias) where dbias is the fp32 [Cout] bias gradient if this launch can produce it for free,
    else None (the caller then reduces dy itself).  dbias_acc (with accumulate=True): an fp32 [Cout] tensor the launch ADDS
    the bias gradient to (a view of the gradient arena); returns (dw, True) when it did."""
    B, Cin, H, W, xcs = geom(x)
    _, Cout, _, _, dcs = geom(dy)
    if dw is None:
        shape = (B, Cout, KH * KW, Cin) if per_image else (Cout, KH * KW, Cin)
        dw = torch.empty(shape, device=x.device, dtype=torch.float32)
        accumulate = False
    d = L.WgradDesc()
    d.B, d.H, d.W, d.Cin, d.Cout = B, H, W, Cin, Cout
    d.KH, d.KW, d.pad_h, d.pad_w = KH, KW, pad_h, pad_w
    d.x, d.x_cstride = x.data_ptr(), xcs
    d.dy, d.dy_cstride = dy.data_ptr(), dcs
    d.dw, d.accumulate, d.per_image = dw.data_ptr(), 1 if accumulate else 0, 1 if per_image else 0
    dbias = None
    if dbias_acc is not None:
        assert accumulate and dbias_acc.dtype == torch.float32 and dbias_acc.numel() == Cout and dbias_acc.is_contiguous()
        if L.load().sgb_conv_wgrad_fuses_dbias(ctypes.byref(d)):
            d.dbias = dbias_acc.data_ptr()
            dbias = True
        want_dbias = True
    elif want_dbias and L.load().sgb_conv_wgrad_fuses_dbias(ctypes.byref(d)):
        # accumulate: the launch zeroes neither dw nor dbias, so dbias starts from zeros here
        dbias = (torch.zeros if accumulate else torch.empty)(Cout, device=x.device, dtype=torch.float32)
        d.dbias = dbias.data_ptr()
    L.call("sgb_conv_wgrad", ctypes.byref(d), _s(), tag="conv_wgrad %dx%d %d->%d @%dx%d%s" % (KH, KW, Cin, Cout, H, W, " per-image" if per_image else ""),
           flops=2.0 * B * H * W * Cout * Cin * KH * KW, nbytes=2.0 * B * H * W * (Cin + Cout) + 4.0 * dw.numel())
    return (dw, dbias) if want_dbias else dw


# ---------------------------------------------------------------------------------------------- spectral norm
def sn_workspace(R, K, device):
    n = L.load().sgb_sn_workspace_floats(R, K)
    return torch.zeros(n, device=device, dtype=torch.float32)


def sn_power_iter(W, u, v, sigma, ws, eps, do_power_iteration):
    R = W.shape[0]
    K = W.numel() // R
    L.call("sgb_sn_power_iter", L.ptr(W), L.ptr(u), L.ptr(v), L.ptr(sigma), L.ptr(ws), R, K, eps,
           1 if do_power_iteration else 0, _s())


def _nb(*ts):
    """Algorithmic bytes of an element-wise launch: every operand read or written once (profile accounting only)."""
    return float(sum(t.numel() * t.element_size() for t in ts if t is not None))


def pad8(c):
    return (c + 7) // 8 * 8


def weight_pack(W, sigma, Cout, Cin, taps, want_fprop=True, want_dgrad=True, perm_S=1):
    """bf16 packs of W/sigma; channel extents are zero-padded to multiples of 8 (TMA stride granularity)."""
    Cout_p, Cin_p = pad8(Cout), pad8(Cin)
    alloc = torch.zeros if (Cout_p != Cout or Cin_p != Cin) else torch.empty
    wf = alloc((Cout_p, taps, Cin_p), device=W.device, dtype=bf16) if want_fprop else None
    wd = alloc((Cin_p, taps, Cout_p), device=W.device, dtype=bf16) if want_dgrad else None
    L.call("sgb_weight_pack", L.ptr(W), L.ptr(sigma), L.ptr(wf), L.ptr(wd), Cout, Cin, taps, perm_S, Cout_p, Cin_p, _s())
    return wf, wd


def sn_backward(G, W, u, v, sigma, Cout, Cin, taps, perm_S=1, out=None):
    """G: fp32 [Cout_p][taps][Cin_p] from conv_wgrad -> dL/dW in the module's [Cout][Cin][taps] layout.
    out: accumulate into this tensor (a view of the flat gradient arena) instead of returning a new one."""
    dW = torch.empty_like(W) if out is None else out
    scratch = torch.empty(1, device=W.device, dtype=torch.float32) if sigma is not None else None
    L.call("sgb_sn_backward", L.ptr(G), L.ptr(W), L.ptr(u), L.ptr(v), L.ptr(sigma), L.ptr(scratch), L.ptr(dW), Cout, Cin, taps,
           perm_S, pad8(Cin), 0 if out is None else 1, _s())
    return dW


# ---------------------------------------------------------------------------------------------- batch norm
def bn_stats(x):
    B, C, H, W, cs = geom(x)
    s = torch.empty((2, C), device=x.device, dtype=torch.float32)
    L.call("sgb_bn_stats", L.ptr(x), B * H * W, C, cs, L.ptr(s[0]), L.ptr(s[1]), _s(), nbytes=_nb(x))
    return s


def bn_finalize(stats, count, running_mean, running_var, momentum, eps, use_batch_stats, track, mode, gain, bias, nb, C,
                device):
    mean = torch.empty(C, device=device, dtype=torch.float32)
    rstd = torch.empty(C, device=device, dtype=torch.float32)
    scale = torch.empty((nb, C), device=device, dtype=torch.float32)
    shift = torch.empty((nb, C), device=device, dtype=torch.float32)
    L.call("sgb_bn_finalize", L.ptr(stats[0]) if stats is not None else None, L.ptr(stats[1]) if stats is not None else None,
           float(count), L.ptr(running_mean), L.ptr(running_var), float(momentum), float(eps), int(use_batch_stats),
           1 if track else 0, mode, L.ptr(gain), L.ptr(bias), nb, C, L.ptr(mean), L.ptr(rstd), L.ptr(scale), L.ptr(shift),
           _affine_ld(gain, bias, mode, C), _s())
    return mean, rstd, scale, shift


def _affine_ld(gain, bias, mode, C):
    """Row stride of the per-image gain / bias of a conditional batch norm: C, or the width of the batched affine GEMM output
    they are column slices of (snbatch.cbn_affine_all)."""
    if mode != 0 or gain is None or gain.dim() != 2 or gain.stride(0) == C:
        return 0
    assert gain.stride(1) == 1 and bias.stride(1) == 1 and gain.stride(0) == bias.stride(0)
    return gain.stride(0)


def scale_shift_act(x, scale, shift, per_image, relu, up2):
    B, C, H, W, cs = geom(x)
    y = empty_nhwc(B, C, 2 * H if up2 else H, 2 * W if up2 else W, x.device)
    L.call("sgb_scale_shift_act", L.ptr(x), B, H, W, C, cs, L.ptr(scale), L.ptr(shift), 1 if per_image else 0, 1 if relu else 0,
           1 if up2 else 0, L.ptr(y), geom(y)[4], _s(), nbytes=_nb(x, y))
    return y


def bn_bwd_reduce(dy, x, scale, shift, per_image, mean, rstd, relu, up2):
    B, C, H, W, cs = geom(x)
    s12 = torch.empty((2, B, C), device=x.device, dtype=torch.float32)
    S12 = torch.empty((2, C), device=x.device, dtype=torch.float32)
    L.call("sgb_bn_bwd_reduce", L.ptr(dy), geom(dy)[4], L.ptr(x), cs, B, H, W, C, L.ptr(scale), L.ptr(shift),
           1 if per_image else 0, L.ptr(mean), L.ptr(rstd), 1 if relu else 0, 1 if up2 else 0, L.ptr(s12[0]), L.ptr(s12[1]),
           L.ptr(S12[0]), L.ptr(S12[1]), _s(), nbytes=_nb(dy, x))
    return s12, S12


def bn_bwd_apply(dy, x, scale, shift, per_image, mean, rstd, S12, count, relu, up2, use_batch_stats):
    B, C, H, W, cs = geom(x)
    dx = empty_nhwc(B, C, H, W, x.device)
    L.call("sgb_bn_bwd_apply", L.ptr(dy), geom(dy)[4], L.ptr(x), cs, B, H, W, C, L.ptr(scale), L.ptr(shift),
           1 if per_image else 0, L.ptr(mean), L.ptr(rstd), L.ptr(S12[0]) if S12 is not None else None,
           L.ptr(S12[1]) if S12 is not None else None, float(count), 1 if relu else 0, 1 if up2 else 0,
           1 if use_batch_stats else 0, L.ptr(dx), geom(dx)[4], _s(), nbytes=_nb(dy, x, dx))
    return dx


# ---------------------------------------------------------------------------------------------- element-wise
def axpby(x, y=None, a=1.0, b=1.0, a_dev=None, mask=None, relu=False, out=None):
    B, C, H, W, xs = geom(x)
    if out is None:
        out = empty_nhwc(B, C, H, W, x.device)
    L.call("sgb_axpby", L.ptr(x), xs, L.ptr(y), geom(y)[4] if y is not None else 0, L.ptr(mask),
           geom(mask)[4] if mask is not None else 0, L.ptr(out), geom(out)[4], B * H * W, C, float(a), L.ptr(a_dev), float(b),
           1 if relu else 0, _s(), nbytes=_nb(x, y, mask, out))
    return out


def pool2_fwd(x, mode, out=None):
    """mode 0 average, 1 max (2x2, stride 2)."""
    B, C, H, W, xs = geom(x)
    if out is None:
        out = empty_nhwc(B, C, H // 2, W // 2, x.device)
    L.call("sgb_pool2_fwd", L.ptr(x), xs, L.ptr(out), geom(out)[4], B, H // 2, W // 2, C, mode, _s(), nbytes=_nb(x, out))
    return out


def relu_pool2(x):
    """(relu(x), avgpool2(relu(x))) in one pass."""
    B, C, H, W, xs = geom(x)
    a0 = empty_nhwc(B, C, H, W, x.device)
    y = empty_nhwc(B, C, H // 2, W // 2, x.device)
    L.call("sgb_relu_pool2", L.ptr(x), xs, L.ptr(a0), geom(a0)[4], L.ptr(y), geom(y)[4], B, H // 2, W // 2, C, _s(),
           nbytes=_nb(x, a0, y))
    return a0, y


def pool2_bwd(dy, mode, x=None, add=None, relu_src=None, relu_bits=None):
    """relu_bits: the bit planes of the post-ReLU input (see conv_fprop), used instead of ``relu_src``."""
    B, C, Ho, Wo, dys = geom(dy)
    dx = empty_nhwc(B, C, 2 * Ho, 2 * Wo, dy.device)
    if relu_bits is not None:
        assert relu_bits.dtype == torch.uint8 and relu_bits.numel() == B * 4 * Ho * Wo * C // 8 and C % 64 == 0
        rsrc, rs = relu_bits.data_ptr(), -1
        BITS_STATS["used"] += 1
    else:
        rsrc, rs = L.ptr(relu_src), geom(relu_src)[4] if relu_src is not None else 0
    L.call("sgb_pool2_bwd", L.ptr(dy), dys, L.ptr(x), geom(x)[4] if x is not None else 0, L.ptr(add),
           geom(add)[4] if add is not None else 0, rsrc, rs, L.ptr(dx),
           geom(dx)[4], B, Ho, Wo, C, mode, _s(), nbytes=_nb(dy, x, add, relu_bits if relu_bits is not None else relu_src, dx))
    return dx


def softmax_rows(s, n, out=None):
    if out is None:
        out = torch.empty_like(s)
    L.call("sgb_softmax_rows", L.ptr(s), L.ptr(out), s.numel() // n, n, _s(), nbytes=_nb(s, out))
    return out


def softmax_bwd_rows(p, dp, n, out=None):
    if out is None:
        out = torch.empty_like(p)
    L.call("sgb_softmax_bwd_rows", L.ptr(p), L.ptr(dp), L.ptr(out), p.numel() // n, n, _s(), nbytes=_nb(p, dp, out))
    return out


def dot(x, y):
    out = torch.empty(1, device=x.device, dtype=torch.float32)
    L.call("sgb_dot", L.ptr(x), L.ptr(y), x.numel(), L.ptr(out), _s())
    return out


def sum_hw(x, relu):
    B, C, H, W, xs = geom(x)
    h = torch.empty((B, C), device=x.device, dtype=torch.float32)
    L.call("sgb_sum_hw", L.ptr(x), xs, B, H * W, C, 1 if relu else 0, L.ptr(h), _s())
    return h


def sum_hw_bwd(dh, x, relu):
    B, C, H, W, xs = geom(x)
    dx = empty_nhwc(B, C, H, W, x.device)
    L.call("sgb_sum_hw_bwd", L.ptr(dh), L.ptr(x), xs, L.ptr(dx), geom(dx)[4], B, H * W, C, 1 if relu else 0, _s())
    return dx


def img_to_nhwc(img, Cp=8):
    """NCHW fp32 image -> NHWC bf16 activation with channels zero-padded to Cp."""
    B, C, H, W = img.shape
    img = img.contiguous()
    out = empty_nhwc(B, Cp, H, W, img.device)
    L.call("sgb_img_to_nhwc", L.ptr(img), L.ptr(out), B, C, H * W, Cp, _s())
    return out


def nhwc_to_img(x, C, tanh=False):
    """First C channels of an NHWC activation (bf16 or fp32) -> contiguous NCHW fp32 (optionally tanh)."""
    B, Cx, H, W, cs = geom(x)
    img = torch.empty((B, C, H, W), device=x.device, dtype=torch.float32)
    L.call("sgb_nhwc_to_img", L.ptr(x), 1 if x.dtype == torch.float32 else 0, cs, L.ptr(img), B, C, H * W, 1 if tanh else 0, _s())
    return img


def img_grad_to_nhwc(dimg, y=None, Cp=8):
    B, C, H, W = dimg.shape
    dimg = dimg.contiguous()
    out = empty_nhwc(B, Cp, H, W, dimg.device)
    L.call("sgb_img_grad_to_nhwc", L.ptr(dimg), L.ptr(y), L.ptr(out), B, C, H * W, Cp, _s())
    return out


def col27(src):
    """3x3 patch gather of a 3-channel image: NCHW fp32 [B,3,H,W] or NHWC bf16 activation (first 3 channels) -> [B,32,H,W]."""
    if src.dtype == torch.float32:
        B, C, H, W = src.shape
        src = src.contiguous()
        nchw, cs = 1, 0
    else:
        B, C, H, W, cs = geom(src)
        nchw = 0
    out = empty_nhwc(B, 32, H, W, src.device)
    L.call("sgb_col27", L.ptr(src), nchw, cs, L.ptr(out), B, H, W, _s())
    return out


def col27_bwd(dcol):
    B, C, H, W, cs = geom(dcol)
    assert C == 32 and cs == 32
    dimg = torch.empty((B, 3, H, W), device=dcol.device, dtype=torch.float32)
    L.call("sgb_col27_bwd", L.ptr(dcol), L.ptr(dimg), B, H, W, _s())
    return dimg


def zero_stuff2(x):
    """[B, C, H, W] -> [B, C, 2H, 2W] with x at the even positions and zeros elsewhere (adjoint of ``[::2, ::2]``)."""
    B, C, H, W, xs = geom(x)
    y = empty_nhwc(B, C, 2 * H, 2 * W, x.device)
    L.call("sgb_zero_stuff2", L.ptr(x), xs, L.ptr(y), geom(y)[4], B, H, W, C, _s(), nbytes=_nb(x, y))
    return y


def pool3x3(x, stride, pad, mode, out=None):
    """Inception 3x3 pooling; mode 0 = average (count_include_pad=False), 1 = max."""
    B, C, H, W, xs = geom(x)
    Ho, Wo = (H + 2 * pad - 3) // stride + 1, (W + 2 * pad - 3) // stride + 1
    if out is None:
        out = empty_nhwc(B, C, Ho, Wo, x.device)
    L.call("sgb_pool3x3", L.ptr(x), xs, L.ptr(out), geom(out)[4], B, H, W, C, stride, pad, mode, _s())
    return out


def quantize_u8(img):
    img = img.contiguous()
    out = torch.empty(img.shape, device=img.device, dtype=torch.uint8)
    L.call("sgb_quantize_u8", L.ptr(img), L.ptr(out), img.numel(), _s())
    return out


def quantize_resize_normalize(img, S=299, quantize=True, want_image=False, want_col=True, resizer="legacy"):
    """Fused eval pre-processing; returns (normalised resized image NCHW fp32 | None, stride-2 3x3 patch tensor | None).
    resizer: "legacy" (torch bilinear) or "friendly" (PIL 'F'-mode bilinear), src/utils/resize.py:50-94."""
    B, C, H, W = img.shape
    assert C == 3
    img = img.contiguous()
    So = (S - 3) // 2 + 1
    out_img = torch.empty((B, 3, S, S), device=img.device, dtype=torch.float32) if want_image else None
    out_col = empty_nhwc(B, 32, So, So, img.device) if want_col else None
    L.call("sgb_quantize_resize_normalize", L.ptr(img), 1 if quantize else 0, B, H, W, S, L.ptr(out_img), L.ptr(out_col),
           {"legacy": 0, "friendly": 1}[resizer], _s())
    return out_img, out_col


def u8_to_img(u8, flip=None, out=None):
    """uint8 NHWC [B,H,W,3] device tensor (+ optional uint8 [B] flip flags) -> NCHW fp32 in [-1,1]."""
    B, H, W, C = u8.shape
    assert C == 3 and u8.dtype == torch.uint8 and u8.is_contiguous()
    if out is None:
        out = torch.empty((B, 3, H, W), device=u8.device, dtype=torch.float32)
    L.call("sgb_u8_to_img", L.ptr(u8), L.ptr(flip), L.ptr(out), B, H, W, _s())
    return out


def cast_f32_to_bf16(x, scale=1.0, out=None):
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=bf16)
    L.call("sgb_cast_f32_to_bf16", L.ptr(x), L.ptr(out), x.numel(), float(scale), _s())
    return out


def cast_bf16_to_f32(x):
    out = torch.empty(x.shape, device=x.device, dtype=torch.float32)
    L.call("sgb_cast_bf16_to_f32", L.ptr(x), L.ptr(out), x.numel(), _s())
    return out


def adam_ema_step(p, g, m, v, lr, beta1, beta2, eps, step, ema=None, ema_decay=0.0, grad_scale=1.0, step_dev=None):
    """``step_dev``: optional int32 device scalar holding the step count (used instead of ``step``; CUDA-graph safe)."""
    L.call("sgb_adam_ema_step", L.ptr(p), L.ptr(g), L.ptr(m), L.ptr(v), p.numel(), float(lr), float(beta1), float(beta2),
           float(eps), int(step), L.ptr(step_dev), L.ptr(ema), float(ema_decay), float(grad_scale), _s())


def ema_lerp(ema, p, decay):
    L.call("sgb_ema_lerp", L.ptr(ema), L.ptr(p), p.numel(), float(decay), _s())


# ---------------------------------------------------------------------------------------------- gradient penalty
def gp_interpolate(real, fake, alpha):
    """alpha[b] * real + (1 - alpha[b]) * fake on contiguous fp32 [B, ...] tensors (torch's operation order)."""
    real, fake = real.contiguous(), fake.contiguous()
    out = torch.empty_like(real)
    B = real.shape[0]
    L.call("sgb_gp_interpolate", L.ptr(real), L.ptr(fake), L.ptr(alpha), L.ptr(out), B, real.numel() // B, _s())
    return out


def gp_sumsq(g):
    g = g.contiguous()
    B = g.shape[0]
    out = torch.empty(B, device=g.device, dtype=torch.float32)
    L.call("sgb_gp_sumsq", L.ptr(g), L.ptr(out), B, g.numel() // B, _s())
    return out


def gp_seed(g, sumsq):
    g = g.contiguous()
    B = g.shape[0]
    v = torch.empty_like(g)
    L.call("sgb_gp_seed", L.ptr(g), L.ptr(sumsq), L.ptr(v), B, g.numel() // B, _s())
    return v


def bn_tangent_bwd_reduce(x, a, c, mean, rstd):
    B, C, H, W, xs = geom(x)
    sums = torch.empty((5, C), device=x.device, dtype=torch.float32)
    L.call("sgb_bn_tangent_bwd_reduce", L.ptr(x), xs, L.ptr(a), geom(a)[4], L.ptr(c), geom(c)[4], B * H * W, C, L.ptr(mean),
           L.ptr(rstd), L.ptr(sums), _s())
    return sums


def bn_tangent_bwd_apply(x, a, c, gamma, mean, rstd, sums, count, use_batch_stats, want_dx=True, want_da=True):
    B, C, H, W, xs = geom(x)
    dx = empty_nhwc(B, C, H, W, x.device) if want_dx else None
    da = empty_nhwc(B, C, H, W, x.device) if want_da else None
    L.call("sgb_bn_tangent_bwd_apply", L.ptr(x), xs, L.ptr(a), geom(a)[4], L.ptr(c), geom(c)[4], B * H * W, C,
           L.ptr(gamma) if gamma is not None else None, L.ptr(mean), L.ptr(rstd), L.ptr(sums) if sums is not None else None,
           float(count), 1 if use_batch_stats else 0, L.ptr(dx) if dx is not None else None, geom(dx)[4] if dx is not None else 0,
           L.ptr(da) if da is not None else None, geom(da)[4] if da is not None else 0, _s())
    return dx, da
