"""torch.autograd.Function wrappers: the forward/backward of every hot-path op is a sequence of libsgb200 calls.

Conventions
* activations: NHWC-in-memory bf16 tensors of logical shape [B, C, H, W] (see kernels.py)
* "premasked" protocol for ReLU chains in the discriminators: a conv with ``relu=True`` stores its post-ReLU
  output; whoever consumes that output is responsible for delivering a gradient already masked by (output > 0)
  (the consumer's dgrad epilogue does it for free via ``mask_input=True``).  That gradient is therefore the
  gradient w.r.t. the pre-activation and is used as is.
"""
import torch
import torch.distributed as dist
from torch.autograd import Function

from . import kernels as K

bf16 = torch.bfloat16

# ---- tangent tape (gradient penalty, utils/gp.py) ---------------------------------------------------------------------
# While TAPE is a list, every op applied through ``<Fn>.call(...)`` is appended as (rule, args, outputs); replaying the
# tape with ``rule.tangent(args, outputs, tan)`` pushes a tangent (directional derivative) through the same network.
# ``tan(t)`` returns the tangent of primal tensor t or None (zero).  SKIP_PARAM_GRADS suppresses weight gradients in a
# backward pass that only needs the input gradient (first pass of the penalty).
TAPE = None
SKIP_PARAM_GRADS = False


def tape_record(rule, args, out):
    if TAPE is not None:
        TAPE.append((rule, args, out))


class TFunction(Function):
    """autograd.Function + ``call`` (apply and record on the tangent tape) + ``tangent`` (its JVP rule, itself built
    from differentiable Functions so that the tangent pass can be back-propagated)."""

    @classmethod
    def call(cls, *args):
        out = cls.apply(*args)
        if TAPE is not None:
            TAPE.append((cls, args, out))
        return out

    @staticmethod
    def tangent(args, out, tan):
        raise NotImplementedError("no tangent rule for this op (gradient penalty through it is unsupported)")


def _direct_grad(p):
    """The arena-backed ``.grad`` of a leaf parameter that opted in (utils/arena.GradArena.attach), else None.  ConvFn then
    adds its weight gradient there itself and reports no gradient to autograd, which would otherwise launch one tiny add
    per parameter and backward pass (~1.6 k per step for BigGAN-Deep)."""
    if not getattr(p, "_sgb_direct_grad", False) or not p.is_leaf or torch.is_grad_enabled():
        return None
    g = p.grad
    if g is None or g.dtype != torch.float32 or not g.is_contiguous() or g.shape != p.shape:
        return None
    return g


def _tadd(a, b):
    if a is None:
        return b
    if b is None:
        return a
    return AddFn.apply(a, b)


class SpectralNormState:
    """u / v buffers + workspace of one spectrally-normalised weight (torch/nn/utils/spectral_norm.py semantics)."""

    def __init__(self, module, eps):
        self.module = module
        self.eps = eps
        self.ws = None

    def tensors(self):
        m = self.module
        W = m.weight_orig
        if self.ws is None or self.ws.device != W.device:
            R = W.shape[0]
            self.ws = K.sn_workspace(R, W.numel() // R, W.device)
        return m.weight_u, m.weight_v, self.ws


def _grad_bf16(dy):
    """Incoming gradient as NHWC bf16 (fp32 grads appear only on the tiny [B,C,1,1] cBN gain/bias branches)."""
    if dy.dtype == torch.float32:
        B, C, H, W = dy.shape
        out = K.empty_nhwc(B, C, H, W, dy.device)
        if H * W == 1:
            K.cast_f32_to_bf16(dy.contiguous(), out=out)
        else:
            K.cast_f32_to_bf16(dy.permute(0, 2, 3, 1).contiguous(), out=out)
        return out
    return K.as_nhwc(dy)


def _direct_grad_ptr(p):
    """Device address of the arena-backed ``.grad`` of a parameter (see _direct_grad), else None.  Frozen parameters keep
    their arena slot, so the batched spectral-norm backward may address it (their pass buffer holds zeros)."""
    if not getattr(p, "_sgb_direct_grad", False) or not p.is_leaf:
        return None
    g = p.grad
    if g is None or g.dtype != torch.float32 or not g.is_contiguous() or g.shape != p.shape:
        return None
    return g.data_ptr()


def conv_param_grads(x, dz, weight, need_w, need_b, KH, KW, pad, dims, sigma, u_saved, v_saved, perm_S=1, sn_pass=None, bias=None):
    """Weight and bias gradient of y = conv(x, W / sigma) + b given dz = dL/dy (NHWC bf16): tcgen05 weight-gradient kernel,
    then the spectral-norm chain rule (sgb_sn_backward).  The weight gradient is added straight into the flat gradient
    arena when the parameter opted in (returns None for it then).  The bias gradient rides on the weight-gradient launch
    (a constant-ones operand on the tensor pipe, sgb_conv_wgrad_fuses_dbias); only a frozen weight with a live bias falls
    back to a reduction pass."""
    Cout, Cin, taps = dims
    dW = dbias = None
    if need_w and sn_pass is not None and sn_pass[0] is not None and _direct_grad(weight) is not None and sn_pass[0].usable():
        # batched path: accumulate the raw weight gradient into this forward pass's flat buffer; the spectral-norm chain
        # rule of ALL layers runs as one launch pair when the backward pass ends (snbatch._Pass.flush)
        G = sn_pass[0].g_slice(sn_pass[1])
        btgt = _direct_grad(bias) if (need_b and bias is not None and dz.shape[1] == Cout) else None
        if btgt is not None:
            # the bias gradient is added straight into the gradient arena by the same launch (no tensor, no accumulate kernel)
            _, done = K.conv_wgrad(x, dz, KH, KW, pad, pad, dw=G, accumulate=True, dbias_acc=btgt)
            if done:
                need_b = False
        elif need_b:
            _, dbias = K.conv_wgrad(x, dz, KH, KW, pad, pad, dw=G, accumulate=True, want_dbias=True)
            if dbias is not None:
                dbias = dbias[:Cout]
        else:
            K.conv_wgrad(x, dz, KH, KW, pad, pad, dw=G, accumulate=True)
    elif need_w:
        if need_b:
            G, dbias = K.conv_wgrad(x, dz, KH, KW, pad, pad, want_dbias=True)
            if dbias is not None:
                dbias = dbias[:Cout]
        else:
            G = K.conv_wgrad(x, dz, KH, KW, pad, pad)
        tgt = _direct_grad(weight)
        if tgt is not None:       # accumulate straight into the flat gradient arena: no per-parameter add kernel
            K.sn_backward(G, weight, u_saved, v_saved, sigma, Cout, Cin, taps, perm_S, out=tgt)
        else:
            dW = K.sn_backward(G, weight, u_saved, v_saved, sigma, Cout, Cin, taps, perm_S)
    if need_b and dbias is None:
        dbias = K.bn_stats(dz)[0][:Cout]
    return dW, dbias


class ConvFn(TFunction):
    """y = [relu](conv(x, W / sigma) + bias [+ residual])  — conv2d (stride 1) or linear (H = W = 1).

    cfg keys: KH, KW, pad, relu, premasked, mask_input, res_up2, res_channels, out_fp32, perm_S, sn (SpectralNormState|None),
    do_power_iteration.
    """

    @staticmethod
    def forward(ctx, x, weight, bias, residual, cfg):
        KH, KW, pad = cfg["KH"], cfg["KW"], cfg["pad"]
        Cout = weight.shape[0]
        Cin = weight.numel() // (Cout * KH * KW)
        taps = KH * KW
        sn = cfg.get("sn")
        sigma = u_saved = v_saved = None
        need_dx = ctx.needs_input_grad[0]
        need_dw = ctx.needs_input_grad[1]
        cache = cfg.get("sn_cache")
        if cache is not None:                       # power iteration + packs already done by the network's batched pass
            wf, wd, sigma, u_saved, v_saved = cache
            u = v = None
        else:
            if sn is not None:
                u, v, ws = sn.tensors()
                sigma = torch.empty(1, device=weight.device, dtype=torch.float32)
                K.sn_power_iter(weight, u, v, sigma, ws, sn.eps, cfg.get("do_power_iteration", True))
            wf, wd = K.weight_pack(weight, sigma, Cout, Cin, taps, True, need_dx, cfg.get("perm_S", 1))
        Cout_p = K.pad8(Cout)
        res = residual
        y = K.conv_fprop(x, wf, Cout_p, KH, KW, pad, pad, bias=bias if Cout_p == Cout else _pad_bias(bias, Cout_p),
                         residual=res, res_up2=cfg.get("res_up2", False), relu=cfg.get("relu", False),
                         out_fp32=cfg.get("out_fp32", False), stride=cfg.get("stride", 1),
                         want_relu_bits=cfg.get("premasked", False) and any(ctx.needs_input_grad))
        ctx.x_bits = getattr(x, "_sgb_relu_bits", None) if (need_dx and cfg.get("mask_input", False)) else None
        if need_dw and sn is not None and cache is None:
            u_saved, v_saved = u.clone(), v.clone()
        ctx.cfg = cfg
        ctx.dims = (Cout, Cin, taps)
        ctx.bias_ref = bias                          # the parameter object (arena-backed .grad), not a saved activation
        ctx.has_res = residual is not None
        ctx.res_shape = residual.shape if residual is not None else None
        ctx.save_for_backward(x, weight, wd, sigma, u_saved, v_saved, y if cfg.get("relu", False) else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, wd, sigma, u_saved, v_saved, y = ctx.saved_tensors
        cfg = ctx.cfg
        KH, KW, pad = cfg["KH"], cfg["KW"], cfg["pad"]
        Cout, Cin, taps = ctx.dims
        dz = _grad_bf16(dy)
        if cfg.get("relu", False) and not cfg.get("premasked", False):
            dz = K.axpby(dz, mask=y)
        if cfg.get("stride", 1) == 2:
            # y = conv_same(x)[::2, ::2] (the engine's out_sub store): the gradient on the stride-1 grid is dz zero-stuffed
            dz = K.zero_stuff2(dz)
        dx = dW = dbias = dres = None
        if ctx.needs_input_grad[0]:
            mask = x if cfg.get("mask_input", False) else None
            mbits = ctx.x_bits
            if Cout <= 3 and KH == 3 and KW == 3 and pad == 1 and cfg.get("perm_S", 1) == 1:
                # C -> 3 image convolution (generator output layer): its input gradient is a 3 -> C convolution of the
                # 3-channel dz; gather dz's 3x3 patches (K = 27 -> 32) and run it as a 1x1 GEMM instead of a K-padded 3x3.
                wsn = weight if sigma is None else weight / sigma
                wcol = wsn.flip(2, 3).permute(1, 2, 3, 0).reshape(Cin, 27).contiguous()
                wf2, _ = K.weight_pack(wcol, None, Cin, 27, 1, True, False)
                dx = K.conv_fprop(K.col27(dz), wf2, K.pad8(Cin), 1, 1, 0, 0, mask=mask)
            else:
                dx = K.conv_fprop(dz, wd, K.pad8(Cin), KH, KW, KH - 1 - pad, KW - 1 - pad, mask=mask, mask_bits=mbits)
            if dx.shape[1] != x.shape[1]:
                dx = dx[:, :x.shape[1]]
        if not SKIP_PARAM_GRADS:
            dW, dbias = conv_param_grads(x, dz, weight, ctx.needs_input_grad[1], ctx.needs_input_grad[2], KH, KW, pad, ctx.dims,
                                         sigma, u_saved, v_saved, cfg.get("perm_S", 1), cfg.get("sn_pass"), ctx.bias_ref)
        if ctx.has_res and ctx.needs_input_grad[3]:
            dres = K.pool2_fwd(dz, 2) if cfg.get("res_up2", False) else dz
            rc = ctx.res_shape[1]
            if dres.shape[1] != rc:  # residual was read from the first Cout channels of a wider tensor
                full = K.zeros_nhwc(dres.shape[0], rc, dres.shape[2], dres.shape[3], dres.device)
                K.axpby(dres, out=full[:, :dres.shape[1]])
                dres = full
        return dx, dW, dbias, dres, None

    @staticmethod
    def tangent(args, out, tan):
        """d/d(eps) [relu](conv(x) + b + res) = [y > 0] * (conv(tx) + t_res): same weights, no bias, no new power
        iteration (the primal call's sigma / packs are reused through cfg['sn_cache'])."""
        x, weight, bias, residual, cfg = args
        tx, tres = tan(x), tan(residual)
        if cfg.get("out_fp32", False) or cfg.get("perm_S", 1) != 1:
            raise NotImplementedError("tangent of fp32-output / permuted linear layers")
        if tx is None:
            t = tres
            if t is not None and cfg.get("res_up2", False):
                raise NotImplementedError("tangent through an up-sampled residual without a main-branch tangent")
        else:
            tcfg = {"KH": cfg["KH"], "KW": cfg["KW"], "pad": cfg["pad"], "relu": False, "res_up2": cfg.get("res_up2", False),
                    "sn": cfg.get("sn"), "sn_cache": cfg.get("sn_cache"), "sn_pass": cfg.get("sn_pass"), "do_power_iteration": False}
            t = ConvFn.apply(tx, weight, None, tres, tcfg)
        if t is not None and cfg.get("relu", False):
            t = MaskFn.apply(t, out)
        return t


class ConvTranspose4x4s2Fn(TFunction):
    """nn.ConvTranspose2d(kernel 4, stride 2, padding 1) (DCGAN generator, src/models/deep_conv.py:20) on the stride-1 engine:
       y = conv_same_4x4(zero_stuff(x), W~) with W~[co][ci][kh][kw] = W[ci][co][3-kh][3-kw] and tap offsets -2..+1.
    Reading the [Cin, Cout, 4, 4] module weight as a conv weight V ("Cout" = Cin), the DGRAD pack of V is exactly the fprop
    pack of W~ and the FPROP pack of V its dgrad pack, so no new pack kernel is needed.  Backward: dx = the even positions of
    the 4x4 dgrad (the engine's out_sub store); dW~ from the weight-gradient kernel on (zero_stuff(x), dy), re-indexed to W."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        Cin, Cout = weight.shape[0], weight.shape[1]
        assert tuple(weight.shape[2:]) == (4, 4)
        xu = K.zero_stuff2(x)
        v_f, v_d = K.weight_pack(weight, None, Cin, Cout, 16, True, True)      # V = weight as [rows = Cin][cols = Cout][16]
        y = K.conv_fprop(xu, v_d, Cout, 4, 4, 2, 2, bias=bias)
        ctx.dims = (Cin, Cout)
        ctx.save_for_backward(xu, v_f)
        return y

    @staticmethod
    def backward(ctx, dy):
        xu, v_f = ctx.saved_tensors
        Cin, Cout = ctx.dims
        dz = _grad_bf16(dy)
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            dx = K.conv_fprop(dz, v_f, Cin, 4, 4, 1, 1, stride=2)
        if ctx.needs_input_grad[1] and not SKIP_PARAM_GRADS:
            G, db = K.conv_wgrad(xu, dz, 4, 4, 2, 2, want_dbias=ctx.needs_input_grad[2])     # dW~ as [Cout][tap][Cin]
            dW = G.flip(1).permute(2, 0, 1).reshape(Cin, Cout, 4, 4).contiguous()            # dW[ci][co][t] = dW~[co][15 - t][ci]
        if ctx.needs_input_grad[2] and db is None and not SKIP_PARAM_GRADS:
            db = K.bn_stats(dz)[0][:Cout]
        return dx, dW, db


class MaskFn(TFunction):
    """t * [src > 0]: tangent of a ReLU whose (post- or pre-activation) primal is ``src``; linear in t, no gradient to
    src (the mask is piecewise constant)."""

    @staticmethod
    def forward(ctx, t, src):
        ctx.save_for_backward(src)
        return K.axpby(K.as_nhwc(t), mask=src)

    @staticmethod
    def backward(ctx, dy):
        (src,) = ctx.saved_tensors
        return K.axpby(K.as_nhwc(dy), mask=src), None


def _pad_bias(bias, Cout_p):
    if bias is None:
        return None
    out = torch.zeros(Cout_p, device=bias.device, dtype=torch.float32)
    out[:bias.numel()] = bias
    return out


class BNActFn(TFunction):
    """y = [relu](batch_norm(x) * g + b) with g/b per image (cBN), per channel (affine) or absent; optional nearest x2
    upsample of the result.  cfg keys: mode (0 cBN, 1 affine, 2 plain), relu, up2, use_batch_stats, track, momentum, eps, group.
    """

    @staticmethod
    def forward(ctx, x, gain, bias, running_mean, running_var, cfg):
        B, C, H, W, _ = K.geom(x)
        mode = cfg["mode"]
        stats = None
        count = float(B * H * W)
        group = cfg.get("group")
        if cfg["use_batch_stats"]:
            stats = K.bn_stats(x)
            if group is not None:
                dist.all_reduce(stats, group=group)
                count *= dist.get_world_size(group)
        nb = B if mode == 0 else 1
        g = gain.reshape(nb, C) if gain is not None else None
        b = bias.reshape(nb, C) if bias is not None else None
        rows_ok = lambda t: t.dim() == 2 and t.stride(1) == 1      # column slice of the batched affine GEMM: row stride > C
        if g is not None and not g.is_contiguous() and not (rows_ok(g) and b is not None and rows_ok(b) and g.stride(0) == b.stride(0)):
            g = g.contiguous()
        if b is not None and not b.is_contiguous() and not (g is not None and rows_ok(g) and rows_ok(b) and g.stride(0) == b.stride(0)):
            b = b.contiguous()
        mean, rstd, scale, shift = K.bn_finalize(stats, count, running_mean, running_var, cfg["momentum"], cfg["eps"],
                                                 (2 if cfg.get("clamp_eps") else 1) if cfg["use_batch_stats"] else 0,
                                                 cfg["track"], mode, g, b, nb, C, x.device)
        y = K.scale_shift_act(x, scale, shift, mode == 0, cfg["relu"], cfg["up2"])
        ctx.cfg = cfg
        ctx.count = count
        ctx.gshape = gain.shape if gain is not None else None
        ctx.bshape = bias.shape if bias is not None else None
        ctx.save_for_backward(x, scale, shift, mean, rstd)
        if TAPE is not None:
            cfg["_tangent_stats"] = (mean, rstd, count)
        return y

    @staticmethod
    def tangent(args, out, tan):
        x, gain, bias, running_mean, running_var, cfg = args
        tx = tan(x)
        if tx is None:
            return None
        if cfg["mode"] == 0 or cfg["up2"]:
            raise NotImplementedError("tangent of conditional / up-sampling batch norm (generator-side op)")
        mean, rstd, count = cfg["_tangent_stats"]
        t = BNTangentFn.apply(x, tx, gain, mean, rstd, {"count": count, "use_batch_stats": cfg["use_batch_stats"],
                                                         "group": cfg.get("group")})
        return MaskFn.apply(t, out) if cfg["relu"] else t

    @staticmethod
    def backward(ctx, dy):
        x, scale, shift, mean, rstd = ctx.saved_tensors
        cfg = ctx.cfg
        mode = cfg["mode"]
        dy = K.as_nhwc(dy)
        s12, S12 = K.bn_bwd_reduce(dy, x, scale, shift, mode == 0, mean, rstd, cfg["relu"], cfg["up2"])
        group = cfg.get("group")
        if cfg["use_batch_stats"] and group is not None:
            dist.all_reduce(S12, group=group)
        if cfg.get("clamp_eps") and cfg["use_batch_stats"]:
            # DataParallel-mode variant: where the variance was clamped, inv_std is a constant and the variance term of the
            # gradient vanishes (rare mode; a [C]-sized tensor op)
            S12[1].mul_((rstd < (cfg["eps"] ** -0.5) * (1.0 - 1e-6)).to(S12.dtype))
        dx = None
        if ctx.needs_input_grad[0]:
            dx = K.bn_bwd_apply(dy, x, scale, shift, mode == 0, mean, rstd, S12, ctx.count, cfg["relu"], cfg["up2"],
                                cfg["use_batch_stats"])
        dgain = dbias = None
        if mode == 0:
            if ctx.needs_input_grad[1]:
                dgain = s12[1].reshape(ctx.gshape)
            if ctx.needs_input_grad[2]:
                dbias = s12[0].reshape(ctx.bshape)
        elif mode == 1:
            if ctx.needs_input_grad[1]:
                dgain = s12[1].sum(0).reshape(ctx.gshape)
            if ctx.needs_input_grad[2]:
                dbias = s12[0].sum(0).reshape(ctx.bshape)
        return dx, dgain, dbias, None, None, None


class BNTangentFn(TFunction):
    """t = gamma * r * (a - mean(a) - xhat * mean(xhat * a)): the tangent map of y = gamma * xhat + beta with batch
    statistics (r = rstd; running statistics: t = gamma * r * a).  Its own backward returns the derivatives w.r.t. the
    primal input x, the incoming tangent a and gamma (torch: batchnorm_double_backward); mean / rstd are treated as the
    functions of x they are."""

    @staticmethod
    def forward(ctx, x, a, gamma, mean, rstd, cfg):
        B, C, H, W, _ = K.geom(x)
        a = K.as_nhwc(a)
        g = gamma if gamma is not None else torch.ones(C, device=x.device, dtype=torch.float32)
        scale = (g * rstd).reshape(1, C).contiguous()
        shift = torch.zeros_like(scale)
        S12 = None
        if cfg["use_batch_stats"]:
            _, S12 = K.bn_bwd_reduce(a, x, scale, shift, False, mean, rstd, False, False)
            if cfg.get("group") is not None:
                dist.all_reduce(S12, group=cfg["group"])
        t = K.bn_bwd_apply(a, x, scale, shift, False, mean, rstd, S12, cfg["count"], False, False, cfg["use_batch_stats"])
        ctx.cfg = cfg
        ctx.has_gamma = gamma is not None
        ctx.save_for_backward(x, a, gamma, mean, rstd)
        return t

    @staticmethod
    def backward(ctx, c):
        x, a, gamma, mean, rstd = ctx.saved_tensors
        cfg = ctx.cfg
        c = K.as_nhwc(c)
        M = cfg["count"]
        sums = K.bn_tangent_bwd_reduce(x, a, c, mean, rstd)
        if cfg["use_batch_stats"] and cfg.get("group") is not None:
            dist.all_reduce(sums, group=cfg["group"])
        dx, da = K.bn_tangent_bwd_apply(x, a, c, gamma, mean, rstd, sums, M, cfg["use_batch_stats"],
                                        want_dx=ctx.needs_input_grad[0] and cfg["use_batch_stats"], want_da=ctx.needs_input_grad[1])
        dgamma = None
        if ctx.has_gamma and ctx.needs_input_grad[2]:
            Sa, Sc, Sxa, Sxc, Sac = sums.unbind(0)
            dgamma = rstd * (Sac - (Sa * Sc + Sxa * Sxc) / M) if cfg["use_batch_stats"] else rstd * Sac
        return dx, da, dgamma, None, None, None


class SplitResidualFn(TFunction):
    """x -> (x, x[:, :c]): main branch and channel-drop skip branch of a generator block
    (src/models/big_resnet_deep_legacy.py:50-53).  Backward adds the narrower skip gradient into the first channels of
    the main gradient in place."""

    @staticmethod
    def forward(ctx, x, c):
        return x.view_as(x), x[:, :c]

    @staticmethod
    def backward(ctx, d_main, d_res):
        if d_res is None:
            return d_main, None
        if d_main is None:
            raise RuntimeError("SplitResidualFn: skip gradient without a main-branch gradient")
        d_main = K.as_nhwc(d_main)
        d_res = K.as_nhwc(d_res)
        c = d_res.shape[1]
        tgt = d_main[:, :c]
        K.axpby(tgt, d_res, out=tgt)
        return d_main, None


class DBlockEntryFn(TFunction):
    """x -> (a0, skip_src) with a0 = relu(x) and skip_src = avgpool2(a0) | a0: the two consumers of a discriminator
    block input (src/models/big_resnet_deep_legacy.py:211-224).  The reference's d_act_fn is nn.ReLU(inplace=True)
    (src/config.py:486), which rectifies the aliased skip tensor ``x0`` as well, so the skip path carries relu(x).
    Both incoming gradients refer to a0; the result is masked once by (a0 > 0)."""

    @staticmethod
    def forward(ctx, x, downsample):
        if downsample and x.shape[2] % 2 == 0 and x.shape[3] % 2 == 0:
            a0, px = K.relu_pool2(x)
        else:
            a0 = K.axpby(x, relu=True)
            px = K.pool2_fwd(a0, 0) if downsample else a0.view_as(a0)
        ctx.downsample = downsample
        ctx.save_for_backward(a0)
        return a0, px

    @staticmethod
    def backward(ctx, da0, dpx):
        (a0,) = ctx.saved_tensors
        da0 = K.as_nhwc(da0) if da0 is not None else None
        dpx = K.as_nhwc(dpx) if dpx is not None else None
        if dpx is None:
            return K.axpby(da0, mask=a0), None
        if ctx.downsample:
            return K.pool2_bwd(dpx, 0, add=da0, relu_src=a0), None
        if da0 is None:
            return K.axpby(dpx, mask=a0), None
        return K.axpby(da0, dpx, mask=a0), None

    @staticmethod
    def tangent(args, out, tan):
        x, downsample = args
        tx = tan(x)
        if tx is None:
            return None, None
        ta0 = MaskFn.apply(tx, out[0])
        return ta0, (PoolFn.apply(ta0) if downsample else ta0)


class AvgPoolFn(TFunction):
    """2x2 average pooling; ``relu_src``: the input is a post-ReLU tensor and the gradient is returned premasked."""

    @staticmethod
    def forward(ctx, x, input_is_relu_out):
        ctx.input_is_relu_out = input_is_relu_out
        ctx.x_bits = getattr(x, "_sgb_relu_bits", None) if input_is_relu_out else None
        ctx.save_for_backward(x if (input_is_relu_out and ctx.x_bits is None) else None)
        return K.pool2_fwd(x, 0)

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        return K.pool2_bwd(K.as_nhwc(dy), 0, relu_src=x, relu_bits=ctx.x_bits), None

    @staticmethod
    def tangent(args, out, tan):
        tx = tan(args[0])
        return PoolFn.apply(tx) if tx is not None else None


class ReluFn(TFunction):
    @staticmethod
    def forward(ctx, x):
        y = K.axpby(x, relu=True)
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        return K.axpby(K.as_nhwc(dy), mask=y)

    @staticmethod
    def tangent(args, out, tan):
        tx = tan(args[0])
        return MaskFn.apply(tx, out) if tx is not None else None


class AddFn(TFunction):
    @staticmethod
    def forward(ctx, a, b):
        return K.axpby(a, b)

    @staticmethod
    def backward(ctx, dy):
        return dy, dy

    @staticmethod
    def tangent(args, out, tan):
        return _tadd(tan(args[0]), tan(args[1]))


class ReluPassFn(TFunction):
    """a0 = relu(x) for a consumer that returns its gradient already masked by (a0 > 0) (DEntryConvFn): the backward is the
    identity.  Used where the producer could not apply the ReLU in its own epilogue (after a self-attention block)."""

    @staticmethod
    def forward(ctx, x):
        return K.axpby(x, relu=True)

    @staticmethod
    def backward(ctx, da0):
        return da0


def _sn_packs(weight, cfg, Cout, Cin, taps, need_dx):
    """(fprop pack, dgrad pack, sigma, u, v) of a conv weight: the network's batched spectral-norm pass left them in
    cfg['sn_cache']; stand-alone use runs the per-layer kernels."""
    cache = cfg.get("sn_cache")
    if cache is not None:
        return cache
    sn = cfg.get("sn")
    sigma = us = vs = None
    if sn is not None:
        u, v, ws = sn.tensors()
        sigma = torch.empty(1, device=weight.device, dtype=torch.float32)
        K.sn_power_iter(weight, u, v, sigma, ws, sn.eps, cfg.get("do_power_iteration", True))
        us, vs = u.clone(), v.clone()
    wf, wd = K.weight_pack(weight, sigma, Cout, Cin, taps, True, need_dx)
    return wf, wd, sigma, us, vs


class DEntryConvFn(TFunction):
    """Entry of a BigGAN-Deep discriminator block (src/models/big_resnet_deep_legacy.py:211-224) as one op:
         a0 (= relu(block input); the producer's epilogue applied the in-place ReLU) ->
         h1 = relu(conv1x1(a0) + b1)  and  px = avgpool2(a0) | a0   (the skip source)
       px is written into the first channels of the concat-skip buffer (cfg['skip_channels'] wide) when the block has a
       learnable shortcut, so the concatenation of :225-226 needs no copy.
       backward: ONE dgrad launch forms  dx = [a0 > 0] * (dgrad1(dh1) + 0.25 * up2(dpx))  (or ... + dpx without pooling):
       the average-pool backward and both ReLU masks live in the conv epilogue (residual, res_up2, res_scale, mask)."""

    @staticmethod
    def forward(ctx, a0, weight, bias, cfg):
        B, Cin, H, W, _ = K.geom(a0)
        hid = weight.shape[0]
        wf, wd, sigma, us, vs = _sn_packs(weight, cfg, hid, Cin, 1, True)
        h1 = K.conv_fprop(a0, wf, hid, 1, 1, 0, 0, bias=bias, relu=True, want_relu_bits=any(ctx.needs_input_grad))
        ctx.a0_bits = getattr(a0, "_sgb_relu_bits", None) if ctx.needs_input_grad[0] else None
        down = cfg["downsample"]
        if down:
            sc = cfg.get("skip_channels", 0) or Cin
            buf = K.empty_nhwc(B, sc, H // 2, W // 2, a0.device)
            px = buf[:, :Cin] if sc != Cin else buf
            K.pool2_fwd(a0, 0, out=px)
            if sc != Cin:
                px._sgb_concat_buf = buf
        else:
            px = a0.view_as(a0)
        ctx.cfg = cfg
        ctx.dims = (hid, Cin, 1)
        ctx.bias_ref = bias
        ctx.save_for_backward(a0, weight, wd, sigma, us, vs)
        return h1, px

    @staticmethod
    def backward(ctx, dh1, dpx):
        a0, weight, wd, sigma, us, vs = ctx.saved_tensors
        cfg = ctx.cfg
        hid, Cin, _ = ctx.dims
        dz = K.as_nhwc(dh1)                       # premasked by conv2d2's dgrad epilogue
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            down = cfg["downsample"]
            dx = K.conv_fprop(dz, wd, Cin, 1, 1, 0, 0, mask=a0, mask_bits=ctx.a0_bits, residual=K.as_nhwc(dpx) if dpx is not None else None,
                              res_up2=down, res_scale=0.25 if down else 1.0)
        if not SKIP_PARAM_GRADS:
            dW, db = conv_param_grads(a0, dz, weight, ctx.needs_input_grad[1], ctx.needs_input_grad[2], 1, 1, 0, ctx.dims,
                                      sigma, us, vs, 1, cfg.get("sn_pass"), ctx.bias_ref)
        return dx, dW, db, None


class ConcatSkipFn(TFunction):
    """skip = cat([px, conv1x1(px)], channel) written into one buffer (learnable shortcut of the BigGAN-Deep D block,
    src/models/big_resnet_deep_legacy.py:225-226)."""

    @staticmethod
    def forward(ctx, px, weight, bias, cfg):
        B, Cin, H, W, _ = K.geom(px)
        Cextra = weight.shape[0]
        sn = cfg.get("sn")
        sigma = u_saved = v_saved = None
        need_dx = ctx.needs_input_grad[0]
        cache = cfg.get("sn_cache")
        if cache is not None:
            wf, wd, sigma, u_saved, v_saved = cache
        else:
            if sn is not None:
                u, v, ws = sn.tensors()
                sigma = torch.empty(1, device=weight.device, dtype=torch.float32)
                K.sn_power_iter(weight, u, v, sigma, ws, sn.eps, cfg.get("do_power_iteration", True))
            wf, wd = K.weight_pack(weight, sigma, Cextra, Cin, 1, True, need_dx)
        skip = getattr(px, "_sgb_concat_buf", None)       # DEntryConvFn pooled straight into the concat buffer
        if skip is None or skip.shape[1] != Cin + Cextra:
            skip = K.empty_nhwc(B, Cin + Cextra, H, W, px.device)
            K.axpby(px, out=skip[:, :Cin])
        K.conv_fprop(skip[:, :Cin], wf, Cextra, 1, 1, 0, 0, bias=bias, out=skip[:, Cin:])
        if ctx.needs_input_grad[1] and sn is not None and cache is None:
            u_saved, v_saved = u.clone(), v.clone()
        ctx.cfg = cfg
        ctx.dims = (Cextra, Cin)
        ctx.bias_ref = bias
        ctx.save_for_backward(px, weight, wd, sigma, u_saved, v_saved)
        return skip

    @staticmethod
    def backward(ctx, dskip):
        px, weight, wd, sigma, u_saved, v_saved = ctx.saved_tensors
        Cextra, Cin = ctx.dims
        dskip = K.as_nhwc(dskip)
        d_lo, d_hi = dskip[:, :Cin], dskip[:, Cin:]
        dpx = dW = dbias = None
        if ctx.needs_input_grad[0]:
            dpx = K.conv_fprop(d_hi, wd, Cin, 1, 1, 0, 0, residual=d_lo)
        if not SKIP_PARAM_GRADS:
            dW, dbias = conv_param_grads(px, d_hi, weight, ctx.needs_input_grad[1], ctx.needs_input_grad[2], 1, 1, 0,
                                         (Cextra, Cin, 1), sigma, u_saved, v_saved, 1, ctx.cfg.get("sn_pass"), ctx.bias_ref)
        return dpx, dW, dbias, None

    @staticmethod
    def tangent(args, out, tan):
        px, weight, bias, cfg = args
        tpx = tan(px)
        if tpx is None:
            return None
        return ConcatSkipFn.apply(tpx, weight, None, {"sn": cfg.get("sn"), "sn_cache": cfg.get("sn_cache"), "sn_pass": cfg.get("sn_pass"),
                                                       "do_power_iteration": False})


class SumHWFn(TFunction):
    """h[b, c] = sum_{h,w} relu(x) in fp32 (src/models/big_resnet_deep_legacy.py:344-345)."""

    @staticmethod
    def forward(ctx, x, relu):
        ctx.relu = relu
        ctx.save_for_backward(x)
        return K.sum_hw(x, relu)

    @staticmethod
    def backward(ctx, dh):
        (x,) = ctx.saved_tensors
        return K.sum_hw_bwd(dh.contiguous(), x, ctx.relu), None

    @staticmethod
    def tangent(args, out, tan):
        x, relu = args
        tx = tan(x)
        if tx is None:
            return None
        return SumHWFn.apply(MaskFn.apply(tx, x) if relu else tx, False)


class DHeadFn(TFunction):
    """Discriminator head on the sum-pooled features (src/models/big_resnet_deep_legacy.py:346-349,366-368; the same lines in
    big_resnet.py / resnet.py):  adv = <h, W1 / sigma1> + b1 [+ <h, E[y] / sigmaE>]  (projection discriminator or unconditional),
    one launch forward, two backward; the spectral-norm power iteration and chain rule use the same kernels as every layer.
    cfg: sn1 / snE (SpectralNormState | None), training, no_bias, reuse = the (sigma1, u1, v1, sigmaE, uE, vE) of an earlier call
    (tangent pass: same effective weights, no new power iteration); the call leaves its own tuple in cfg["saved"]."""

    @staticmethod
    def forward(ctx, h, w1, b1, E, labels, cfg):
        h = h.contiguous()
        reuse = cfg.get("reuse")
        if reuse is not None:
            s1, u1, v1, sE, uE, vE = reuse
        else:
            def power(w, sn):
                if sn is None:
                    return None, None, None
                u, v, ws = sn.tensors()
                sg = torch.empty(1, device=w.device, dtype=torch.float32)
                K.sn_power_iter(w.detach(), u, v, sg, ws, sn.eps, cfg.get("training", True))
                return sg, u.clone(), v.clone()
            s1, u1, v1 = power(w1, cfg.get("sn1"))
            sE, uE, vE = power(E, cfg.get("snE")) if E is not None else (None, None, None)
        cfg["saved"] = (s1, u1, v1, sE, uE, vE)
        adv = K.dhead_fwd(h, w1, s1, None if cfg.get("no_bias", False) else b1, E, sE, labels)
        ctx.has_E = E is not None
        ctx.has_b = b1 is not None and not cfg.get("no_bias", False)
        ctx.save_for_backward(h, w1, E, labels, s1, u1, v1, sE, uE, vE)
        return adv

    @staticmethod
    def backward(ctx, dadv):
        h, w1, E, labels, s1, u1, v1, sE, uE, vE = ctx.saved_tensors
        need_dh = ctx.needs_input_grad[0]
        need_w = ctx.needs_input_grad[1] or (ctx.has_E and ctx.needs_input_grad[3])
        dh, gw1, gE, db1 = K.dhead_bwd(dadv.contiguous().float(), h, w1, s1, E, sE, labels, need_dh, need_w and not SKIP_PARAM_GRADS)
        dW1 = dE = db = None
        if gw1 is not None and ctx.needs_input_grad[1]:
            C = h.shape[1]
            dW1 = K.sn_backward(gw1, w1, u1, v1, s1, 1, C, 1)
            if ctx.has_b and ctx.needs_input_grad[2]:
                db = db1
        if gE is not None and ctx.needs_input_grad[3]:
            dE = K.sn_backward(gE, E, uE, vE, sE, E.shape[0], E.shape[1], 1)
        return dh, dW1, db, dE, None, None

    @staticmethod
    def tangent(args, out, tan):
        h, w1, b1, E, labels, cfg = args
        th = tan(h)
        if th is None:
            return None
        return DHeadFn.apply(th, w1, None, E, labels, {"reuse": cfg["saved"], "no_bias": True})


class ToBF16Fn(TFunction):
    """[B, K] fp32 -> [B, Kp, 1, 1] bf16 activation (input of the linear layers); K is zero-padded to a multiple of 8
    (TMA stride granularity), e.g. the 10-way one-hot cBN input of ResNetGAN or BigGAN's 148-wide [embedding, z-chunk]."""

    @staticmethod
    def forward(ctx, x):
        B, Kd = x.shape
        Kp = K.pad8(Kd)
        ctx.Kd = Kd
        if Kp != Kd:
            xp = torch.zeros((B, Kp), device=x.device, dtype=x.dtype)
            xp[:, :Kd] = x
            x = xp
        out = torch.empty((B, Kp), device=x.device, dtype=bf16)
        K.cast_f32_to_bf16(x.contiguous(), out=out)
        return out.view(B, Kp, 1, 1)

    @staticmethod
    def backward(ctx, dy):
        B, Kp = dy.shape[0], dy.shape[1]
        g = dy.reshape(B, Kp) if dy.dtype == torch.float32 else K.cast_bf16_to_f32(dy.reshape(B, Kp).contiguous())
        return g[:, :ctx.Kd] if Kp != ctx.Kd else g


class ImageInFn(TFunction):
    """NCHW fp32 image in [-1, 1] -> NHWC bf16 activation with 8 (zero-padded) channels."""

    @staticmethod
    def forward(ctx, img):
        ctx.C = img.shape[1]
        return K.img_to_nhwc(img, 8)

    @staticmethod
    def backward(ctx, dy):
        return K.nhwc_to_img(K.as_nhwc(dy), ctx.C, tanh=False)

    @staticmethod
    def tangent(args, out, tan):
        t = tan(args[0])
        return ImageInFn.apply(t) if t is not None else None


class ImageColFn(TFunction):
    """NCHW fp32 image -> [B, 32, H, W] bf16 tensor of its 3x3 patches (k = tap*3 + c, zero padded): the operand of the
    3 -> C input convolution run as a K = 32 GEMM (see ops._ConvBase.forward)."""

    @staticmethod
    def forward(ctx, img):
        return K.col27(img)

    @staticmethod
    def backward(ctx, dcol):
        return K.col27_bwd(K.as_nhwc(dcol))

    @staticmethod
    def tangent(args, out, tan):
        t = tan(args[0])
        return ImageColFn.apply(t) if t is not None else None


class ImageOutFn(TFunction):
    """NHWC activation (>= 3 channels) -> tanh -> NCHW fp32 image (nn.Tanh at big_resnet_deep_legacy.py:183)."""

    @staticmethod
    def forward(ctx, x, C):
        img = K.nhwc_to_img(x, C, tanh=True)
        ctx.Cp = x.shape[1]
        ctx.save_for_backward(img)
        return img

    @staticmethod
    def backward(ctx, dimg):
        (img,) = ctx.saved_tensors
        return K.img_grad_to_nhwc(dimg, img, ctx.Cp), None


class SelfAttentionFn(TFunction):
    """ops.SelfAttention.forward (src/utils/ops.py:83-103) with the attention map materialised in bf16:
       theta = conv(x), phi = maxpool(conv(x)), g = maxpool(conv(x)); P = softmax(theta . phi^T); o = P . g;
       out = x + sigma * conv(o).  All contractions run on the tcgen05 engine (batched modes 1/2)."""

    @staticmethod
    def forward(ctx, x, w_theta, w_phi, w_g, w_o, sigma, cfgs):
        B, C, H, W, _ = K.geom(x)
        c8, c2 = C // 8, C // 2
        N, M = H * W, (H // 2) * (W // 2)
        packs = []
        sn_saved = []
        for w, cfg, cin, cout in ((w_theta, cfgs[0], C, c8), (w_phi, cfgs[1], C, c8), (w_g, cfgs[2], C, c2), (w_o, cfgs[3], c2, C)):
            sn = cfg.get("sn")
            sg = None
            us = vs = None
            cache = cfg.get("sn_cache")
            if cache is not None and cache[1] is not None:
                wf, wd, sg, us, vs = cache
            else:
                if sn is not None:
                    u, v, ws = sn.tensors()
                    sg = torch.empty(1, device=w.device, dtype=torch.float32)
                    K.sn_power_iter(w, u, v, sg, ws, sn.eps, cfg.get("do_power_iteration", True))
                    us, vs = u.clone(), v.clone()
                wf, wd = K.weight_pack(w, sg, cout, cin, 1, True, True)
            packs.append((wf, wd))
            sn_saved.append((sg, us, vs))
        theta = K.conv_fprop(x, packs[0][0], c8, 1, 1, 0, 0)                      # [B, c8, H, W]
        phi_f = K.conv_fprop(x, packs[1][0], c8, 1, 1, 0, 0)
        g_f = K.conv_fprop(x, packs[2][0], c2, 1, 1, 0, 0)
        phi = K.pool2_fwd(phi_f, 1)                                               # [B, c8, H/2, W/2]  keys  [M][c8]
        g = K.pool2_fwd(g_f, 1)                                                   # [B, c2, H/2, W/2]  values [M][c2]
        if M % 64 == 0:
            # the score GEMM runs twice (K = C/8 is tiny): a statistics pass that stores nothing, then the pass whose epilogue
            # writes P = softmax(theta . phi^T) directly -- the score matrix S never exists in memory
            S, stats = K.conv_fprop(theta, phi, M, 1, 1, 0, 0, w_mode=1, sm_mode=1)
            K.conv_fprop(theta, phi, M, 1, 1, 0, 0, w_mode=1, sm_mode=2, sm_stats=stats, out=S)
        else:
            S = K.conv_fprop(theta, phi, M, 1, 1, 0, 0, w_mode=1)                 # [B, M, H, W] == [B][N][M]
            K.softmax_rows(S, M, out=S)                                           # P in place
        o = K.conv_fprop(S, g, c2, 1, 1, 0, 0, w_mode=2)                          # [B, c2, H, W]
        t = K.conv_fprop(o, packs[3][0], C, 1, 1, 0, 0)                           # conv1x1_attn
        out = K.axpby(t, x, a=1.0, a_dev=sigma, b=1.0)
        ctx.dims = (B, C, H, W, c8, c2, N, M)
        ctx.sn_saved = sn_saved
        ctx.packs = packs
        ctx.save_for_backward(x, theta, phi_f, phi, g_f, g, S, o, t, sigma, w_theta, w_phi, w_g, w_o)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, theta, phi_f, phi, g_f, g, P, o, t, sigma, w_theta, w_phi, w_g, w_o = ctx.saved_tensors
        B, C, H, W, c8, c2, N, M = ctx.dims
        packs, sn_saved = ctx.packs, ctx.sn_saved
        dout = K.as_nhwc(dout)
        dsigma = K.dot(dout, t).reshape(sigma.shape)
        dt = K.axpby(dout, a=1.0, a_dev=sigma)
        # conv1x1_attn
        do = K.conv_fprop(dt, packs[3][1], c2, 1, 1, 0, 0)
        G_o = K.conv_wgrad(o, dt, 1, 1, 0, 0)
        # o = P . g   ->  dP = do . g^T (keys as output channels), dg = P^T . do (per image)
        dg_pool = K.conv_wgrad(do, P, 1, 1, 0, 0, per_image=True)                 # [B][M][1][c2] fp32
        if M % 64 == 0:
            # dS = P * (dP - delta) in the epilogue of the dP GEMM, delta = rowsum(dP * P) = rowsum(do * o): dP never exists
            dS = K.conv_fprop(do, g, M, 1, 1, 0, 0, w_mode=1, sm_mode=3, sm_delta=K.rowdot(do, o), sm_p=P)
        else:
            dP = K.conv_fprop(do, g, M, 1, 1, 0, 0, w_mode=1)                     # g as [B][M][c2] K-major operand
            dS = K.softmax_bwd_rows(P, dP, M, out=dP)
        # S = theta . phi^T -> dtheta = dS . phi (phi as [B][K=M][N=c8] MN-major), dphi = dS^T . theta (per image)
        dtheta = K.conv_fprop(dS, phi, c8, 1, 1, 0, 0, w_mode=2)
        dphi_pool = K.conv_wgrad(theta, dS, 1, 1, 0, 0, per_image=True)           # [B][M][1][c8] fp32
        dphi_p = K.cast_f32_to_bf16(dphi_pool.view(B, H // 2, W // 2, c8)).permute(0, 3, 1, 2)
        dg_p = K.cast_f32_to_bf16(dg_pool.view(B, H // 2, W // 2, c2)).permute(0, 3, 1, 2)
        dphi_f = K.pool2_bwd(dphi_p, 1, x=phi_f)
        dg_f = K.pool2_bwd(dg_p, 1, x=g_f)
        # the three input 1x1 convs: dx = dout + dgrads (chained through the residual epilogue)
        dx = K.conv_fprop(dtheta, packs[0][1], C, 1, 1, 0, 0, residual=dout)
        dx = K.conv_fprop(dphi_f, packs[1][1], C, 1, 1, 0, 0, residual=dx)
        dx = K.conv_fprop(dg_f, packs[2][1], C, 1, 1, 0, 0, residual=dx)
        grads_w = []
        for (w, xin, dyv, cout, cin, idx) in ((w_theta, x, dtheta, c8, C, 0), (w_phi, x, dphi_f, c8, C, 1), (w_g, x, dg_f, c2, C, 2),
                                              (w_o, o, None, C, c2, 3)):
            if not ctx.needs_input_grad[1 + idx]:
                grads_w.append(None)
                continue
            G = G_o if idx == 3 else K.conv_wgrad(xin, dyv, 1, 1, 0, 0)
            sg, us, vs = sn_saved[idx]
            grads_w.append(K.sn_backward(G, w, us, vs, sg, cout, cin, 1))
        return dx, grads_w[0], grads_w[1], grads_w[2], grads_w[3], dsigma, None


class ForkFn(TFunction):
    """x -> (x, x) for a tensor with two consumers; the two gradients are summed by the library instead of by autograd's
    implicit accumulation (keeps every full-size element-wise pass on the hot path inside libsgb200)."""

    @staticmethod
    def forward(ctx, x):
        return x.view_as(x), x.view_as(x)

    @staticmethod
    def backward(ctx, g1, g2):
        if g1 is None:
            return g2
        if g2 is None:
            return g1
        return K.axpby(K.as_nhwc(g1), K.as_nhwc(g2))

    @staticmethod
    def tangent(args, out, tan):
        t = tan(args[0])
        return t, t


class PoolFn(TFunction):
    """2x2 average pooling of a tensor that is not a ReLU output (no mask in the backward)."""

    @staticmethod
    def forward(ctx, x):
        return K.pool2_fwd(x, 0)

    @staticmethod
    def backward(ctx, dy):
        return K.pool2_bwd(K.as_nhwc(dy), 0)

    @staticmethod
    def tangent(args, out, tan):
        t = tan(args[0])
        return PoolFn.apply(t) if t is not None else None
