"""FP32-accurate launch plan (cfg.ESF.PRECISION = "fp32"): the north star's "FP32/TF32 path, rel err <= 1e-4".

The reference computes in FP32 everywhere (SlowFast/slowfast/models/resnet_helper.py:182-240, wdf_attention_helper.py:
42-53).  The tensor cores take 16-bit operands, so this plan carries every GEMM operand as a PAIR of FP16 numbers
x = hi + lo (22 mantissa bits) and evaluates x.w = x_hi.w_hi + x_lo.w_hi + x_hi.w_lo with FP32 accumulation -- on the
SAME tcgen05 implicit-GEMM kernel as the 16-bit plan, with no kernel change:

  * an activation is an `Act32`: the FP32 tensor (what the element-wise kernels read: residuals, pooling, ECA, head)
    plus a channels-last FP16 buffer of three planes [hi | lo | hi] (what the GEMM reads as 3 C input channels);
  * a folded weight becomes [w_hi | w_hi | w_lo] along its input-channel axis, rows pre-scaled by a power of two so that
    w_lo is a normal FP16 number;
  * every conv is `igemm (FP32 out, raw accumulators) -> esf_p32_post (un-scale + bias + residual + activation -> FP32
    tensor + the three planes)`.
Concat stays free: a producer writes its channel slice of the FP32 buffer and of each plane.  The position attention
runs in FP32 on the CUDA cores (esf_p32_attention, flash style): the tcgen05 attention kernel rounds P and V to FP16,
which alone costs 5e-4 on the probabilities (measured).

Scope: every classification model of nets_resnet.py -- the two-stream models and the single-pathway ResNet (C2D / I3D /
Slow), grouped bottlenecks, Non-local blocks (also with temporal groups), any attention head dim and the
fully-convolutional test head.  Depthwise convolutions (the efficient backbones) and the detection head are not covered.
About 3x the tensor-core work and ~5x the activation bytes of the FP16 plan: an accuracy mode, benchmarked beside it.
"""
import torch

from . import runtime as rt
from .engine import Plan, block_diagonal, fold_conv_bn, fold_time_groups, stem_route


class Act32:
    """One activation of the FP32-accurate plan: `f32` (B,T,H,W,C) FP32 view and the [hi|lo|hi] FP16 buffer `x3`
    (B,T,H,W,3*plane) it is mirrored into at channel offset `c0` of every plane.  Supports the `[..., a:b]` channel
    slicing the model code uses for concat buffers."""

    def __init__(self, f32, x3, plane, c0, c_total, weight_order=False, has_f32=True, has_planes=True):
        self.f32, self.x3, self.plane, self.c0, self.c_total = f32, x3, plane, c0, c_total
        self.weight_order = weight_order    # planes [hi | hi | lo]: the tensor is the WEIGHT operand of a per-clip GEMM
        # an intermediate that is only ever a GEMM operand keeps no FP32 copy (f32 is a shape-only meta tensor), one that
        # is only ever a residual keeps no planes (PrecisePlan.act(role=...)): 4 resp. 6 bytes per element the post-pass
        # does not write
        self.has_f32, self.has_planes = has_f32, has_planes

    @property
    def shape(self):
        return self.f32.shape

    @property
    def whole(self):
        return self.c0 == 0 and self.f32.shape[4] == self.c_total

    @property
    def hi(self):
        return self.x3[..., self.c0:self.c0 + self.f32.shape[4]]

    def __getitem__(self, idx):
        assert isinstance(idx, tuple) and len(idx) == 2 and idx[0] is Ellipsis and isinstance(idx[1], slice)
        start, stop, step = idx[1].indices(self.f32.shape[4])
        assert step == 1
        return Act32(self.f32[..., start:stop], self.x3, self.plane, self.c0 + start, self.c_total, self.weight_order,
                     self.has_f32, self.has_planes)

    def need_f32(self, who):
        assert self.has_f32, "%s reads the FP32 copy of an activation that was planned without one" % who
        return self.f32

    def fold_time_groups(self, group):
        """engine.fold_time_groups of the FP32 tensor and of the planes."""
        return Act32(fold_time_groups(self.f32, group), fold_time_groups(self.x3, group) if self.has_planes else None,
                     self.plane, self.c0, self.c_total, self.weight_order, self.has_f32, self.has_planes)


def split_weight_rows(w):
    """Folded FP64 weight (Cout, Cin, kT, kH, kW) -> (w_hi, w_lo, inv_scale): rows scaled by 2^k so that max|row| lies in
    [1024, 2048) -- w_lo = fp16(w s - w_hi) ~ 2^-12 of that stays far above the FP16 subnormals -- then split into two
    FP16-representable parts; inv_scale[n] = 2^-k undoes the scaling in the FP32 post-pass (exact)."""
    cout = w.shape[0]
    amax = w.reshape(cout, -1).abs().amax(dim=1).clamp_min(1e-30)
    k = torch.floor(torch.log2(1024.0 / amax))
    s = torch.pow(torch.tensor(2.0, dtype=torch.float64), k)
    ws = w * s.view(-1, 1, 1, 1, 1)
    hi = ws.to(torch.float16).to(torch.float64)
    lo = (ws - hi).to(torch.float16).to(torch.float64)
    return hi, lo, 1.0 / s


def split_operand_weight(w, plane, c0):
    """Folded FP64 weight (Cout, Cin, kT, kH, kW) of a conv that reads channels [c0, c0 + Cin) of every [hi|lo|hi] plane
    of a buffer of plane width `plane` -> the [w_hi | w_hi | w_lo] weight over the whole 3 * plane channels (zero
    elsewhere) and the inv_scale of split_weight_rows."""
    cout, cin = w.shape[:2]
    hi, lo, inv_scale = split_weight_rows(w)
    w3 = torch.zeros((cout, 3 * plane) + tuple(w.shape[2:]), dtype=torch.float64)
    w3[:, c0:c0 + cin] = hi
    w3[:, plane + c0:plane + c0 + cin] = hi
    w3[:, 2 * plane + c0:2 * plane + c0 + cin] = lo
    return w3, inv_scale


class PrecisePlan(Plan):
    wfold = False    # the banded thin-layer GEMM has no FP32 output; every conv is the plain igemm

    def __init__(self, device, precision="fp32", family=None):
        super().__init__(device, precision="fp32", family=family)
        self.precise = True

    # ---------------------------------------------------------------- memory
    def act(self, B, T, H, W, C, name=None, dtype=None, role=None):
        """role "operand": the tensor is only read as a GEMM operand (planes, no FP32 copy); "residual": only as a
        residual (FP32, no planes); None: both."""
        if dtype is not None and dtype != self.adt:
            return super().act(B, T, H, W, C, name=name, dtype=dtype)
        assert role in (None, "operand", "residual") and not (name and role)
        plane = (C + 7) // 8 * 8
        has_f32, has_planes = role != "operand", role != "residual"
        f32 = (self.alloc((B, T, H, W, C), torch.float32) if has_f32 else
               torch.empty((B, T, H, W, C), dtype=torch.float32, device="meta"))
        # zero-filled: the row padding [C, plane) of every plane meets zero weights in the GEMM and must stay finite
        x3 = self.alloc((B, T, H, W, 3 * plane), torch.float16, zero=True) if has_planes else None
        if name:
            self.buffers[name] = f32
        return Act32(f32, x3, plane, 0, C, has_f32=has_f32, has_planes=has_planes)

    def _post(self, acc, y, scale=None, bias=None, res=None, act=rt.ACT_NONE, label=""):
        """esf_p32_post: y.f32 = act(acc * scale + bias + res) and its three FP16 planes (y: Act32 or FP32 tensor)."""
        if isinstance(res, Act32):
            res = res.need_f32("a residual add")
        if isinstance(y, Act32):
            in_place = y.has_f32 and y.f32.data_ptr() == acc.data_ptr() and scale is None and bias is None and \
                res is None and act == rt.ACT_NONE
            y32 = None if (in_place or not y.has_f32) else y.f32
            y3, plane, worder = (y.hi if y.has_planes else None), y.plane, int(y.weight_order)
        else:
            y32, y3, plane, worder = y, None, 0, 0
        self._launch("esf_p32_post", acc, scale, bias, res, act, y32, y3, plane, worder, kind="p32_post", label=label,
                     nbytes=acc.numel() * (4 + (4 if res is not None else 0) + (4 if y32 is not None else 0) +
                                           (6 if y3 is not None else 0)))

    # ---------------------------------------------------------------- ops
    def conv(self, x, y, w_folded, bias, stride=(1, 1, 1), padding=(0, 0, 0), dilation=(1, 1, 1), groups=1,
             act=rt.ACT_NONE, res=None, out_dtype=None):
        """Conv3d + folded BN (+ residual) + activation at ~FP32 accuracy: igemm over the [hi|lo|hi] planes with the
        [w_hi|w_hi|w_lo] weight (raw FP32 accumulators), then the FP32 post-pass.

        groups > 1 (RESNET.NUM_GROUPS, resnet_helper.py:196-205) runs as ONE dense split GEMM over a block-diagonal
        weight: `groups` times the MACs of the layer, spent on structural zeros, for a single launch on the same kernel.
        Depthwise convolutions (one input channel per group: the efficient backbones) are not covered."""
        assert isinstance(x, Act32) and not x.weight_order
        assert x.has_planes, "a convolution reads the planes of an activation that was planned without them"
        if groups != 1:
            if w_folded.shape[1] == 1:
                raise NotImplementedError("depthwise convolutions are not part of the FP32-accurate plan (efficient "
                                          "backbones); run them with 'fp16' / 'bf16'")
            w_folded = block_diagonal(w_folded, groups)
        w = w_folded.to(torch.float64)
        cout, cin = w.shape[:2]
        assert cin == x.shape[4]
        # the GEMM reads the WHOLE parent buffer: a channel slice (x_s of a concat buffer) gets zero weights elsewhere
        w3, inv_scale = self.once(split_operand_weight, w, x.plane, x.c0)
        yshape = tuple(y.shape)
        acc = self.scratch(yshape, torch.float32)
        zero = torch.zeros(cout, dtype=torch.float64)
        self.conv_igemm(x.x3, acc, w3, zero, stride, padding, dilation, rt.ACT_NONE, None)
        self.meta[-1]["label"] += " x3"
        self._post(acc, y, self.tensor(inv_scale), self.tensor(bias), res, act)

    def stem(self, x_nc, y, w_folded, bias, stride, padding, act=rt.ACT_RELU):
        """Stem conv + folded BN + ReLU at FP32 accuracy.  Tensor-core GEMM (the kernel stem_route picks) when the
        geometry allows: the clip is packed twice (hi and lo halves), the band weight is split like any other weight, and
        the three products hi.hi, lo.hi, hi.lo are three launches of the same GEMM with FP32 outputs (its tap table
        cannot hold 3 x kT x kH taps), summed, un-scaled, biased and activated by esf_p32_post3.  Else the FP32
        CUDA-core stem."""
        route = stem_route(x_nc.shape, w_folded.shape, stride, padding)
        if route is None or not y.f32.is_contiguous():
            self.stem_conv(x_nc, y.f32, w_folded, bias, stride, padding, act)
            return self._post(y.f32, y, label="split")
        pitch, lpad, twb = route
        B, Cin, T, H, W = x_nc.shape
        cout = w_folded.shape[0]
        hi, lo, inv_scale = self.once(split_weight_rows, w_folded.to(torch.float64))
        zero = torch.zeros(cout, dtype=torch.float64)

        def pack(fn_name, xp):      # reads the caller's clip: its pointer is looked up at launch time
            return lambda s: self._call(fn_name, self._in_ptr(x_nc), B, Cin, T, H, W, pitch, lpad, rt.F16, xp.data_ptr(), s)

        xps, accs = [], []
        for fn_name, part in (("esf_stem_pack", "hi"), ("esf_stem_pack_lo", "lo")):
            xp = self.alloc((B, T, H, pitch), torch.float16)
            self._add(pack(fn_name, xp), "stem_pack", part, nbytes=self._nbytes(x_nc, xp), eager=True)
            xps.append(xp)
        for name, xp, wpart in (("hi.hi", xps[0], hi), ("lo.hi", xps[1], hi), ("hi.lo", xps[0], lo)):
            acc = self.alloc(tuple(y.shape), torch.float32)
            self._stem_gemm_op(xp, x_nc.shape, acc, wpart, zero, stride, padding, rt.ACT_NONE, pitch, twb, name)
            accs.append(acc)
        self._launch("esf_p32_post3", *accs, self.tensor(inv_scale), self.tensor(bias), act, y.f32, y.hi, y.plane,
                     kind="p32_post", label="stem sum", nbytes=accs[0].numel() * (12 + 4 + 6))

    def pool(self, x, y, kernel, stride, padding, is_avg=False, act=rt.ACT_NONE):
        assert act == rt.ACT_NONE
        self._pool32(x.f32, y.f32, kernel, stride, padding, is_avg)
        self._post(y.f32, y, label="split")

    def _pool32(self, x, y, kernel, stride, padding, is_avg):
        """esf_p32_pool3d between two FP32 tensors."""
        self._launch("esf_p32_pool3d", x, y, *kernel, *stride, *padding, int(is_avg), kind="p32_pool",
                     label="%s C=%d" % (tuple(kernel), x.shape[4]), nbytes=self._nbytes(x, y))

    def eca_fuse(self, x_fast, y_slice, alpha, eca_weight, bn):
        self._eca_fuse("esf_p32_eca_fuse", "esf_p32_eca_scratch_floats", "p32_eca_fuse", x_fast.f32, y_slice.f32, alpha,
                       eca_weight, bn)
        self._post(y_slice.f32, y_slice, label="split")

    def position_attention(self, x_slow, y_slice, alpha, w_down, att, bn):
        """Same composition as Plan.position_attention; the projection GEMM runs on the split operands, the fused
        attention kernel writes FP32 into the concat slice, which is then split into planes.  Any head dim: the split
        tensor-core kernel up to d = 64 (its geometry pads d like the 16-bit kernel's), FP32 flash attention on the CUDA
        cores up to 128, the generic FP32 CUDA-core kernel of the 16-bit plan above."""
        proj, geo = self._attention_operands(x_slow, alpha, w_down, att, bn)
        B, T, H, W, d = geo[:5]
        N = T * H * W
        y = y_slice.f32
        if d <= 64:
            # tensor cores at FP32 accuracy: the logits are hi/lo split already; P and V become FP16 pairs too
            # (esf_attn_tc_create_split: O += P_hi V_hi + P_lo V_hi + P_hi V_lo, row sums in FP32 registers)
            nbytes = self._size("esf_attn_tc_pack_bytes", B, N, d)
            nlo = self._size("esf_attn_tc_vlo_bytes", B, N, d)
            packed = self.alloc((nbytes,), torch.uint8, flat=True)
            vlo = self.alloc((nlo,), torch.uint8, flat=True)
            h = self._create("esf_attn_tc_create_split", packed, vlo, *geo, y)
            pack = self._bind("esf_attn_tc_pack", proj, B, N, d, rt.F16, packed)
            pack_vlo = self._bind("esf_attn_tc_pack_vlo", proj, B, N, d, vlo)
            self._add(lambda s: (pack(s), pack_vlo(s)), "attn_pack", "N=%d d=%d split" % (N, d),
                      nbytes=self._nbytes(proj) + nbytes + nlo, launches=2)
            self._launch("esf_op_launch", h, kind="attention", label="N=%d d=%d split" % (N, d),
                         flops=8.0 * B * N * N * d, exps=float(B) * N * N, nbytes=nbytes + nlo + self._nbytes(y))
        elif d <= 128:
            # d in (64, 128] has no hi/lo logit split on the tensor cores (the split Q tile does not fit in shared
            # memory): FP32 flash attention on the CUDA cores (d = 128: N = 1 568 there)
            self._launch("esf_p32_attention", proj, *geo, y, kind="p32_attention", label="N=%d d=%d" % (N, d),
                         flops=4.0 * B * N * N * d, exps=float(B) * N * N, nbytes=self._nbytes(proj, y))
        else:
            self._attention_generic(proj, geo, y)
        self._post(y, y_slice, label="split")

    def _head_pool(self, xs, feat):
        """xs: Act32 activations, or plain FP32 tensors (the pooled rows of positions_head): one esf_p32_head_pool per
        pathway into its slice of feat."""
        off = 0
        for x in xs:
            x = x.f32 if isinstance(x, Act32) else x
            self._launch("esf_p32_head_pool", x, feat, feat.shape[1], off, kind="p32_head_pool", nbytes=self._nbytes(x))
            off += x.shape[4]

    def _head_avg_pool(self, x, kernel, shape):
        """The head's AvgPool3d into a plain FP32 buffer: nothing multiplies it on the tensor cores, so it gets no
        planes (esf_p32_head_pool of its one-position rows in positions_head is a copy)."""
        y = super().act(*shape, dtype=torch.float32)
        self._pool32(x.need_f32("the head"), y, kernel, (1, 1, 1), (0, 0, 0), is_avg=True)
        return y

    def nonlocal_block(self, x, y, nln, group=1):
        """Nonlocal.forward (nonlocal_helper.py:105-148) at FP32 accuracy: theta / phi / g / out are split-operand convs;
        the two matrix products are per-clip-weight GEMMs on split operands as well -- theta and the normalised affinity
        are A operands ([hi | lo | hi] planes), the clip's phi rows and transposed g rows are the weight operands
        ([hi | hi | lo]); the affinity is materialised in FP32 and normalised by esf_p32_row_softmax.  (Not fused: an
        accuracy mode.)  NONLOCAL.GROUP > 1: the (b, t) -> (b * group, t / group) view of Plan.nonlocal_block, applied to
        the FP32 tensor and to the planes of x and y."""
        if group > 1:
            x, y = x.fold_time_groups(group), y.fold_time_groups(group)
        B, T, H, W, C = x.shape
        d = nln.dim_inner
        dp = (d + 7) // 8 * 8
        xp, softmax = self._nonlocal_keys(x, nln)
        Tp, Hp, Wp = xp.shape[1:4]
        Nq, Nk = T * H * W, Tp * Hp * Wp
        wb = self._weight_bias
        theta = self.act(B, T, H, W, d)
        self.conv(x, theta, *wb(nln.conv_theta))
        # phi rows of a clip ARE the [n][k] weight matrix of theta^T phi (k = the 3 d plane channels): allocate them
        # inside a zero-padded (B, n_pad, 3 dp) matrix and view its first Nk rows as the activation
        kc1, kch1, _, npad1 = rt.igemm_geometry(3 * dp, Nk)
        assert kc1 * kch1 == 3 * dp, "3 x dim_inner must fill whole K chunks"
        phi_rows = self.alloc((B, npad1, 3 * dp), torch.float16, zero=True)
        phi32 = self.alloc((B, Tp, Hp, Wp, d), torch.float32)
        phi_x3 = phi_rows.as_strided((B, Tp, Hp, Wp, 3 * dp), (npad1 * 3 * dp, Hp * Wp * 3 * dp, Wp * 3 * dp, 3 * dp, 1))
        phi = Act32(phi32, phi_x3, dp, 0, d, weight_order=True)
        g32 = self.alloc((B, Tp, Hp, Wp, d), torch.float32)
        g_x3 = self.alloc((B, Tp, Hp, Wp, 3 * dp), torch.float16, zero=True)
        g = Act32(g32, g_x3, dp, 0, d, weight_order=True)
        self.conv(xp, phi, *wb(nln.conv_phi))
        self.conv(xp, g, *wb(nln.conv_g))
        # affinity S = theta^T phi (FP32), one launch for the whole batch
        S = self.scratch((B, T, H, W, (Nk + 3) // 4 * 4), torch.float32)
        zero1 = self.scratch((npad1,), torch.float32, zero=True)
        self.gemm_rows(theta.x3, S[..., :Nk], phi_rows, zero1, "nl_gemm", "theta.phi x3 N=%dx%d d=%d" % (Nq, Nk, d))
        # normalise into the [hi | lo | hi] planes of the second product's A operand
        nkp = (Nk + 7) // 8 * 8
        P3 = self.scratch((B, T, H, W, 3 * nkp), torch.float16, zero=True)
        scale, mode = (float(d) ** -0.5, 0) if softmax else (1.0 / Nk, 1)
        self._launch("esf_p32_row_softmax", S, B * Nq, Nk, S.shape[4], scale, mode, P3, 3 * nkp, nkp,
                     kind="p32_nl_softmax", label=nln.instantiation, nbytes=B * Nq * Nk * 10.0, exps=float(B * Nq * Nk))
        # g^T in weight order: gT3[b][c][plane * nkp + k] = plane(g)[b, k, c], planes (hi, hi, lo)
        kc2, kch2, _, npad2 = rt.igemm_geometry(3 * nkp, d)
        kpad = kc2 * kch2
        gT3 = self.alloc((B, npad2, kpad), torch.float16, zero=True)
        for pl in range(3):
            self._launch("esf_transpose16", g_x3.data_ptr() + 2 * pl * dp, B, Nk, d, Nk * 3 * dp, 3 * dp,
                         gT3.data_ptr() + 2 * pl * nkp, npad2 * kpad, kpad, kind="nl_transpose", label="g plane %d" % pl,
                         nbytes=4.0 * B * Nk * d)
        att = self.act(B, T, H, W, d)
        acc = self.scratch((B, T, H, W, d), torch.float32)
        zero2 = self.scratch((npad2,), torch.float32, zero=True)
        self.gemm_rows(P3, acc, gT3, zero2, "nl_gemm", "p.g x3 N=%dx%d d=%d" % (Nq, Nk, d))
        self._post(acc, att, label="split")
        w, bias = self.once(fold_conv_bn, nln.conv_out.weight, nln.conv_out.bias, nln.bn)
        self.conv(att, y, w, bias, res=x)
