"""Launch-plan builder: turns a model's parameters into folded/packed device weights and an ordered list of
libesf_b200 kernel launches over pre-allocated channels-last BF16 activation buffers.

Design (B200-first, not a module-by-module translation of the reference):
  * activations are (B,T,H,W,C) BF16; every torch.cat of the reference is a channel slice of one wider buffer that
    the producers write into directly (concat is free), every eval BatchNorm3d is folded into the preceding conv,
    ReLU / residual adds live in the conv epilogue;
  * a plan is built once per input shape, captured into a CUDA graph and replayed;
  * there is no PyTorch compute on the path -- torch only owns the memory and the stream.
"""
import ctypes

import torch

from . import runtime as rt

BN_EPS_DEFAULT = 1e-5
_VIEW_P = ctypes.POINTER(rt.EsfView)


def host64(t):
    """Parameter / buffer -> FP64 tensor on the HOST.  All weight preparation (BN folding, composition of 1x1x1 convs,
    packing into the kernels' layouts) is plan-build-time work on a few MB and runs on the CPU: one D2H copy per
    parameter and one H2D copy per packed tensor, no element-wise GPU launches -- the first kernels a process launches
    are the forward path's own (the round-1 build issued > 1 000 tiny FP64 ATen kernels per plan)."""
    return t.detach().cpu().to(torch.float64)


def to_device(t, device, dtype):
    """Host tensor -> contiguous device tensor of `dtype`; the conversion happens on the host."""
    return t.detach().to(dtype).contiguous().to(device)


def bn_affine(bn):
    """Eval-mode BatchNorm as y = x * scale + shift (FP64 math on the host)."""
    var = host64(bn.running_var)
    w = host64(bn.weight) if bn.weight is not None else torch.ones_like(var)
    b = host64(bn.bias) if bn.bias is not None else torch.zeros_like(var)
    scale = w / torch.sqrt(var + bn.eps)
    shift = b - host64(bn.running_mean) * scale
    return scale, shift


def fold_conv_bn(weight, conv_bias, bn):
    """(Cout,Cin/g,kT,kH,kW) conv weight (+ optional bias) followed by eval BN -> folded FP64 weight and bias."""
    w = host64(weight)
    cout = w.shape[0]
    b = host64(conv_bias) if conv_bias is not None else torch.zeros(cout, dtype=torch.float64)
    if bn is not None:
        scale, shift = bn_affine(bn)
        w = w * scale.view(-1, 1, 1, 1, 1)
        b = b * scale + shift
    return w, b


def pack_igemm_weight(w, bias, device, dtype=torch.bfloat16):
    """Folded (Cout,Cin,kT,kH,kW) FP64 weight -> 16-bit [n_pad][taps*kchunks*kc] (tap-major, then input channel) and
    FP32 bias [n_pad], the layout esf_conv_igemm_create expects."""
    cout, cin, kt, kh, kw = w.shape
    kc, kchunks, _, n_pad = rt.igemm_geometry(cin, cout)
    cpad = kc * kchunks
    wp = torch.zeros(n_pad, kt * kh * kw, cpad, dtype=torch.float64, device=w.device)
    wp[:cout, :, :cin] = w.permute(0, 2, 3, 4, 1).reshape(cout, kt * kh * kw, cin)
    bp = torch.zeros(n_pad, dtype=torch.float64, device=w.device)
    bp[:cout] = bias
    return to_device(wp.reshape(n_pad, -1), device, dtype), to_device(bp, device, torch.float32)


STEM_WB = 8  # output columns per banded-GEMM block (csrc/esf_igemm.cu kStemWB)


def pack_stem_band(w, bias, stride_w, device, dtype=torch.bfloat16):
    """Folded (Cout,Cin,kT,kH,kW) stem weight -> band matrix BF16 [n_pad][kT*kH*64] and tiled bias FP32 [n_pad].
    Row n = i*Cout + co (i = output column inside the 8-wide block); column k = (kt*kH + kh)*64 + j where
    (w_in, c) = divmod(j, Cin) is the j-th element of the contiguous input run the block reads and kw = w_in - sW*i."""
    cout, cin, kt, kh, kw = w.shape
    N = STEM_WB * cout
    _, _, _, n_pad = rt.igemm_geometry(64, N)
    band = torch.zeros(n_pad, kt * kh, 64, dtype=torch.float64, device=w.device)
    win = ((STEM_WB - 1) * stride_w + kw) * cin
    assert win <= 64
    wt = w.permute(0, 2, 3, 4, 1).reshape(cout, kt * kh, kw, cin)          # [co][tap][kw][c]
    for i in range(STEM_WB):
        j0 = stride_w * i * cin
        band[i * cout:(i + 1) * cout, :, j0:j0 + kw * cin] = wt.reshape(cout, kt * kh, kw * cin)
    bt = torch.zeros(n_pad, dtype=torch.float64, device=w.device)
    bt[:N] = bias.repeat(STEM_WB)
    return to_device(band.reshape(n_pad, -1), device, dtype), to_device(bt, device, torch.float32)


def pack_stem_tband(w, bias, WB, stride_w, device, dtype=torch.bfloat16):
    """Folded (Cout,Cin,kT,kH,kW) stem weight -> band matrix [kT*NB][kH*64] and tiled bias FP32 [NB] of the temporal-band
    stem (esf_stem_tband_create), NB = WB*Cout.  Row n = u*NB + i*Cout + co: u is the output frame relative to the oldest
    frame an input frame touches, i.e. the weights of time tap kt = kT-1-u; i = output column inside the WB-wide block.
    Column k = kh*64 + j, (w_in, c) = divmod(j, Cin) the j-th element of the input run the block reads, kw = w_in - sW*i."""
    cout, cin, kt, kh, kw = w.shape
    NB = WB * cout
    assert ((WB - 1) * stride_w + kw) * cin <= 64
    band = torch.zeros(kt, WB, cout, kh, 64, dtype=torch.float64, device=w.device)
    wt = w.to(torch.float64).permute(2, 0, 3, 4, 1).reshape(kt, cout, kh, kw * cin)      # [kt][co][kh][(kw, c)]
    for i in range(WB):
        j0 = stride_w * i * cin
        band[:, i, :, :, j0:j0 + kw * cin] = wt.flip(0)                                   # u = kT-1-kt
    bt = bias.to(torch.float64).repeat(WB)
    return to_device(band.reshape(kt * NB, kh * 64), device, dtype), to_device(bt, device, torch.float32)


def stem_route(x_shape, w_shape, stride, padding):
    """Stem kernel for a (B,Cin,T,H,W) clip and a (Cout,Cin,kT,kH,kW) weight: None for the CUDA-core stem
    (esf_stem_conv), else (pitch, lpad, twb) -- the packed-row geometry of esf_stem_pack and the output-column block of
    the temporal-band GEMM (esf_stem_tband_create: kT > 1, time taps folded into N), twb == 0 for the banded GEMM
    (esf_stem_igemm_create)."""
    _, cin, _, _, W = x_shape
    cout, _, kt, kh, kw = w_shape
    geo = rt.stem_geometry(W, cin, kw, stride[2], padding[2]) if stride[0] == 1 else None
    if geo is None:
        return None
    pitch, lpad, _ = geo
    return pitch, lpad, rt.stem_tband_wb(W, cin, cout, kt, kh, kw, stride[2], padding[2])


def pack_wfold_band(w, bias, WB, stride_w, device, dtype=torch.bfloat16):
    """Folded (Cout,Cin,kT,kH,kW) weight of a thin layer -> band matrix [n_pad][kT*kH*kchunks*64] and tiled bias [n_pad]
    for esf_conv_wfold_create.  Row n = i*Cout + co (i = output column inside the WB-wide block); column
    k = (kt*kH + kh)*kchunks*64 + j where (w_in, c) = divmod(j, Cin) indexes the contiguous input run the block reads
    (starting at input column WB*sW*block - pW) and kw = w_in - sW*i."""
    cout, cin, kt, kh, kw = w.shape
    N = WB * cout
    _, _, _, n_pad = rt.igemm_geometry(64, N)
    win = ((WB - 1) * stride_w + kw) * cin
    kpad = -(-win // 64) * 64
    band = torch.zeros(n_pad, kt * kh, kpad, dtype=torch.float64, device=w.device)
    wt = w.permute(0, 2, 3, 4, 1).reshape(cout, kt * kh, kw * cin).to(torch.float64)   # [co][tap][(kw, c)]
    for i in range(WB):
        j0 = stride_w * i * cin
        band[i * cout:(i + 1) * cout, :, j0:j0 + kw * cin] = wt
    bt = torch.zeros(n_pad, dtype=torch.float64, device=w.device)
    bt[:N] = bias.repeat(WB)
    return to_device(band.reshape(n_pad, -1), device, dtype), to_device(bt, device, torch.float32)


def wfold_block(x, y, res, w_shape, stride, padding, dilation):
    """Width of the output-column block to fold into the GEMM's N for a thin layer, or 0 when the regular implicit
    GEMM should run.  Mirrors the argument checks of esf_conv_wfold_create."""
    cout, cin, kt, kh, kw = w_shape
    if cin > 32 or cin % 8 or stride[0] != 1 or tuple(dilation) != (1, 1, 1):
        return 0
    if x.stride(3) != cin or x.stride(4) != 1:
        return 0
    Wo = y.shape[3]
    sliced = y.stride(3) != cout or (res is not None and res.stride(3) != cout)
    best, best_key = 0, None
    for wb in range(1, 33):
        N = wb * cout
        win = ((wb - 1) * stride[2] + kw) * cin
        if Wo % wb or N > 256 or win > 128:
            continue
        if sliced and (N & (N - 1) or (64 % cout if cout < 64 else cout % 64)):
            continue
        key = (N, -((win + 63) // 64))      # widest MMA first, then fewest K chunks
        if best_key is None or key > best_key:
            best, best_key = wb, key
    return best if best >= 2 else 0     # a block of one column is the plain implicit GEMM


def attention_projection(w_down, att):
    """The slow->fast fuse's 1x1x1 C->d conv composed with SpatialAttention's q/k/v 1x1x1 convs
    (wdf_attention_helper.py:33-54): one FP64 (4d, C, 1, 1, 1) weight and (4d,) bias whose output rows are
    [x_d | q | k | v], and the head dim d."""
    wd = host64(w_down).reshape(w_down.shape[0], -1)                      # (d, C)
    d, C = wd.shape
    mats, biases = [wd], [torch.zeros(d, dtype=torch.float64)]
    for conv in (att.query_conv, att.key_conv, att.value_conv):
        wc = host64(conv.weight).reshape(conv.weight.shape[0], d)
        bc = host64(conv.bias)
        if wc.shape[0] < d:
            # SpatialAttention(reduction > 1) (wdf_attention_helper.py:17-26): query / key have d / reduction
            # channels.  Zero rows up to d leave every logit q.k unchanged and keep the kernels' one head dim.
            # (No cfg key reaches this: every call site of the reference hard-codes reduction = 1.)
            assert conv is not att.value_conv, "value_conv keeps all channels"
            pad = d - wc.shape[0]
            wc = torch.cat([wc, torch.zeros(pad, d, dtype=wc.dtype)], 0)
            bc = torch.cat([bc, torch.zeros(pad, dtype=bc.dtype)], 0)
        mats.append(wc @ wd)
        biases.append(bc)
    return torch.cat(mats, 0).reshape(4 * d, C, 1, 1, 1), torch.cat(biases, 0), d


def block_diagonal(w, groups):
    """Grouped (Cout, Cin/groups, kT, kH, kW) weight -> the dense (Cout, Cin, kT, kH, kW) weight of the same convolution:
    group g's block at output rows g*Cout/groups and input channels g*Cin/groups, zeros elsewhere."""
    cout, cin_g = w.shape[:2]
    cout_g = cout // groups
    wd = torch.zeros((cout, cin_g * groups) + tuple(w.shape[2:]), dtype=w.dtype, device=w.device)
    for g in range(groups):
        wd[g * cout_g:(g + 1) * cout_g, g * cin_g:(g + 1) * cin_g] = w[g * cout_g:(g + 1) * cout_g]
    return wd


def fold_time_groups(t, group):
    """(B, T, H, W, C) view -> (B * group, T / group, H, W, C): the temporal group folding of ResStage.forward
    (resnet_helper.py:541-560) for the Non-local blocks, a pure view in channels-last memory."""
    B, T, H, W, C = t.shape
    assert T % group == 0 and t.stride(0) == T * t.stride(1)
    return t.as_strided((B * group, T // group, H, W, C),
                        (t.stride(1) * (T // group), t.stride(1), t.stride(2), t.stride(3), 1), t.storage_offset())


def conv_weight_bias(conv):
    """A conv's weight and bias as FP64 host tensors."""
    return host64(conv.weight), host64(conv.bias)


def nonlocal_offset(nln, d, npad_d):
    """The per-channel offset mu of Plan.nonlocal_block's last product: least-squares solution of
    conv_out.weight mu = bn.running_mean - conv_out.bias.  Returns mu as FP64 (the FP32-rounded value actually
    subtracted) and the FP32 bias [npad_d] of that product, -mu padded with zeros."""
    C = nln.conv_out.weight.shape[0]
    w_out = host64(nln.conv_out.weight).reshape(C, d)
    rhs = (host64(nln.bn.running_mean) - host64(nln.conv_out.bias)).reshape(C, 1)
    mu = torch.linalg.lstsq(w_out, rhs).solution.reshape(d)
    bias2 = torch.zeros(npad_d, dtype=torch.float32)
    bias2[:d] = (-mu).to(torch.float32)
    return -bias2[:d].to(torch.float64), bias2


def _shape_only(x):
    """Host tensors of a weight-preparation result as meta tensors of the same shape and dtype (device tensors and
    other values as they are)."""
    if isinstance(x, tuple):
        return tuple(_shape_only(v) for v in x)
    if isinstance(x, torch.Tensor) and x.device.type == "cpu":
        return torch.empty_like(x, device="meta")
    return x


class Family:
    """What the plans of one per-clip input shape share when cfg.ESF.MAX_BATCH is set.  The CAPACITY plan, compiled at
    the largest batch, records every device tensor it allocates (Plan.alloc) and every result of its host weight
    preparation (Plan.once), in call order.  A VARIANT, compiled later at a smaller batch, replays both lists: it
    allocates no activation arena and folds no weights.  It keeps its own op handles, metadata and CUDA graph.  The
    family also holds the run-time state of its plans (Plan.shared): frame-route tables and the detection rows."""

    def __init__(self):
        self.allocs = []      # (tensor, zero, flat) of every Plan.alloc of the capacity plan
        self.memo = []        # (function name, result) of every Plan.once of the capacity plan
        self.built = False    # the capacity plan is compiled: every later plan of the family is a variant
        self.roi_feat = self.roi_out = None


def head_fc_launches(B, cin, K, act):
    """Kernel launches of one esf_head_fc call: the tiled kernel (B >= 8, or rows too long for one block) applies the
    class softmax in a second, tiny kernel."""
    tiled = B >= 8 or (cin + K) * 4 > 48 * 1024
    return 2 if (tiled and act == rt.HEAD_SOFTMAX) else 1


class Plan:
    """Ordered kernel launches + every tensor they touch.  `eager` ops read the caller's input tensors and are
    launched on every forward; `graph` ops only touch plan-owned memory and are replayed from one CUDA graph."""

    wfold = True     # thin layers (C_in <= 32) as W-folded banded GEMMs

    def __init__(self, device, precision="bf16", family=None):
        self.device = device
        self.family = family
        self.variant = family is not None and family.built
        self.variants = {}    # capacity plan of a family: batch rows -> variant plan
        self._n_alloc = self._n_memo = 0     # variant: position in the family's lists
        self.precision = precision
        self.adt = rt.TORCH_DTYPE[precision]      # 16-bit storage format of activations / tensor-core operands
        self.a16 = rt.dtype_code(self.adt)
        self.keep = []        # tensors / ctypes structs that must outlive the plan
        self.ops = []         # callables taking a stream pointer
        self.eager = []       # per op: launched outside the CUDA graph (reads a caller-provided input tensor)
        self.input_override = {}   # plan-owned input data_ptr -> data_ptr of the caller's tensor for this run
        self.stem_routes = {}      # plan-owned input data_ptr -> (packed stem rows, pitch, lpad) of a banded stem
        self.gather = {}           # plan-owned input data_ptr -> (source clip ptr, its frame count, device int32 frame
                                   # index ptr): this run packs the pathway out of ANOTHER clip's frames (slow from fast)
        self.padded = {}           # data_ptr of a channel-padded activation -> (logical C, padded C)
        self.handles = []     # esf_op* to destroy
        self.graph = None
        self.out = None
        self.launches_per_run = 0
        self.buffers = {}     # name -> activation tensor (for tests / debugging)
        self.meta = []        # one dict per op: kind, label, algorithmic flops / bytes / exps, launches
        self._scratch = {}    # (shape, dtype, zero) -> tensor shared by the ops of this plan (scratch())

    # ---------------------------------------------------------------- memory
    @property
    def shared(self):
        """Holder of the run-time state (frame tables, detection rows) of this plan: its family, else the plan."""
        return self.family if self.family is not None else self

    def alloc(self, shape, dtype, zero=False, flat=False):
        """Every device tensor a plan allocates while it is compiled comes from here (zero-filled with `zero`).  A
        variant of a Family allocates nothing: its i-th call resolves to the capacity plan's i-th tensor -- that tensor
        itself when the shape does not depend on the batch, its first rows when only dim 0 does (zero-filled state thus
        keeps its per-clip layout), and a prefix of it for `flat` scratch: 1-D, written before it is read, of a size
        that grows with the batch.  Any other mismatch is an error."""
        shape = tuple(int(n) for n in shape)
        assert not (zero and flat), "flat scratch is written before it is read"
        if not self.variant:
            t = (torch.zeros if zero else torch.empty)(shape, dtype=dtype, device=self.device)
            self.keep.append(t)
            if self.family is not None:
                self.family.allocs.append((t, bool(zero), bool(flat)))
            return t
        allocs = self.family.allocs
        assert self._n_alloc < len(allocs), "a variant allocates more tensors than its capacity plan"
        t, z, f = allocs[self._n_alloc]
        self._n_alloc += 1
        same = t.dtype == dtype and z == bool(zero) and f == bool(flat) and len(shape) == t.dim()
        if same and shape == tuple(t.shape):
            return t
        if same and (t.dim() > 1 or flat) and shape[1:] == tuple(t.shape[1:]) and shape[0] <= t.shape[0]:
            return t[:shape[0]]
        raise AssertionError("allocation %d of a variant, %s %s (zero=%s, flat=%s), does not fit the capacity plan's "
                             "%s %s (zero=%s, flat=%s)" % (self._n_alloc - 1, shape, dtype, zero, flat,
                                                           tuple(t.shape), t.dtype, z, f))

    def once(self, fn, *args):
        """fn(*args), for host-side weight preparation (folding, packing, uploads).  A variant of a Family does not run
        it: it gets the capacity plan's result of the same call, by call order -- device tensors themselves, host
        tensors as meta tensors of their shape (a variant's host code reads only the shapes of folded weights)."""
        if not self.variant:
            out = fn(*args)
            if self.family is not None:
                self.family.memo.append((fn.__name__, _shape_only(out)))
            return out
        memo = self.family.memo
        assert self._n_memo < len(memo), "a variant prepares more weights than its capacity plan"
        name, out = memo[self._n_memo]
        self._n_memo += 1
        assert name == fn.__name__, "weight preparation %d: the variant calls %s, the capacity plan called %s" % (
            self._n_memo - 1, fn.__name__, name)
        return out

    def end_compile(self):
        """A family's plan is compiled: the capacity plan's lists are complete, a variant has used all of them."""
        if self.variant:
            assert (self._n_alloc, self._n_memo) == (len(self.family.allocs), len(self.family.memo)), \
                "a variant made %d allocations and %d weight preparations, its capacity plan %d and %d" % (
                    self._n_alloc, self._n_memo, len(self.family.allocs), len(self.family.memo))
        elif self.family is not None:
            self.family.built = True

    def act(self, B, T, H, W, C, name=None, dtype=None, role=None):
        """role: a hint for the FP32-accurate plan (engine_fp32.PrecisePlan.act); 16-bit activations have one form."""
        dtype = dtype or self.adt
        # 16-bit activations with C >= 8 get a channel pitch that is a multiple of 8 elements (16 bytes), so that every
        # buffer -- also with C = 27, 36, 180, 540 ... of the efficient backbones -- is addressable by TMA and by
        # 16-byte vector accesses; the logical tensor is the [..., :C] view
        Cp = C if (dtype != self.adt or C < 8) else (C + 7) // 8 * 8
        t = self.alloc((B, T, H, W, Cp), dtype)
        if Cp != C:
            self.padded[t.data_ptr()] = (C, Cp)     # channels [C, Cp) of every row are padding owned by this tensor
            t = t[..., :C]
        if name:
            self.buffers[name] = t
        return t

    def arena_bytes(self):
        """Device bytes this plan keeps alive (activations, packed weights, scratch, static inputs)."""
        seen, total = set(), 0
        for t in list(self.keep) + list(getattr(self, "inputs", [])):
            if isinstance(t, torch.Tensor) and t.device.type == "cuda":
                st = t.untyped_storage()
                if st.data_ptr() not in seen:
                    seen.add(st.data_ptr())
                    total += st.nbytes()
        return total

    def tensor(self, t, dtype=torch.float32):
        """Plan-lifetime device copy of a (small) parameter-derived tensor; host tensors are converted on the host."""
        return self.once(self._upload, t, dtype)

    def _upload(self, t, dtype):
        if t.device.type == "cpu":
            t = to_device(t, self.device, dtype)
        else:
            t = t.detach().to(device=self.device, dtype=dtype).contiguous()
        self.keep.append(t)
        return t

    def _add(self, fn, kind, label="", flops=0, nbytes=0, exps=0, launches=1, eager=False):
        """`eager` ops read the caller's input tensors (their source pointer can change per call): they stay outside
        the CUDA graph and are launched on every run, ahead of the graph replay."""
        self.ops.append(fn)
        self.eager.append(bool(eager))
        self.meta.append(dict(kind=kind, label=label, flops=float(flops), bytes=float(nbytes), exps=float(exps),
                              launches=launches))
        self.launches_per_run += launches

    def _bind(self, fn_name, *args):
        """The library function `fn_name` with every argument but the last (the stream, or the esf_op** of a create
        call) converted now, by the function's argtypes: a tensor for an esf_view* becomes a pointer to its view (None:
        the null view), a tensor for a void* its data pointer.  A launch replays these pointers for the plan's lifetime,
        so every converted tensor and view is kept.  Returns the checked call taking that last argument."""
        f = getattr(rt.lib(), fn_name)
        assert len(args) == len(f.argtypes) - 1, fn_name
        frozen = []
        for a, t in zip(args, f.argtypes):
            if t is _VIEW_P:
                v = rt.view(a) if a is not None else rt.null_view()
                self.keep += [a, v]
                a = ctypes.byref(v)
            elif t is ctypes.c_void_p and isinstance(a, torch.Tensor):
                self.keep.append(a)
                a = a.data_ptr()
            frozen.append(a)
        return lambda s: rt.check(f(*frozen, s), fn_name)

    def _launch(self, fn_name, *args, kind, label="", flops=0, nbytes=0, exps=0, launches=1, eager=False):
        """Record one launch of `fn_name` (arguments as _bind converts them) as an op of the plan."""
        self._add(self._bind(fn_name, *args), kind, label, flops, nbytes, exps, launches, eager)

    def _create(self, fn_name, *args):
        """Plan an esf_op with the create function `fn_name` (arguments as _bind converts them); returns its handle, which
        the plan destroys."""
        h = ctypes.c_void_p()
        self._bind(fn_name, *args)(ctypes.byref(h))
        self.handles.append(h)
        return h

    @staticmethod
    def _call(fn_name, *args):
        """Checked call of `fn_name` with arguments read at launch time (the ops that read the caller's clip)."""
        rt.check(getattr(rt.lib(), fn_name)(*args), fn_name)

    @staticmethod
    def _size(fn_name, *args):
        """A host-side size query of the library (esf_*_bytes, esf_*_scratch_floats); a negative result is its error."""
        n = int(getattr(rt.lib(), fn_name)(*args))
        rt.check(min(n, 0), fn_name)
        return n

    def _conv_desc(self, x, y, res, w, bias, ksize, stride=(1, 1, 1), padding=(0, 0, 0), dilation=(1, 1, 1), groups=1,
                   act=rt.ACT_NONE):
        """esf_conv_desc* of a convolution into `y` (output format: y's dtype); the descriptor and its tensors are kept."""
        d = rt.EsfConvDesc(rt.view(x), rt.view(y), rt.view(res) if res is not None else rt.null_view(), w.data_ptr(),
                           bias.data_ptr(), *ksize, *stride, *padding, *dilation, groups, act, rt.dtype_code(y))
        self.keep += [d, x, y, res, w, bias]
        return ctypes.byref(d)

    def _head_fc(self, feat, w, b, act, out, out_stride=None, kind="head_fc", **meta):
        """esf_head_fc: out = act(feat @ w^T + b) on FP32 rows (feat (B, Cin), w (K, Cin), out rows of stride
        out_stride, default K)."""
        (B, cin), K = feat.shape, w.shape[0]
        self._launch("esf_head_fc", feat, B, cin, cin, w, b, K, act, out, out_stride or K, kind=kind,
                     launches=head_fc_launches(B, cin, K, act), **meta)

    @staticmethod
    def _nbytes(*tensors):
        return sum(t.numel() * t.element_size() for t in tensors if t is not None)

    # ---------------------------------------------------------------- ops
    def conv_igemm(self, x, y, w_folded, bias, stride=(1, 1, 1), padding=(0, 0, 0), dilation=(1, 1, 1), act=rt.ACT_NONE,
                   res=None, out_dtype=None):
        wp, bp = self.once(pack_igemm_weight, w_folded, bias, self.device, self.adt)
        kt, kh, kw = w_folded.shape[2:]
        h = self._create("esf_conv_igemm_create",
                         self._conv_desc(x, y, res, wp, bp, (kt, kh, kw), stride, padding, dilation, 1, act))
        cout, cin = w_folded.shape[:2]
        m = y.shape[0] * y.shape[1] * y.shape[2] * y.shape[3]
        self._launch("esf_op_launch", h, kind="conv_igemm",
                     label="%dx%dx%d s%s %d->%d @%s" % (kt, kh, kw, "".join(map(str, stride)), cin, cout,
                                                        tuple(y.shape[1:4])),
                     flops=2.0 * m * cout * cin * kt * kh * kw, nbytes=self._nbytes(x, y, res) + wp.numel() * 2)

    def gemm_rows(self, x, y, w_rows, bias, kind, label):
        """y[b, pos, n] = sum_c x[b, pos, c] * w_rows[b, n, c] + bias[n] on the implicit-GEMM kernel with one
        DEVICE-RESIDENT weight matrix per clip, in the kernel's own layout ([B][n_pad][kchunks * kc] 16-bit rows, FP32
        bias [n_pad]) -- used where the "weights" are activations of the same clip (Non-local block)."""
        cin, cout = x.shape[4], y.shape[4]
        kc, kchunks, _, n_pad = rt.igemm_geometry(cin, cout)
        assert tuple(w_rows.shape) == (x.shape[0], n_pad, kc * kchunks) and w_rows.is_contiguous()
        assert w_rows.dtype == self.adt and bias.numel() == n_pad and bias.dtype == torch.float32
        h = self._create("esf_gemm_clip_weights_create", self._conv_desc(x, y, None, w_rows, bias, (1, 1, 1)))
        m = y.shape[0] * y.shape[1] * y.shape[2] * y.shape[3]
        self._launch("esf_op_launch", h, kind=kind, label=label, flops=2.0 * m * cout * cin,
                     nbytes=self._nbytes(x, y) + x.shape[0] * cout * cin * 2)

    def scratch(self, shape, dtype, zero=False, flat=False):
        """Plan-lifetime scratch tensor shared by every op that asks for the same (shape, dtype): the launches of a
        plan are serialised on one stream, so the Non-local blocks of a model reuse one affinity matrix.  `zero`,
        `flat`: as in alloc."""
        key = (tuple(shape), dtype, bool(zero), bool(flat))
        if key not in self._scratch:
            self._scratch[key] = self.alloc(shape, dtype, zero, flat)
        return self._scratch[key]

    def _weight_bias(self, conv):
        return self.once(conv_weight_bias, conv)

    def _nonlocal_keys(self, x, nln):
        """Key side of a Non-local block on the (group-folded) input x: x max-pooled by nln.pool_size when nln.use_pool,
        else x itself, and whether the instantiation is "softmax" (else "dot_product")."""
        softmax = nln.instantiation == "softmax"
        if not softmax and nln.instantiation != "dot_product":
            raise NotImplementedError("Unknown norm type {}".format(nln.instantiation))
        if not nln.use_pool:
            return x, softmax
        B, T, H, W, C = x.shape
        ps = tuple(int(v) for v in nln.pool_size)
        xp = self.act(B, (T - ps[0]) // ps[0] + 1, (H - ps[1]) // ps[1] + 1, (W - ps[2]) // ps[2] + 1, C)
        self.pool(x, xp, ps, ps, (0, 0, 0))
        return xp, softmax

    def nonlocal_block(self, x, y, nln, group=1):
        """Nonlocal.forward (nonlocal_helper.py:105-148) + the temporal group folding of ResStage.forward
        (resnet_helper.py:541-560): y = x + bn(conv_out(normalise(theta^T phi) g^T)).

        theta / phi / g / out are ordinary implicit GEMMs (bias in the epilogue; BN folded into conv_out, the residual
        add in its epilogue).  The two matrix products are implicit GEMMs as well (esf_gemm_clip_weights_create: one
        launch for the whole batch, the weight tile of an M tile is selected by its clip), whose weight operand is
        the clip's own phi rows ([N_keys][d], exactly the kernel's [n][k] layout) and g^T rows
        ([d][N_keys], written by esf_transpose16); the affinity matrix is materialised once in FP32, normalised by
        esf_row_softmax (softmax with d^-0.5, or the 1/N_keys of "dot_product") into the 16-bit A operand of the
        second product."""
        if group > 1:
            x, y = fold_time_groups(x, group), fold_time_groups(y, group)
        B, T, H, W, C = x.shape
        d = nln.dim_inner
        xp, softmax = self._nonlocal_keys(x, nln)
        Tp, Hp, Wp = xp.shape[1:4]
        Nq, Nk = T * H * W, Tp * Hp * Wp
        wb = self._weight_bias
        # Precision: with near-uniform attention the block output is a large per-channel constant plus a small
        # variation, and the BN behind conv_out removes the constant -- 16-bit rounding of `att` would then be
        # amplified by |mean| / std.  conv_out is linear, so a per-channel offset mu can be subtracted in the FP32
        # epilogue of the last product (its bias) and added back through conv_out's bias: W (att - mu) + (W mu + b).
        # mu = least-squares solution of W mu = running_mean - b, the att-space mean the BN statistics imply.
        _, _, _, npad_d = rt.igemm_geometry(Nk if softmax else d, d)
        mu, bias2_h = self.once(nonlocal_offset, nln, d, npad_d)
        bias2 = self.tensor(bias2_h)
        att = self.act(B, T, H, W, d)

        def transposed(t, name):
            """(B, Tp, Hp, Wp, d) rows -> [B][n_pad][k_pad] = t^T per clip, zero padded: the [n][k] weight layout of a
            GEMM that contracts over the keys."""
            kc, kch, _, npad = rt.igemm_geometry(Nk, d)
            kpad = kc * kch
            tT = self.alloc((B, npad, kpad), self.adt, zero=True)
            self._launch("esf_transpose16", t, B, Nk, d, t.stride(0), t.stride(3), tT, npad * kpad, kpad,
                         kind="nl_transpose", label=name, nbytes=2 * self._nbytes(t))
            return tT

        if softmax:
            # phi rows of a clip = the [n][k] weight matrix of theta^T phi: rows padded to the GEMM's n_pad
            kc1, kch1, _, npad1 = rt.igemm_geometry(d, Nk)
            assert kc1 * kch1 == d, "dim_inner must fill whole K chunks"
            theta = self.act(B, T, H, W, d)
            self.conv(x, theta, *wb(nln.conv_theta))
            phi_rows = self.alloc((B, npad1, d), self.adt, zero=True)
            phi = phi_rows.as_strided((B, Tp, Hp, Wp, d), (npad1 * d, Hp * Wp * d, Wp * d, d, 1))
            g = self.act(B, Tp, Hp, Wp, d)
            self.conv(xp, phi, *wb(nln.conv_phi))
            self.conv(xp, g, *wb(nln.conv_g))
            gT = transposed(g, "g")
            Sbuf = self.scratch((B, T, H, W, (Nk + 3) // 4 * 4), torch.float32)
            S = Sbuf[..., :Nk]
            Pbuf = self.scratch((B, T, H, W, (Nk + 7) // 8 * 8), self.adt)
            P = Pbuf[..., :Nk]
            zero1 = self.scratch((npad1,), torch.float32, zero=True)
            self.gemm_rows(theta, S, phi_rows, zero1, "nl_gemm", "theta.phi N=%dx%d d=%d" % (Nq, Nk, d))
            self._launch("esf_row_softmax", Sbuf, B * Nq, Nk, Sbuf.shape[4], float(d) ** -0.5, 0, self.a16, Pbuf,
                         Pbuf.shape[4], kind="nl_softmax", label=nln.instantiation, nbytes=self._nbytes(S, P),
                         exps=float(B * Nq * Nk))
            self.gemm_rows(P, att, gT, bias2, "nl_gemm", "p.g N=%dx%d d=%d" % (Nq, Nk, d))
        else:
            # "dot_product" has no non-linearity between the two products:  (theta^T phi / Nk) g^T = theta^T (phi g^T / Nk),
            # a d x d matrix per clip instead of the Nq x Nk affinity -- 2 Nk d^2 + 2 Nq d^2 FLOP instead of 4 Nq Nk d,
            # and nothing of size Nq x Nk is ever written.  M^T[c][c'] = sum_p (g[p][c] / Nk) phi[p][c'] is itself a
            # per-clip-weights GEMM over the transposed rows, and its 16-bit output IS the [n][k] weight matrix of
            # att = theta M.  (The 1 / Nk goes into the g conv so that M stays O(1) in 16 bits.)
            assert rt.igemm_geometry(d, d)[3] == d, "dim_inner must be a whole N tile"
            theta = self.act(B, T, H, W, d)
            self.conv(x, theta, *wb(nln.conv_theta))
            phi = self.act(B, Tp, Hp, Wp, d)
            g = self.act(B, Tp, Hp, Wp, d)
            self.conv(xp, phi, *wb(nln.conv_phi))
            wg, bg = wb(nln.conv_g)
            self.conv(xp, g, wg / Nk, bg / Nk)
            phiT, gT = transposed(phi, "phi"), transposed(g, "g")
            MT = self.alloc((B, 1, 1, d, d), self.adt, zero=True)
            zero_d = self.scratch((d,), torch.float32, zero=True)
            kpad = gT.shape[2]
            gT_act = gT.as_strided((B, 1, 1, d, Nk), (gT.stride(0), d * kpad, d * kpad, kpad, 1))
            self.gemm_rows(gT_act, MT, phiT, zero_d, "nl_gemm", "g^T.phi d=%d Nk=%d" % (d, Nk))
            self.gemm_rows(theta, att, MT.reshape(B, d, d), bias2, "nl_gemm", "theta.M N=%d d=%d" % (Nq, d))
        w, bias = self.once(fold_conv_bn, nln.conv_out.weight, nln.conv_out.bias, nln.bn)
        bias = bias + w.reshape(C, d) @ mu
        self.conv(att, y, w, bias, res=x)

    def conv_wfold(self, x, y, w_folded, bias, WB, stride=(1, 1, 1), padding=(0, 0, 0), act=rt.ACT_NONE, res=None):
        """Thin-layer (C_in <= 32) conv as a W-folded banded GEMM: see esf_conv_wfold_create."""
        wp, bp = self.once(pack_wfold_band, w_folded, bias, WB, stride[2], self.device, self.adt)
        kt, kh, kw = w_folded.shape[2:]
        h = self._create("esf_conv_wfold_create",
                         self._conv_desc(x, y, res, wp, bp, (kt, kh, kw), stride, padding, act=act), WB)
        cout, cin = w_folded.shape[:2]
        m = y.shape[0] * y.shape[1] * y.shape[2] * y.shape[3]
        self._launch("esf_op_launch", h, kind="conv_wfold",
                     label="%dx%dx%d s%s %d->%d @%s wb%d" % (kt, kh, kw, "".join(map(str, stride)), cin, cout,
                                                             tuple(y.shape[1:4]), WB),
                     flops=2.0 * m * cout * cin * kt * kh * kw, nbytes=self._nbytes(x, y, res) + wp.numel() * 2)

    @staticmethod
    def _aligned(t):
        """True when a view can be addressed by TMA / 16-byte vector accesses."""
        if t is None:
            return True
        q = 16 // t.element_size()
        return t.data_ptr() % 16 == 0 and all(st % q == 0 for st in t.stride()[:4])

    def conv(self, x, y, w_folded, bias, stride=(1, 1, 1), padding=(0, 0, 0), dilation=(1, 1, 1), groups=1,
             act=rt.ACT_NONE, res=None, out_dtype=None):
        """Conv3d + folded BN (+ residual) + activation: tensor-core implicit GEMM when the layer is dense and its
        views are 16-byte addressable, CUDA-core direct conv otherwise (grouped / depthwise / odd channel counts)."""
        if groups == 1 and x.shape[4] >= 8 and self._aligned(x) and self._aligned(y) and self._aligned(res):
            wb = wfold_block(x, y, res, w_folded.shape, stride, padding, dilation) if self.wfold else 0
            if wb:
                return self.conv_wfold(x, y, w_folded, bias, wb, stride, padding, act, res)
            return self.conv_igemm(x, y, w_folded, bias, stride, padding, dilation, act, res, out_dtype)
        cout, cin_g = w_folded.shape[:2]
        if (not self._aligned(y) and self._aligned(x) and self._aligned(res) and x.shape[4] >= 8 and cout >= 8
                and groups <= 8 and groups != x.shape[4] and y.dtype == self.adt and (out_dtype in (None, rt.dtype_code(y)))
                and y.data_ptr() % 4 == 0 and all(st % 2 == 0 for st in y.stride()[:4])):
            # The only obstacle to the tensor-core path is an output slice at a channel offset that is not a multiple of
            # 8 (ShuffleNet: the fast pathway's 15 -> 60 grouped conv lands behind the 60 fused channels of the concat
            # buffer; 0.72 ms on the generic CUDA-core kernel against 0.03 ms of HBM time): run the GEMM into an aligned
            # buffer of its own and copy the rows into the slice.
            tmp = self.act(*y.shape[:4], cout)
            # (with these preconditions the recursion always ends on the implicit GEMM: dense, per-group or block-diagonal)
            self.conv(x, tmp, w_folded, bias, stride, padding, dilation, groups, act, res, out_dtype)
            return self.shuffle_concat(tmp, None, 1, y)
        if (groups > 1 and cin_g % 8 == 0 and (cout // groups) % 8 == 0 and cin_g >= 16 and self._aligned(x)
                and self._aligned(y) and self._aligned(res)):
            # grouped dense conv (ShuffleNet's grouped 1x1x1): one implicit GEMM per group on channel slices
            cout_g = cout // groups
            for g in range(groups):
                self.conv_igemm(x[..., g * cin_g:(g + 1) * cin_g], y[..., g * cout_g:(g + 1) * cout_g],
                                w_folded[g * cout_g:(g + 1) * cout_g], bias[g * cout_g:(g + 1) * cout_g], stride,
                                padding, dilation, act, None if res is None else res[..., g * cout_g:(g + 1) * cout_g],
                                out_dtype)
            return
        if (1 < groups <= 8 and cin_g * groups >= 8 and x.shape[4] != groups and self._aligned(x) and self._aligned(y)
                and self._aligned(res)):
            # grouped conv whose group slices are not 16-byte addressable (ShuffleNet g3: 180 / 18 / 5 channels per
            # group): one dense GEMM over all input channels with a block-diagonal weight.  The layer is HBM bound, the
            # `groups`-fold MACs on structural zeros cost nothing next to the CUDA-core fallback.
            return self.conv_igemm(x, y, block_diagonal(w_folded, groups), bias, stride, padding, dilation, act, res,
                                   out_dtype)
        self.conv_direct(x, y, w_folded, bias, stride, padding, dilation, groups, act, res, out_dtype)
        why = [n for n, t in (("x", x), ("y", y), ("res", res)) if not self._aligned(t)]
        self.meta[-1]["why_direct"] = ("groups=%d " % groups if groups != 1 else "") + \
            ("cin<8 " if x.shape[4] < 8 else "") + ("unaligned " + ",".join(
                "%s(off %d, strides %s)" % (n, (t.data_ptr() % 16) // 2, tuple(t.stride()[:4]))
                for n, t in (("x", x), ("y", y), ("res", res)) if n in why) if why else "")

    def conv_direct(self, x, y, w_folded, bias, stride=(1, 1, 1), padding=(0, 0, 0), dilation=(1, 1, 1), groups=1,
                    act=rt.ACT_NONE, res=None, out_dtype=None):
        wd = self.tensor(w_folded.permute(0, 2, 3, 4, 1))  # [Cout][kT][kH][kW][Cin/g]
        bd = self.tensor(bias)
        kt, kh, kw = w_folded.shape[2:]
        d = self._conv_desc(x, y, res, wd, bd, (kt, kh, kw), stride, padding, dilation, groups, act)
        m = y.shape[0] * y.shape[1] * y.shape[2] * y.shape[3]
        depthwise = groups == x.shape[4] == y.shape[4] and kw in (3, 5)
        C = x.shape[4]
        pad_of = lambda t: self.padded.get(t.data_ptr()) if t is not None else (C, (C + 7) // 8 * 8)
        if (depthwise and C % 8 != 0 and C >= 8 and tuple(dilation) == (1, 1, 1) and stride[2] in (1, 2)
                and all(pad_of(t) == (C, (C + 7) // 8 * 8) for t in (x, y, res)) and y.dtype == x.dtype == self.adt):
            # rows padded to a multiple of 8 channels by act(): 16-byte vectors over the padded width (zero weights)
            cp = (C + 7) // 8 * 8
            self._launch("esf_dwconv_padded", d, cp, kind="dwconv",
                         label="%dx%dx%d s%d%d%d g%d %d->%d pad%d @%s" % (kt, kh, kw, *stride, groups, C, C, cp,
                                                                          tuple(x.shape[1:4])),
                         flops=2.0 * m * C * kt * kh * kw, nbytes=self._nbytes(x, y, res) + wd.numel() * 4)
            return
        cout = y.shape[4]
        call = ("esf_conv_direct", d)
        if (groups == 1 and (kt, kh, kw) == (1, 1, 1) and cout >= 8 and cout % 8 != 0 and y.dtype == self.adt
                and self.padded.get(y.data_ptr()) == (cout, (cout + 7) // 8 * 8)):
            # y is a whole padded allocation (not a concat slice): the kernel may write the row padding too
            call = ("esf_pointwise_padded", d, (cout + 7) // 8 * 8)
        self._launch(*call, kind="dwconv" if depthwise else "conv_direct",
                     label="%dx%dx%d s%d%d%d g%d %d->%d @%s" % (kt, kh, kw, *stride, groups, x.shape[4], y.shape[4],
                                                                tuple(x.shape[1:4])),
                     flops=2.0 * m * y.shape[4] * (x.shape[4] // groups) * kt * kh * kw,
                     nbytes=self._nbytes(x, y, res) + wd.numel() * 4)

    def stem_conv(self, x_nc, y, w_folded, bias, stride, padding, act=rt.ACT_RELU):
        """x_nc: FP32 (B,Cin,T,H,W) contiguous plan-owned input buffer."""
        ws = self.tensor(w_folded.permute(2, 3, 4, 1, 0))  # [kT][kH][kW][Cin][Cout]
        bs = self.tensor(bias)
        B, Cin, T, H, W = x_nc.shape
        cout = w_folded.shape[0]
        kt, kh, kw = w_folded.shape[2:]
        yv = rt.view(y)
        self.keep += [y, yv]
        m = y.shape[0] * y.shape[1] * y.shape[2] * y.shape[3]
        self._add(lambda s: self._call(
            "esf_stem_conv", self._in_ptr(x_nc), B, Cin, T, H, W, ws.data_ptr(), bs.data_ptr(), cout, kt, kh, kw, *stride,
            *padding, act, ctypes.byref(yv), s), "stem_conv",
            "%dx%dx%d %d->%d" % (kt, kh, kw, Cin, cout), flops=2.0 * m * cout * Cin * kt * kh * kw,
            nbytes=self._nbytes(x_nc, y), eager=True)

    def _in_ptr(self, x_nc):
        p = x_nc.data_ptr()
        return self.input_override.get(p, p)

    def stem(self, x_nc, y, w_folded, bias, stride, padding, act=rt.ACT_RELU):
        """Stem conv + folded BN + ReLU on the kernel stem_route picks; an output that is not dense takes the CUDA-core
        stem as well."""
        route = stem_route(x_nc.shape, w_folded.shape, stride, padding)
        if route is None or not y.is_contiguous():
            return self.stem_conv(x_nc, y, w_folded, bias, stride, padding, act)
        self.stem_gemm(x_nc, y, w_folded, bias, stride, padding, act, *route)

    def _stem_gemm_op(self, xp, x_shape, y, w_folded, bias, stride, padding, act, pitch, twb, name=""):
        """One tensor-core stem GEMM from the packed 16-bit rows `xp` into the dense `y`: the weight is band-packed for the
        temporal-band kernel (twb > 0 output columns per block) or the banded kernel (twb == 0), the op is created and
        its launch appended to the plan."""
        B, Cin, T, H, W = x_shape
        cout = w_folded.shape[0]
        kt, kh, kw = w_folded.shape[2:]
        if twb:
            wb, bt = self.once(pack_stem_tband, w_folded, bias, twb, stride[2], self.device, self.adt)
        else:
            wb, bt = self.once(pack_stem_band, w_folded, bias, stride[2], self.device, self.adt)
        h = self._create("esf_stem_tband_create" if twb else "esf_stem_igemm_create", xp, B, Cin, T, H, W, pitch, wb, bt,
                         cout, kt, kh, kw, stride[1], stride[2], padding[0], padding[1], padding[2], act, y)
        label = "%dx%dx%d %d->%d %s" % (kt, kh, kw, Cin, cout, "t-band" if twb else "banded")
        m = y.shape[0] * y.shape[1] * y.shape[2] * y.shape[3]
        self._launch("esf_op_launch", h, kind="stem_igemm", label=label + (" " + name if name else ""),
                     flops=2.0 * m * cout * Cin * kt * kh * kw, nbytes=self._nbytes(xp, y) + wb.numel() * 2)

    def stem_gemm(self, x_nc, y, w_folded, bias, stride, padding, act, pitch, lpad, twb):
        """Stem on the tensor cores: the clip is packed into 16-bit rows (`pitch`, `lpad`: esf_stem_geometry), then one
        GEMM -- temporal-band for twb > 0, banded for twb == 0 (see stem_route)."""
        B, Cin, T, H, W = x_nc.shape
        xp = self.alloc((B, T, H, pitch), self.adt)
        self.stem_routes[x_nc.data_ptr()] = (xp, pitch, lpad)   # the uint8 frame route writes xp itself (frames.py)

        def pack(s):
            g = self.gather.get(x_nc.data_ptr())
            if g is not None:       # frames of this pathway are read out of another pathway's clip (slow from fast)
                src, tsrc, idx = g
                self._call("esf_stem_pack_gather", src, B, Cin, tsrc, H, W, idx, T, pitch, lpad, self.a16, xp.data_ptr(), s)
            else:
                self._call("esf_stem_pack", self._in_ptr(x_nc), B, Cin, T, H, W, pitch, lpad, self.a16, xp.data_ptr(), s)

        self._add(pack, "stem_pack", "", nbytes=self._nbytes(x_nc, xp), eager=True)
        self.meta[-1]["is_pack"] = True
        self._stem_gemm_op(xp, x_nc.shape, y, w_folded, bias, stride, padding, act, pitch, twb)

    def pool(self, x, y, kernel, stride, padding, is_avg=False, act=rt.ACT_NONE):
        self._launch("esf_pool3d", x, y, *kernel, *stride, *padding, int(is_avg), act, kind="pool",
                     label="%s C=%d" % (tuple(kernel), x.shape[4]), nbytes=self._nbytes(x, y))

    def shuffle_concat(self, a, b, groups, y):
        self._launch("esf_shuffle_concat", a, b, groups, y, kind="shuffle", label="g%d" % groups,
                     nbytes=2 * self._nbytes(y))

    def eltwise_add(self, a, b, y, act=rt.ACT_NONE):
        self._launch("esf_eltwise_add", a, b, y, act, kind="add", nbytes=3 * self._nbytes(y))

    def squeeze_excite(self, x, y, se):
        """SqueezeExcite (ghostnet_helper.py:34-52): global mean -> 1x1x1(+bias) -> ReLU -> 1x1x1(+bias) -> hard-sigmoid
        -> channel scale.  Reuses the head kernels for the pooled MLP."""
        B, C = x.shape[0], x.shape[4]
        R = se.conv_reduce.out_channels
        feat = self.alloc((B, C), torch.float32)
        hid = self.alloc((B, R), torch.float32)
        gate = self.alloc((B, C), torch.float32)
        w1, b1 = self.tensor(se.conv_reduce.weight.reshape(R, C)), self.tensor(se.conv_reduce.bias)
        w2, b2 = self.tensor(se.conv_expand.weight.reshape(C, R)), self.tensor(se.conv_expand.bias)
        self.global_mean(x, feat, C, 0, "se_pool")
        self._head_fc(feat, w1, b1, rt.HEAD_RELU, hid, kind="se_fc")
        self._head_fc(hid, w2, b2, rt.HEAD_HARD_SIGMOID, gate, kind="se_fc")
        self._launch("esf_channel_scale", x, gate, y, kind="se_scale", nbytes=2 * self._nbytes(x))

    def global_mean(self, x, feat, feat_stride, feat_off, kind="head_pool"):
        """feat[:, feat_off : feat_off + C] = mean over (T, H, W) of x: the two-pass esf_global_mean for large maps, the
        single-block head kernel for the small ones."""
        B, T, H, W, C = x.shape
        if T * H * W >= 1024 and (C % 8 == 0 or C <= 256):
            scratch = self.scratch((self._size("esf_global_mean_scratch_floats", B, C),), torch.float32, flat=True)
            self._launch("esf_global_mean", x, scratch, feat, feat_stride, feat_off, kind=kind, label="two-pass",
                         nbytes=self._nbytes(x), launches=2)
        else:
            assert feat_off == 0
            self._launch("esf_head_pool", x, None, feat, kind=kind, nbytes=self._nbytes(x))

    def eca_fuse(self, x_fast, y_slice, alpha, eca_weight, bn):
        """MaxPool(alpha,1,1) -> ECA -> BN -> ReLU -> concat slice (custom_video_model_builder.py:131-135)."""
        self._eca_fuse("esf_eca_fuse", "esf_eca_scratch_floats", "eca_fuse", x_fast, y_slice, alpha, eca_weight, bn)

    def _eca_fuse(self, fn_name, scratch_fn_name, kind, x_fast, y_slice, alpha, eca_weight, bn):
        """eca_fuse on the entry point `fn_name` (the 16-bit one or its FP32 form) and its partial-sum scratch."""
        scale, shift = self.once(bn_affine, bn)
        w = self.tensor(eca_weight.reshape(-1))
        sc, sh = self.tensor(scale), self.tensor(shift)
        B, C = x_fast.shape[0], x_fast.shape[4]
        scratch = self.alloc((self._size(scratch_fn_name, B, C),), torch.float32, flat=True)
        self._launch(fn_name, x_fast, alpha, w, int(w.numel()), sc, sh, scratch, y_slice, kind=kind, label="C=%d" % C,
                     nbytes=2 * self._nbytes(x_fast) + self._nbytes(y_slice), launches=2)

    def _attention_operands(self, x_slow, alpha, w_down, att, bn):
        """Common part of position_attention: attention_projection as one conv into the FP32 rows `proj`
        [x_d | q | k | v], and the (B, T, H, W, d, gamma, bn scale, bn shift, alpha) arguments that every attention entry
        point takes after its operand."""
        B, T, H, W, C = x_slow.shape
        w_all, b_all, d = self.once(attention_projection, w_down, att)
        proj = self.act(B, T, H, W, 4 * d, dtype=torch.float32)
        self.conv(x_slow, proj, w_all, b_all)
        scale, shift = self.once(bn_affine, bn)
        sc, sh = self.tensor(scale), self.tensor(shift)
        gamma = float(att.gamma.detach().float().item())
        return proj, (B, T, H, W, d, gamma, sc, sh, alpha)

    def _attention_generic(self, proj, geo, y):
        """esf_attn_generic: the CUDA-core attention for head dims above the tensor-core kernels' (d > 128)."""
        B, T, H, W, d = geo[:5]
        N = T * H * W
        self._launch("esf_attn_generic", proj, *geo, y, kind="attention", label="N=%d d=%d generic" % (N, d),
                     flops=4.0 * B * N * N * d, exps=float(B) * N * N, nbytes=self._nbytes(proj, y))

    def position_attention(self, x_slow, y_slice, alpha, w_down, att, bn):
        """attention_projection as one GEMM (FP32 out), hi/lo packing, fused flash-style attention + gamma*O + x + BN +
        ReLU + x alpha upsample + concat (custom_video_model_builder.py:141-146, wdf_attention_helper.py:33-54): the
        tcgen05 kernel up to d = 128, the CUDA-core fallback above."""
        proj, geo = self._attention_operands(x_slow, alpha, w_down, att, bn)
        B, T, H, W, d = geo[:5]
        N = T * H * W
        if d > 128:
            return self._attention_generic(proj, geo, y_slice)
        nbytes = self._size("esf_attn_tc_pack_bytes", B, N, d)
        packed = self.alloc((nbytes,), torch.uint8, flat=True)
        h = self._create("esf_attn_tc_create", packed, *geo, y_slice)
        self._launch("esf_attn_tc_pack", proj, B, N, d, self.a16, packed, kind="attn_pack", label="N=%d d=%d" % (N, d),
                     nbytes=self._nbytes(proj) + nbytes)
        self._launch("esf_op_launch", h, kind="attention", label="N=%d d=%d" % (N, d), flops=4.0 * B * N * N * d,
                     exps=float(B) * N * N, nbytes=nbytes + self._nbytes(y_slice))

    def head(self, xs, weight, bias, act):
        B = xs[0].shape[0]
        cin = sum(x.shape[4] for x in xs)
        K = weight.shape[0]
        feat = self.alloc((B, cin), torch.float32)
        out = self.alloc((B, K), torch.float32)
        w, b = self.tensor(weight), self.tensor(bias)
        self._head_pool(xs, feat)
        self._head_fc(feat, w, b, act, out, flops=2.0 * B * cin * K, nbytes=self._nbytes(feat, w, out))
        self.out = out
        return out

    def _head_pool(self, xs, feat):
        """feat = the global means of the one or two pathways `xs`, concatenated."""
        self._launch("esf_head_pool", xs[0], xs[1] if len(xs) > 1 else None, feat, kind="head_pool",
                     nbytes=self._nbytes(*xs), launches=len(xs))

    def head_positions(self, xs, pool_sizes, weight, bias, act):
        """ResNetBasicHead.forward, eval branch, general case (head_helper.py:198-223): per-pathway AvgPool3d(kernel,
        stride 1) leaves P = T' * H' * W' positions; Linear + activation at every position, mean over the positions."""
        pooled = []
        for x, ps in zip(xs, pool_sizes):
            B, T, H, W, C = x.shape
            kt, kh, kw = [int(v) for v in ps]
            pooled.append(self._head_avg_pool(x, (kt, kh, kw), (B, T - kt + 1, H - kh + 1, W - kw + 1, C)))
        return self.positions_head(pooled, weight, bias, act)

    def _head_avg_pool(self, x, kernel, shape):
        """AvgPool3d(kernel, stride 1) of head_positions into a new activation of `shape`."""
        y = self.act(*shape)
        self.pool(x, y, kernel, (1, 1, 1), (0, 0, 0), is_avg=True)
        return y

    def positions_head(self, pooled, weight, bias, act):
        """Second half of head_positions: Linear + activation at every position of the pooled maps (B, T', H', W', C)
        of all pathways, then the mean over the positions."""
        B = pooled[0].shape[0]
        pos = tuple(pooled[0].shape[1:4])
        assert all(tuple(y.shape[1:4]) == pos for y in pooled), "pathway dimensions are not consistent."
        P = pos[0] * pos[1] * pos[2]
        rows = []
        for y in pooled:    # (B, T', H', W', C) -> one 1x1x1 "clip" per (clip, position)
            C = y.shape[4]
            assert y.stride(3) * pos[2] == y.stride(2) and y.stride(2) * pos[1] == y.stride(1) and y.stride(1) * pos[0] == y.stride(0)
            rows.append(y.as_strided((B * P, 1, 1, 1, C), (y.stride(3), y.stride(3), y.stride(3), y.stride(3), 1),
                                     y.storage_offset()))
        per_pos = self.head(rows, weight, bias, act)
        K = weight.shape[0]
        out = self.alloc((B, K), torch.float32)
        self._launch("esf_group_mean", per_pos, B, P, K, out, kind="head_mean", label="P=%d" % P,
                     nbytes=self._nbytes(per_pos, out))
        self.out = out
        return out

    def pooled_fc(self, x, weight, bias, act, out, out_stride):
        """global mean over (T,H,W) of one activation -> FC (+bias, act) -> `out` (FP32 rows of stride out_stride):
        the `avg_pool3d -> conv_head_{slow,fast} -> ReLU` tail of GhostNetBasicHead (head_helper.py:676-688)."""
        B, C = x.shape[0], x.shape[4]
        K = weight.shape[0]
        feat = self.alloc((B, C), torch.float32)
        w, b = self.tensor(weight.reshape(K, C)), self.tensor(bias)
        self._head_pool([x], feat)
        self._head_fc(feat, w, b, act, out, out_stride)

    def fc(self, feat, weight, bias, act):
        """out = act(feat @ weight^T + bias) on FP32 rows (final classifier of the GhostNet head)."""
        out = self.alloc((feat.shape[0], weight.shape[0]), torch.float32)
        self._head_fc(feat, self.tensor(weight), self.tensor(bias), act, out)
        self.out = out
        return out

    def temporal_mean(self, x):
        """ResNetRoIHead's temporal AvgPool3d([T, 1, 1]) where it leaves one frame: 16-bit (B, T, H, W, C) -> dense FP32
        (B, H, W, C) map, the input of esf_roi_align_max.  A graph op: it reads plan-owned activations only."""
        B, T, H, W, C = x.shape
        y = self.alloc((B, H, W, C), torch.float32)
        self._launch("esf_temporal_mean", x, y, kind="roi_tpool", label="T=%d C=%d @%s" % (T, C, (H, W)),
                     nbytes=self._nbytes(x, y))
        return y

    def roi_head(self, maps, spatial_scales, resolutions, aligned, weight, bias, act):
        """Box-dependent part of ResNetRoIHead over the FP32 `maps` (one per pathway, written by temporal_mean):
        RoIAlign + MaxPool2d into one FP32 row per box, then Linear + activation.  Nothing is recorded into the plan's
        launch list: the box count is only known per call, so run_boxes() issues these launches after the trunk."""
        self.roi = dict(maps=maps, scales=[float(v) for v in spatial_scales], res=[int(v) for v in resolutions],
                        aligned=int(bool(aligned)), w=self.tensor(weight), b=self.tensor(bias), act=act,
                        cin=sum(m.shape[3] for m in maps), ncls=int(weight.shape[0]))
        self.roi_feat = self.roi_out = None

    def run_boxes(self, boxes):
        """`boxes`: (K, 5) contiguous FP32 on this plan's device, K >= 1, rows [batch index, x1, y1, x2, y2].  Launches
        esf_roi_align_max per pathway (both write slices of the same feature row) and esf_head_fc on the current
        stream; the feat / out buffers grow to the largest K seen and are reused (by every plan of a Family).  Returns a
        view of the first K rows."""
        r = self.roi
        K = boxes.shape[0]
        rows = self.shared
        if rows.roi_out is None or rows.roi_out.shape[0] < K:
            rows.roi_feat = torch.empty((K, r["cin"]), dtype=torch.float32, device=self.device)
            rows.roi_out = torch.empty((K, r["ncls"]), dtype=torch.float32, device=self.device)
        L = rt.lib()
        s = rt.current_stream_ptr()
        off = 0
        for m, scale, res in zip(r["maps"], r["scales"], r["res"]):
            B, H, W, C = m.shape
            rt.check(L.esf_roi_align_max(m.data_ptr(), B, H, W, C, boxes.data_ptr(), K, scale, res, r["aligned"],
                                         rows.roi_feat.data_ptr(), r["cin"], off, s), "esf_roi_align_max")
            off += C
        rt.check(L.esf_head_fc(rows.roi_feat.data_ptr(), K, r["cin"], r["cin"], r["w"].data_ptr(), r["b"].data_ptr(),
                               r["ncls"], r["act"], rows.roi_out.data_ptr(), r["ncls"], s), "esf_head_fc")
        return rows.roi_out[:K]

    # ---------------------------------------------------------------- execution
    def launch_all(self):
        s = rt.current_stream_ptr()
        for op in self.ops:
            op(s)

    def launch_graph_ops(self):
        s = rt.current_stream_ptr()
        for op, eager in zip(self.ops, self.eager):
            if not eager:
                op(s)

    def launch_eager_ops(self):
        s = rt.current_stream_ptr()
        for op, eager in zip(self.ops, self.eager):
            if eager:
                op(s)

    def capture(self):
        """Record every launch that only touches plan-owned memory into one CUDA graph (replayed by run()); the ops
        that read the caller's clips (stem packing) stay outside and run ahead of the replay."""
        torch.cuda.synchronize(self.device)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            self.launch_all()  # warm-up outside capture: sets kernel attributes, faults in the code
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.launch_graph_ops()
        self.graph = g

    def profile_ops(self, repeats=3):
        """Per-op device time (ms, best of `repeats`) with CUDA events on the launching stream, eager launches."""
        s = rt.current_stream_ptr()
        times = [float("inf")] * len(self.ops)
        for _ in range(repeats):
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(self.ops) + 1)]
            evs[0].record()
            for i, op in enumerate(self.ops):
                op(s)
                evs[i + 1].record()
            torch.cuda.synchronize(self.device)
            for i in range(len(self.ops)):
                times[i] = min(times[i], evs[i].elapsed_time(evs[i + 1]))
        return times

    def run_frames(self, fill):
        """Frame route: `fill()` launches the kernels that write the stem inputs from uint8 frames (frames.py); the
        FP32 stem-pack launches are skipped, every other launch is the same as in run()."""
        self.input_override = {}
        fill()
        s = rt.current_stream_ptr()
        for op, eager, meta in zip(self.ops, self.eager, self.meta):
            if meta.get("is_pack"):
                continue
            if eager or self.graph is None:
                op(s)
        if self.graph is not None:
            self.graph.replay()
        return self.out

    def run(self, inputs=None, gather=None):
        """`inputs`: optional caller tensors to read INSTEAD of the plan-owned input buffers (same shape, FP32,
        contiguous, same device; None entries keep the plan's buffer) -- saves the device-to-device staging copy.
        `gather`: {pathway: (source clip tensor, device int32 frame index)} -- that pathway's banded stem packs its rows
        out of the source clip's frames (Plan.stem_gemm / esf_stem_pack_gather)."""
        self.input_override = {}
        if inputs is not None:
            self.input_override = {own.data_ptr(): src.data_ptr() for own, src in zip(self.inputs, inputs)
                                   if src is not None}
        self.gather = {}
        for pw, (src, idx) in (gather or {}).items():
            assert self.inputs[pw].data_ptr() in self.stem_routes
            self.gather[self.inputs[pw].data_ptr()] = (src.data_ptr(), src.shape[2], idx.data_ptr())
        try:
            if self.graph is not None:
                self.launch_eager_ops()
                self.graph.replay()
            else:
                self.launch_all()
        finally:
            self.input_override = {}
            self.gather = {}
        return self.out

    def __del__(self):
        try:
            L = rt.lib()
            for h in self.handles:
                L.esf_op_destroy(h)
        except Exception:
            pass
