"""uint8 frame input (SURVEY 8-f4): the loader-side chain of the reference moved behind the H2D copy.

The reference decodes a clip to uint8 (T, H, W, C) frames, then on the host: `tensor_normalize` (u8 -> float / 255,
- mean, / std; SlowFast/slowfast/datasets/utils.py:298-315), `permute(3, 0, 1, 2)` (datasets/kinetics.py:231-235),
crop, and `pack_pathway_output` (datasets/utils.py:73-112: optional channel reversal, slow pathway = frames gathered at
`linspace(0, T-1, T // ALPHA).long()`).  The result -- 4 bytes per sample, the slow frames twice -- is what crosses
PCIe.  `model.forward_frames(frames_u8)` takes the byte frames instead and the stem-pack kernel does the chain on the
device: 1/5 of the H2D bytes, bit-identical stem input (the byte -> value table is computed here with the reference's
own FP32 operations).

Test-time spatial sampling (`forward_frames(frames, crop_size=S, spatial_idx=(0, 1, 2))`): the reference's Kinetics test
branch resizes every normalised clip so that its short side is S (bilinear, on the CPU) and takes `uniform_crop`s of S x S
(datasets/utils.py spatial_sampling, transform.py).  The byte frames at decode size go to the device instead and one
kernel (csrc/esf_crop.cu) normalises, resizes, crops and packs; the resize follows the per-axis tables of `axis_table`,
which reproduce torch's CPU weights bit for bit.

Mixed decode sizes (`forward_frames([clip, ...], crop_size=S, spatial_idx=...)`): a test split mixes resolutions and
aspect ratios, and the reference's loader resizes and crops every clip on its own before collating the S x S crops.  A
list of B uint8 clips (T, H_b, W_b, C) of one T and C runs the same crops through one launch per 32 clips
(esf_*_crop_ragged); the output shapes, hence the plan, are those of a stacked batch of B clips.

Temporal views (`forward_videos([video, ...], fps=...)`): the reference tests every video as TEST.NUM_ENSEMBLE_VIEWS
temporal clips x TEST.NUM_SPATIAL_CROPS crops.  Its decoder samples temporal clip j out of all decoded frames
(datasets/decoder.py decode with the whole video decoded: get_start_end_idx + temporal_sampling).  `temporal_index`
evaluates those expressions here, and the whole video (N, H, W, C) uint8 goes to the device once; the kernel reads
every view's frames through a per-clip frame table (esf_*_crop_videos).

AVA detection (`forward_ava_frames(frames, boxes)`): the test split of the reference's AVA loader
(datasets/ava_dataset.py _images_and_boxes_preprocessing, PyTorch backend) scales the clip's [0, 1] values so that the
short side is DATA.TEST_CROP_SIZE, with no crop, and normalises AFTER the resize; the boxes go through the same
scale and two clips.  `esf_*_ava` writes the whole resized frame with that order (table u / 255, statistics applied to
the blended value), and `esf_ava_boxes` maps the loader's [0, 1] boxes to resized pixels on the device.
"""
import ctypes
import math

import numpy as np
import torch

from . import runtime as rt


def slow_frame_index(num_frames, alpha):
    """datasets/utils.py:93-102 -- the reference's own expression, so that float rounding of linspace matches."""
    return torch.linspace(0, num_frames - 1, num_frames // alpha).long()


def temporal_index(video_size, fps, num_frames, sampling_rate, target_fps, clip_idx, num_clips):
    """Source frames (int64 [num_frames]) of temporal clip `clip_idx` of `num_clips` out of a video of `video_size`
    decoded frames at `fps`: datasets/decoder.py decode's clip size, get_start_end_idx at clip_idx / num_clips (the
    branch of a fully decoded video; the uniform split, which later upstream versions keep as the default of
    DATA.USE_OFFSET_SAMPLING = False) and temporal_sampling -- the reference's own Python float and torch expressions,
    so that every rounding matches."""
    clip_size = sampling_rate * num_frames / target_fps * fps
    delta = max(video_size - clip_size, 0)
    start_idx = delta * clip_idx / num_clips
    end_idx = start_idx + clip_size - 1
    index = torch.linspace(start_idx, end_idx, num_frames)
    return torch.clamp(index, 0, video_size - 1).long()


def video_frame_tables(video_size, fps, num_frames, sampling_rate, target_fps, num_clips, alpha=None):
    """int32 tables [num_clips][T_p] of the source frames of every pathway frame of the `num_clips` temporal clips of
    one video: [slow, fast] (`alpha` given) or [single].  The slow table is pack_pathway_output's linspace gather of the
    sampled clip, i.e. fast[:, slow_frame_index(num_frames, alpha)]."""
    fast = torch.stack([temporal_index(video_size, fps, num_frames, sampling_rate, target_fps, j, num_clips)
                        for j in range(num_clips)]).to(torch.int32)
    if alpha is None:
        return [fast]
    return [fast[:, slow_frame_index(num_frames, alpha)].contiguous(), fast]


def ensemble_spatial_views(num_spatial_crops):
    """The test loader's spatial indices for TEST.NUM_SPATIAL_CROPS (datasets/kinetics.py): idx % n for n > 1, else
    the centre crop 1."""
    n = int(num_spatial_crops)
    if n < 1:
        raise ValueError("TEST.NUM_SPATIAL_CROPS must be >= 1, got %d" % n)
    return (1,) if n == 1 else tuple(range(n))


def normalization_table(mean, std, channels):
    """FP32 [C][256]: tensor_normalize (datasets/utils.py:298-315) applied to every byte value, per channel."""
    u = torch.arange(256, dtype=torch.uint8).reshape(256, 1).repeat(1, channels)
    t = u.float()
    t = t / 255.0
    t = t - torch.tensor(list(mean)[:channels], dtype=torch.float32)
    t = t / torch.tensor(list(std)[:channels], dtype=torch.float32)
    return t.t().contiguous()


def resized_size(height, width, size):
    """transform.random_short_side_scale_jitter in test mode (min_size = max_size = size): (height, width) after the
    short-side resize; the frame is left alone when its short side already is `size`."""
    if (width <= height and width == size) or (height <= width and height == size):
        return height, width
    if width < height:
        return int(math.floor((float(height) / width) * size)), size
    return size, int(math.floor((float(width) / height) * size))


def crop_offset(height, width, size, spatial_idx):
    """transform.uniform_crop: (y0, x0) of the size x size crop `spatial_idx` (0, 1, 2: start, centre, end of the long
    axis) of a height x width frame."""
    y0 = int(math.ceil((height - size) / 2))
    x0 = int(math.ceil((width - size) / 2))
    if height > width:
        y0 = 0 if spatial_idx == 0 else (height - size if spatial_idx == 2 else y0)
    else:
        x0 = 0 if spatial_idx == 0 else (width - size if spatial_idx == 2 else x0)
    return y0, x0


MAX_VIEWS = 8   # csrc/esf_crop.cu kCropMaxViews
MAX_ROW_BYTES = 16384   # csrc/esf_crop.cu kCropMaxRowBytes: W * C of one source row


def spatial_views(spatial_idx):
    """`spatial_idx` (an int or a sequence of ints from {0, 1, 2}) as a tuple; ValueError otherwise."""
    views = tuple(spatial_idx) if isinstance(spatial_idx, (list, tuple, range)) else (spatial_idx,)
    if not 1 <= len(views) <= MAX_VIEWS:
        raise ValueError("spatial_idx needs 1 to %d views, got %d" % (MAX_VIEWS, len(views)))
    for v in views:
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or int(v) not in (0, 1, 2):
            raise ValueError("spatial_idx values are 0, 1 or 2 (uniform_crop), got %r" % (v,))
    return tuple(int(v) for v in views)


def axis_table(n_in, n_out):
    """Source indices (int32 [n_out][2]: i0, i1) and weights (FP32 [n_out][2]: l0, l1) of one axis of torch's CPU bilinear
    interpolate (align_corners=False, output size given): ATen's compute_source_index_and_lambda with scale =
    float(n_in) / n_out and the source index fma(scale, d + 0.5, -0.5) clamped at 0, as its kernels compile it with FMA
    contraction (AVX2 / AVX512 CPU capability).  An axis that keeps its size is the identity (i0 = d, i1 = 0, 1, 0)."""
    d = np.arange(n_out)
    if n_in == n_out:
        idx = np.stack([d, np.zeros_like(d)], 1)
        wt = np.stack([np.ones(n_out, np.float32), np.zeros(n_out, np.float32)], 1)
        return torch.from_numpy(idx.astype(np.int32)), torch.from_numpy(wt)
    scale = np.float32(n_in) / np.float32(n_out)
    # the product of two FP32 numbers and the sum with 0.5 are exact in FP64: one rounding to FP32, i.e. the FMA
    real = (np.float64(scale) * (d.astype(np.float32) + np.float32(0.5)).astype(np.float64) - 0.5).astype(np.float32)
    real = np.maximum(real, np.float32(0))
    i0 = np.minimum(np.floor(real).astype(np.int64), n_in - 1)
    l1 = np.minimum(np.maximum(real - i0.astype(np.float32), np.float32(0)), np.float32(1)).astype(np.float32)
    i1 = i0 + (i0 < n_in - 1)
    l0 = (np.float32(1) - l1).astype(np.float32)
    return torch.from_numpy(np.stack([i0, i1], 1).astype(np.int32)), torch.from_numpy(np.stack([l0, l1], 1))


def _is_shape(x):
    return all(isinstance(n, (int, np.integer)) and not isinstance(n, bool) for n in x)


def clip_shapes(shapes):
    """`shapes` of a list of clips as (T, H, W, C) int tuples; ValueError unless every clip has 4 dimensions, they share
    T and C, and a source row (W * C bytes) fits the crop kernel."""
    out = []
    for sh in shapes:
        if len(sh) != 4 or not _is_shape(sh):
            raise ValueError("a list of clips holds uint8 clips (T, H, W, C), got shape %s" % (tuple(sh),))
        out.append(tuple(int(n) for n in sh))
    if not out:
        raise ValueError("an empty list of clips has no clip shapes")
    T, C = out[0][0], out[0][3]
    for T_b, H_b, W_b, C_b in out:
        if (T_b, C_b) != (T, C):
            raise ValueError("the clips of a list share T and C: (T, C) = (%d, %d) next to (%d, %d)" % (T, C, T_b, C_b))
        if min(T_b, H_b, W_b, C_b) < 1:
            raise ValueError("empty clip of shape %s" % ((T_b, H_b, W_b, C_b),))
        if W_b * C_b > MAX_ROW_BYTES:
            raise ValueError("clip rows of %d x %d bytes exceed the crop kernel's %d" % (W_b, C_b, MAX_ROW_BYTES))
    return out


def view_shapes(frames_shape, crop_size, spatial_idx, alpha=None):
    """Clip shapes [slow, fast] (`alpha` given) or [single] that `forward_frames(frames, crop_size=, spatial_idx=)` runs
    on for uint8 frames of `frames_shape` (B, T, H, W, C), or for a list of B clips of the shapes (T, H_b, W_b, C)
    (`frames_shape` a list of such shapes, see clip_shapes): B * V rows of crop_size x crop_size.  ValueError when a crop
    does not fit a resized frame."""
    views = spatial_views(spatial_idx)
    S = int(crop_size)
    if len(frames_shape) == 0 or not _is_shape(frames_shape):
        clips = clip_shapes(frames_shape)
        B, (T, _, _, C) = len(clips), clips[0]
        sizes = sorted({(H, W) for _, H, W, _ in clips})
    else:
        B, T, H, W, C = (int(n) for n in frames_shape)
        sizes = [(H, W)]
    for H, W in sizes:
        Hr, Wr = resized_size(H, W, S)
        for v in views:
            y0, x0 = crop_offset(Hr, Wr, S, v)
            if S < 1 or y0 < 0 or x0 < 0 or y0 + S > Hr or x0 + S > Wr:
                raise ValueError("a %d x %d crop does not fit frames of %d x %d resized to %d x %d" % (S, S, H, W, Hr, Wr))
    n = B * len(views)
    if alpha is None:
        return [(n, C, T, S, S)]
    return [(n, C, T // alpha, S, S), (n, C, T, S, S)]


def check_clips(clips):
    """Shapes (T, H, W, C) of a list of clip tensors; ValueError unless they are contiguous uint8 clips of 4 dimensions
    on one device that share T and C (clip_shapes)."""
    for c in clips:
        if not isinstance(c, torch.Tensor) or c.dtype != torch.uint8 or c.dim() != 4 or not c.is_contiguous():
            raise ValueError("a list of clips holds contiguous uint8 tensors (T, H, W, C), got %s"
                             % (("%s %s" % (c.dtype, tuple(c.shape))) if isinstance(c, torch.Tensor) else type(c)))
    if len({c.device for c in clips}) > 1:
        raise ValueError("the clips of a list are on one device, got %s" % sorted({str(c.device) for c in clips}))
    return clip_shapes([tuple(c.shape) for c in clips])


def check_videos(videos, fps, num_clips):
    """Shapes (N, H, W, C) of a list of whole videos and their fps as a list of floats; ValueError unless the videos are
    contiguous uint8 tensors (N, H, W, C) on one device with N >= 1, one C and rows that fit the crop kernel, every fps
    is > 0 and num_clips >= 1."""
    if isinstance(num_clips, bool) or not isinstance(num_clips, (int, np.integer)) or num_clips < 1:
        raise ValueError("num_clips (temporal views per video) must be an int >= 1, got %r" % (num_clips,))
    for v in videos:
        if not isinstance(v, torch.Tensor) or v.dtype != torch.uint8 or v.dim() != 4 or not v.is_contiguous():
            raise ValueError("forward_videos takes contiguous uint8 videos (N, H, W, C), got %s"
                             % (("%s %s" % (v.dtype, tuple(v.shape))) if isinstance(v, torch.Tensor) else type(v)))
    if len({v.device for v in videos}) > 1:
        raise ValueError("the videos of a list are on one device, got %s" % sorted({str(v.device) for v in videos}))
    shapes = [tuple(int(n) for n in v.shape) for v in videos]
    for N, H, W, C in shapes:
        if min(N, H, W, C) < 1:
            raise ValueError("empty video of shape %s" % ((N, H, W, C),))
        if C != shapes[0][3]:
            raise ValueError("the videos of a list share C: %d next to %d" % (shapes[0][3], C))
        if W * C > MAX_ROW_BYTES:
            raise ValueError("video rows of %d x %d bytes exceed the crop kernel's %d" % (W, C, MAX_ROW_BYTES))
    rates = list(fps) if isinstance(fps, (list, tuple)) else [fps] * len(videos)
    if len(rates) != len(videos):
        raise ValueError("%d fps values for %d videos" % (len(rates), len(videos)))
    out = []
    for f in rates:
        if isinstance(f, bool) or not isinstance(f, (int, float, np.integer, np.floating)) or not f > 0 \
                or not math.isfinite(f):
            raise ValueError("fps must be a finite number > 0, got %r" % (f,))
        out.append(float(f))
    return shapes, out


def arena_layout(shapes, capacity=None, align=16):
    """Byte offsets of uint8 clips of `shapes` (T, H, W, C) placed one after another in one buffer, each at a multiple of
    `align` bytes, and the bytes they span.  EsfError when `capacity` (bytes) is given and they need more."""
    offsets, end = [], 0
    for sh in shapes:
        start = -(-end // align) * align
        offsets.append(start)
        end = start + math.prod(int(n) for n in sh)
    if capacity is not None and end > capacity:
        raise rt.EsfError("clips of %d bytes (%d-byte aligned) exceed the %d-byte staging buffer" % (end, align, capacity))
    return offsets, end


class CropTables:
    """Device tables of one (H0, W0, crop size, views) geometry: the per-axis resize tables and the crop offsets."""

    def __init__(self, H0, W0, size, views, device):
        self.H0, self.W0, self.S, self.views = H0, W0, size, views
        self.Hr, self.Wr = resized_size(H0, W0, size)
        self.resize = (self.Hr, self.Wr) != (H0, W0)
        self.tables = None
        if self.resize:
            yi, yw = axis_table(H0, self.Hr)
            xi, xw = axis_table(W0, self.Wr)
            self.tables = [t.to(device) for t in (yi, yw, xi, xw)]
        offs = [crop_offset(self.Hr, self.Wr, size, v) for v in views]
        self.crop_yx = (ctypes.c_int32 * (2 * len(views)))(*[o for yx in offs for o in yx])

    def pointers(self):
        if self.tables is None:
            return None, None, self.Hr, None, None, self.Wr
        yi, yw, xi, xw = self.tables
        return yi.data_ptr(), yw.data_ptr(), self.Hr, xi.data_ptr(), xw.data_ptr(), self.Wr

    def addresses(self):
        """Device addresses of (y_index, y_weight, x_index, x_weight); None where the frames are not resized."""
        return (None,) * 4 if self.tables is None else tuple(t.data_ptr() for t in self.tables)


class ClipList:
    """The host arrays of esf_*_crop_ragged for B clips (T, H_b, W_b, C) of mixed decode sizes: every clip's device
    address and the geometry of its CropTables (FrameInput.crop, cached per geometry).  Built per call; the library
    reads them before the call returns."""

    def __init__(self, clips, tables):
        self.B = len(clips)
        self.T, _, _, self.C = clips[0].shape
        self.S, self.V = tables[0].S, len(tables[0].views)
        self.frames = (ctypes.c_void_p * self.B)(*[c.data_ptr() for c in clips])
        self.geom = (ctypes.c_int32 * (4 * self.B))(*[n for t in tables for n in (t.H0, t.W0, t.Hr, t.Wr)])
        self.tables = (ctypes.c_void_p * (4 * self.B))(*[a for t in tables for a in t.addresses()])
        self.crop_yx = (ctypes.c_int32 * (2 * self.V * self.B))(*[o for t in tables for o in t.crop_yx])


class VideoList:
    """The host arrays of esf_*_crop_videos for the temporal views of whole videos (N_v, H_v, W_v, C): clip
    v * num_clips + j is temporal clip j of video v, with the video's device address, its geometry (N_v, H0, W0, Hr,
    Wr), its CropTables and row v * num_clips + j of every pathway's frame table (`tables[v]`, video_frame_tables).
    `index` is one pinned int32 array, the tables of all pathways one after another, copied to the plan's device
    buffer by launch_video_list.  Built per call."""

    def __init__(self, videos, crops, tables, num_clips):
        self.n, self.num_clips = len(videos), num_clips
        self.B = self.n * num_clips
        self.C = videos[0].shape[3]
        self.S, self.V = crops[0].S, len(crops[0].views)
        rep = [i for i in range(self.n) for _ in range(num_clips)]
        self.frames = (ctypes.c_void_p * self.B)(*[videos[i].data_ptr() for i in rep])
        self.geom = (ctypes.c_int32 * (5 * self.B))(*[n for i in rep for n in (videos[i].shape[0], crops[i].H0,
                                                                                crops[i].W0, crops[i].Hr, crops[i].Wr)])
        self.tables = (ctypes.c_void_p * (4 * self.B))(*[a for i in rep for a in crops[i].addresses()])
        self.crop_yx = (ctypes.c_int32 * (2 * self.V * self.B))(*[o for i in rep for o in crops[i].crop_yx])
        self.T = [int(t.shape[1]) for t in tables[0]]    # frames of every pathway
        parts = [torch.cat([tab[p] for tab in tables]).reshape(-1) for p in range(len(self.T))]
        self.index = torch.empty(sum(int(t.numel()) for t in parts), dtype=torch.int32,
                                 pin_memory=torch.cuda.is_available())
        torch.cat(parts, out=self.index)


def unit_table(channels):
    """FP32 [C][256]: `imgs.float() / 255.0` of every byte value (the AVA branch's first step), per channel."""
    u = torch.arange(256, dtype=torch.uint8).float() / 255.0
    return u.reshape(1, 256).repeat(channels, 1).contiguous()


def ava_channel_source(channels, bgr=False, reverse=False):
    """Source channel of every output channel of the AVA branch: the loader swaps BGR -> RGB when AVA.BGR is false
    (after colour normalisation), and pack_pathway_output reverses again under DATA.REVERSE_INPUT_CHANNEL."""
    swap = (not bgr) != bool(reverse)
    if not swap:
        return list(range(channels))
    if channels != 3:
        raise ValueError("the AVA loader's channel swap needs 3 channels, got %d (set AVA.BGR)" % channels)
    return [2, 1, 0]


def check_ava_frames(frames):
    """(B, T, H, W, C) of the uint8 frames of forward_ava_frames; ValueError unless they are one contiguous uint8 tensor
    of 5 dimensions whose rows fit the frame kernel."""
    if not isinstance(frames, torch.Tensor) or frames.dtype != torch.uint8 or frames.dim() != 5 \
            or not frames.is_contiguous():
        raise ValueError("forward_ava_frames takes contiguous uint8 frames (B, T, H, W, C), got %s"
                         % (("%s %s" % (frames.dtype, tuple(frames.shape))) if isinstance(frames, torch.Tensor)
                            else type(frames).__name__))
    B, T, H, W, C = (int(n) for n in frames.shape)
    if min(T, H, W, C) < 1 or C > 4:
        raise ValueError("forward_ava_frames: bad frame shape %s" % ((B, T, H, W, C),))
    if W * C > MAX_ROW_BYTES:
        raise ValueError("frame rows of %d x %d bytes exceed the frame kernel's %d" % (W, C, MAX_ROW_BYTES))
    return B, T, H, W, C


def check_ava_boxes(boxes, batch):
    """The loader's normalised boxes (K, 5) [batch index, x1, y1, x2, y2] as the tensor esf_ava_boxes reads: FP64 kept,
    any other floating type as FP32, contiguous.  ValueError for a wrong type or shape and, for host boxes, for batch
    indices outside [0, batch) (device boxes are not read: that would synchronise)."""
    if not torch.is_tensor(boxes) or not boxes.is_floating_point() or boxes.dim() != 2 or boxes.shape[1] != 5:
        raise ValueError("boxes must be a floating-point (K, 5) tensor of [batch index, x1, y1, x2, y2] in [0, 1]; got %s"
                         % ((tuple(boxes.shape), boxes.dtype) if torch.is_tensor(boxes) else type(boxes).__name__,))
    b = boxes.detach()
    b = b if b.dtype == torch.float64 else b.to(torch.float32)
    if b.device.type == "cpu":
        idx = b[:, 0]
        bad = ~((idx >= 0) & (idx < batch))
        if bool(bad.any()):
            raise ValueError("boxes[:, 0] must be batch indices in [0, %d); got %s" % (batch, idx[bad][:4].tolist()))
    return b.contiguous()


def ava_boxes(boxes, height, width, size):
    """The arithmetic of esf_ava_boxes on the host: the loader's boxes (K, 5) [batch index, x1, y1, x2, y2] in [0, 1]
    of height x width frames -> FP32 (K, 5) in pixels of the frames resized to resized_size(height, width, size).  FP64
    as numpy runs it: times (width, height), clip_boxes_to_image(height, width), times new / old of the short-side
    resize (random_short_side_scale_jitter; none when the short side already is `size`), clip_boxes_to_image(size,
    size), then FP32 as detection_collate makes it."""
    b = np.array(boxes, dtype=np.float64).reshape(-1, 5)
    Hr, Wr = resized_size(height, width, size)
    out = b.copy()
    for j, extent in ((1, width), (2, height), (3, width), (4, height)):
        v = np.minimum(extent - 1.0, np.maximum(0.0, b[:, j] * extent))
        if (Hr, Wr) != (height, width):
            v = v * float(Hr if width < height else Wr) / (height if width < height else width)
        out[:, j] = np.minimum(size - 1.0, np.maximum(0.0, v))
    return torch.from_numpy(out.astype(np.float32))


class AvaInput:
    """Per-(model, device) state of the AVA frame route: the u / 255 table on the device, the channel order and the
    statistics of every source channel (host arrays of esf_*_ava)."""

    def __init__(self, cfg, device, channels):
        data = cfg.DATA
        ava = cfg.get("AVA", None) if hasattr(cfg, "get") else getattr(cfg, "AVA", None)
        get = (lambda node, k, d: node.get(k, d) if node is not None and hasattr(node, "get") else d)
        mean = list(get(data, "MEAN", [0.45] * channels))
        std = list(get(data, "STD", [0.225] * channels))
        if len(mean) != channels or len(std) != channels:
            raise ValueError("DATA.MEAN / DATA.STD have %d / %d entries for %d channels (color_normalization asserts "
                             "one per channel)" % (len(mean), len(std), channels))
        src = ava_channel_source(channels, bool(get(ava, "BGR", False)), bool(get(data, "REVERSE_INPUT_CHANNEL", False)))
        self.lut32 = unit_table(channels).to(device)
        self.chan_src = (ctypes.c_int32 * channels)(*src)
        # np.array(..., dtype=np.float32) in the loader: the statistics are FP32 numbers
        self.mean = (ctypes.c_float * channels)(*[float(np.float32(m)) for m in mean])
        self.std = (ctypes.c_float * channels)(*[float(np.float32(v)) for v in std])


class FrameInput:
    """Per-(model, device) state of the frame route: look-up tables and frame indices on the device."""

    def __init__(self, cfg, device, adt, channels=3):
        data = cfg.DATA
        mean = data.get("MEAN", [0.45] * channels) if hasattr(data, "get") else data.MEAN
        std = data.get("STD", [0.225] * channels) if hasattr(data, "get") else data.STD
        reverse = bool(data.get("REVERSE_INPUT_CHANNEL", False)) if hasattr(data, "get") else False
        self.channels = channels
        lut = normalization_table(mean, std, channels)
        self.lut32 = lut.to(device)
        self.lut16 = lut.to(adt).to(device)
        src = list(range(channels))
        if reverse:
            assert channels == 3, "DATA.REVERSE_INPUT_CHANNEL needs 3 channels"
            src = [2, 1, 0]
            # the reference reverses AFTER normalising: output channel c holds source channel src[c] normalised with
            # the statistics of the SOURCE channel
            self.lut32 = self.lut32[src].contiguous()
            self.lut16 = self.lut16[src].contiguous()
        self.chan_src = (ctypes.c_int32 * channels)(*src)
        # BGR frames (cv2.VideoCapture's order; the demo swaps with COLOR_BGR2RGB before everything else): RGB channel k
        # is frame channel 2 - k, and the tables stay those of the RGB channels
        self.chan_src_bgr = (ctypes.c_int32 * 3)(*[2 - k for k in src]) if channels == 3 else None
        self.device = device
        self._index = {}
        self._crops = {}
        self._videos = {}

    def ava(self, cfg):
        """AvaInput of this device (built on first use)."""
        if getattr(self, "_ava", None) is None:
            self._ava = AvaInput(cfg, self.device, self.channels)
        return self._ava

    def crop(self, H0, W0, size, views):
        """CropTables of frames H0 x W0 cropped to size x size at `views` (cached per geometry)."""
        key = (H0, W0, size, tuple(views))
        if key not in self._crops:
            self._crops[key] = CropTables(H0, W0, size, tuple(views), self.device)
        return self._crops[key]

    def video_tables(self, video_size, fps, num_frames, sampling_rate, target_fps, num_clips, alpha=None):
        """video_frame_tables, cached per (video length, fps, ...): a test split repeats few lengths and rates."""
        key = (video_size, fps, num_frames, sampling_rate, target_fps, num_clips, alpha)
        if key not in self._videos:
            if len(self._videos) >= 4096:
                self._videos.clear()
            self._videos[key] = video_frame_tables(*key)
        return self._videos[key]

    def index(self, t_src, t_out, alpha):
        """device int32 frame gather for a pathway with t_out of t_src frames (None: identity)."""
        if t_out == t_src:
            return None
        key = (t_src, t_out)
        if key not in self._index:
            idx = slow_frame_index(t_src, alpha)
            assert idx.numel() == t_out, "pathway has %d frames, expected %d" % (t_out, idx.numel())
            self._index[key] = idx.to(torch.int32).to(self.device)
        return self._index[key]


def launch_frames(plan, fin, frames, alpha, frame_index=None, crop=None):
    """Fill the stem inputs of `plan` from uint8 frames (B, T, H, W, C) on the current stream.  `frame_index`: optional
    list (one entry per pathway) of device int32 tensors, source frame of every pathway frame -- replaces the loader's
    rule (slow = linspace gather of the fast frames) for callers that keep frames in a ring (demo.SlidingWindow).
    `crop`: CropTables (FrameInput.crop) -- the frames are at decode size and every clip becomes V rows of crops."""
    L = rt.lib()
    s = rt.current_stream_ptr()
    B, Tsrc, H, W, C = frames.shape
    for pw, own in enumerate(plan.inputs):
        b, c, T, h, w = own.shape
        if crop is not None:
            assert (b, c, h, w) == (B * len(crop.views), C, crop.S, crop.S) and (H, W) == (crop.H0, crop.W0)
        else:
            assert (b, c, h, w) == (B, C, H, W)
        if frame_index is not None:
            idx = frame_index[pw]
            assert idx.dtype == torch.int32 and idx.numel() == T and idx.device == frames.device
        else:
            idx = fin.index(Tsrc, T, alpha)
        iptr = idx.data_ptr() if idx is not None else None
        route = plan.stem_routes.get(own.data_ptr())
        if crop is not None:
            geo = crop.pointers() + (crop.crop_yx, len(crop.views), crop.S)
            if route is not None:
                xp, pitch, lpad = route
                rt.check(L.esf_stem_pack_u8_crop(frames.data_ptr(), B, Tsrc, H, W, C, iptr, T, fin.chan_src,
                                                 fin.lut32.data_ptr(), *geo, rt.dtype_code(xp), pitch, lpad,
                                                 xp.data_ptr(), s), "esf_stem_pack_u8_crop")
            else:
                rt.check(L.esf_frames_to_clip_crop(frames.data_ptr(), B, Tsrc, H, W, C, iptr, T, fin.chan_src,
                                                   fin.lut32.data_ptr(), *geo, own.data_ptr(), s),
                         "esf_frames_to_clip_crop")
        elif route is not None:
            xp, pitch, lpad = route
            rt.check(L.esf_stem_pack_u8(frames.data_ptr(), B, Tsrc, H, W, C, iptr, T, fin.chan_src, fin.lut16.data_ptr(),
                                        pitch, lpad, xp.data_ptr(), s), "esf_stem_pack_u8")
        else:
            rt.check(L.esf_frames_to_clip(frames.data_ptr(), B, Tsrc, H, W, C, iptr, T, fin.chan_src,
                                          fin.lut32.data_ptr(), own.data_ptr(), s), "esf_frames_to_clip")


def launch_rings(plan, fin, bank, rows, positions, bgr=False):
    """Fill the stem inputs of `plan` from a bank of per-camera frame rings (N, L, H, W, C) uint8 on the current stream
    (demo.CameraWindows): output row r, frame t of pathway p is ring slot (positions[p][t] + oldest_r) % L of camera
    camera_r.  `rows`: (device, host) contiguous int32 tables (R, 2) of (camera, oldest slot), R = the plan's rows;
    the library's range checks read the host copy.  `positions`: one (device tensor, host ctypes int32 array) pair of
    window positions [T_p] per pathway (demo.window_indices).  `bgr`: the rings hold BGR frames (FrameInput.chan_src_bgr)."""
    L = rt.lib()
    s = rt.current_stream_ptr()
    N, Lr, H, W, C = bank.shape
    dev_rows, host_rows = rows
    assert host_rows.device.type == "cpu" and host_rows.is_contiguous() and host_rows.dtype == torch.int32
    rows_host = ctypes.cast(host_rows.data_ptr(), ctypes.POINTER(ctypes.c_int32))
    for own, (dev_pos, host_pos) in zip(plan.inputs, positions):
        R, c, T, h, w = own.shape
        assert (c, h, w) == (C, H, W) and dev_pos.numel() == len(host_pos) == T
        assert dev_rows.shape[0] >= R and host_rows.shape[0] >= R
        args = (bank.data_ptr(), N, Lr, H, W, C, dev_rows.data_ptr(), rows_host, R, dev_pos.data_ptr(), host_pos, T,
                fin.chan_src_bgr if bgr else fin.chan_src)
        route = plan.stem_routes.get(own.data_ptr())
        if route is not None:
            xp, pitch, lpad = route
            rt.check(L.esf_stem_pack_u8_rings(*args, fin.lut16.data_ptr(), pitch, lpad, xp.data_ptr(), s),
                     "esf_stem_pack_u8_rings")
        else:
            rt.check(L.esf_frames_to_clip_rings(*args, fin.lut32.data_ptr(), own.data_ptr(), s),
                     "esf_frames_to_clip_rings")


def launch_clip_list(plan, fin, clips, alpha):
    """Fill the stem inputs of `plan` from a ClipList on the current stream: row b * V + v is clip b at view v."""
    L = rt.lib()
    s = rt.current_stream_ptr()
    for own in plan.inputs:
        b, c, T, h, w = own.shape
        assert (b, c, h, w) == (clips.B * clips.V, clips.C, clips.S, clips.S)
        idx = fin.index(clips.T, T, alpha)
        args = (clips.frames, clips.B, clips.T, clips.C, idx.data_ptr() if idx is not None else None, T, fin.chan_src,
                fin.lut32.data_ptr(), clips.geom, clips.tables, clips.crop_yx, clips.V, clips.S)
        route = plan.stem_routes.get(own.data_ptr())
        if route is not None:
            xp, pitch, lpad = route
            rt.check(L.esf_stem_pack_u8_crop_ragged(*args, rt.dtype_code(xp), pitch, lpad, xp.data_ptr(), s),
                     "esf_stem_pack_u8_crop_ragged")
        else:
            rt.check(L.esf_frames_to_clip_crop_ragged(*args, own.data_ptr(), s), "esf_frames_to_clip_crop_ragged")


def launch_video_list(plan, fin, videos):
    """Fill the stem inputs of `plan` from a VideoList on the current stream: row (v * num_clips + j) * V + s is video
    v, temporal clip j, crop s.  The frame tables go to a device buffer of the plan (of its family: Plan.shared) with one
    copy from pinned memory."""
    L = rt.lib()
    s = rt.current_stream_ptr()
    need = sum(own.shape[0] * own.shape[2] for own in plan.inputs)   # >= B * T_p of every pathway
    dev = getattr(plan.shared, "video_index", None)
    if dev is None or dev.numel() < need:
        dev = plan.shared.video_index = torch.empty(need, dtype=torch.int32, device=plan.inputs[0].device)
    n = videos.index.numel()
    assert n <= dev.numel()
    dev[:n].copy_(videos.index, non_blocking=True)
    off = 0
    for own, T in zip(plan.inputs, videos.T):
        b, c, t, h, w = own.shape
        assert (b, c, t, h, w) == (videos.B * videos.V, videos.C, T, videos.S, videos.S)
        args = (videos.frames, videos.B, videos.C, dev[off:].data_ptr(), T, fin.chan_src, fin.lut32.data_ptr(),
                videos.geom, videos.tables, videos.crop_yx, videos.V, videos.S)
        off += videos.B * T
        route = plan.stem_routes.get(own.data_ptr())
        if route is not None:
            xp, pitch, lpad = route
            rt.check(L.esf_stem_pack_u8_crop_videos(*args, rt.dtype_code(xp), pitch, lpad, xp.data_ptr(), s),
                     "esf_stem_pack_u8_crop_videos")
        else:
            rt.check(L.esf_frames_to_clip_crop_videos(*args, own.data_ptr(), s), "esf_frames_to_clip_crop_videos")


def launch_ava(plan, fin, ava, frames, crop, alpha):
    """Fill the stem inputs of `plan` from uint8 frames (B, T, H, W, C) with the AVA test branch on the current stream:
    every clip's whole frame resized to crop.Hr x crop.Wr (CropTables without views), normalised after the resize."""
    L = rt.lib()
    s = rt.current_stream_ptr()
    B, Tsrc, H, W, C = frames.shape
    for own in plan.inputs:
        b, c, T, h, w = own.shape
        assert (b, c, h, w) == (B, C, crop.Hr, crop.Wr) and (H, W) == (crop.H0, crop.W0)
        idx = fin.index(Tsrc, T, alpha)
        args = (frames.data_ptr(), B, Tsrc, H, W, C, idx.data_ptr() if idx is not None else None, T, ava.chan_src,
                ava.lut32.data_ptr(), ava.mean, ava.std) + crop.pointers()
        route = plan.stem_routes.get(own.data_ptr())
        if route is not None:
            xp, pitch, lpad = route
            rt.check(L.esf_stem_pack_u8_ava(*args, rt.dtype_code(xp), pitch, lpad, xp.data_ptr(), s),
                     "esf_stem_pack_u8_ava")
        else:
            rt.check(L.esf_frames_to_clip_ava(*args, own.data_ptr(), s), "esf_frames_to_clip_ava")


# one entry of a cv2_axis_table: the layout esf_resize_u8_cv2 reads (8 bytes, little-endian)
CV2_AXIS = np.dtype([("index", "<i4"), ("w0", "<i2"), ("w1", "<i2")])


def cv2_axis_table(n_in, n_out, clamp):
    """One axis of OpenCV's cv2.resize(..., interpolation=cv2.INTER_LINEAR) on uint8 (imgproc resize.cpp, fixed point
    with 11-bit weights), as a CV2_AXIS array [n_out].  With scale = 1 / (n_out / n_in) in double: f = float32((d + 0.5)
    * scale - 0.5), s = floor(f), f -= s; w0 = rint(float32((1 - f) * 2048)), w1 = rint(float32(f * 2048)).  `clamp` (the
    x axis) is OpenCV's column rule: s < 0 gives (0, f = 0) and s >= n_in - 1 gives (n_in - 1, f = 0).  The y axis keeps
    s and f as they are; its rows are s and s + 1 clamped to the frame (which the kernel applies to both axes)."""
    scale = 1.0 / (float(n_out) / n_in)
    f = ((np.arange(n_out, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f)
    f = (f - s).astype(np.float32)
    s = s.astype(np.int64)
    if clamp:
        for edge, value in ((s < 0, 0), (s >= n_in - 1, n_in - 1)):
            s[edge], f[edge] = value, np.float32(0)
    out = np.empty(n_out, CV2_AXIS)
    out["index"] = s
    out["w0"] = np.rint((np.float32(1) - f) * np.float32(2048)).astype(np.int16)
    out["w1"] = np.rint(f * np.float32(2048)).astype(np.int16)
    return out


def scale_boxes(size, boxes, height, width):
    """datasets/cv2_transform.scale_boxes on a copy of FP32 `boxes` (K, 4) in pixels of height x width frames: unchanged
    when the short side already is `size`, else times float(new long side) / long side, the reference's own torch
    expression (the multiplication runs in FP32 on the boxes' device)."""
    boxes = boxes.detach().to(torch.float32).clone()
    Hs, Ws = resized_size(height, width, size)
    if (Hs, Ws) == (height, width):
        return boxes
    if width < height:
        boxes *= float(Hs) / height
    else:
        boxes *= float(Ws) / width
    return boxes


class Cv2Resize:
    """Device tables of the demo's resize of height x width frames to short side `size` (cv2_transform.scale): the y and
    x cv2_axis_table, uploaded once."""

    def __init__(self, height, width, size, device):
        self.H, self.W = int(height), int(width)
        self.Hs, self.Ws = resized_size(self.H, self.W, int(size))
        self.y = torch.from_numpy(cv2_axis_table(self.H, self.Hs, False).view(np.int32)).to(device)
        self.x = torch.from_numpy(cv2_axis_table(self.W, self.Ws, True).view(np.int32)).to(device)


def launch_resize_cv2(sources, destinations, resizes, channels):
    """esf_resize_u8_cv2 on the current stream: frame b at device address sources[b] (H, W, C) resized by resizes[b]
    (Cv2Resize) into destinations[b] (Hs, Ws, C), in one call."""
    B = len(sources)
    geom = (ctypes.c_int32 * (4 * B))(*[n for r in resizes for n in (r.H, r.W, r.Hs, r.Ws)])
    tables = (ctypes.c_void_p * (2 * B))(*[a for r in resizes for a in (r.y.data_ptr(), r.x.data_ptr())])
    rt.check(rt.lib().esf_resize_u8_cv2((ctypes.c_void_p * B)(*sources), (ctypes.c_void_p * B)(*destinations), geom,
                                        tables, B, channels, rt.current_stream_ptr()), "esf_resize_u8_cv2")


def launch_ava_boxes(boxes, crop, out):
    """esf_ava_boxes on the current stream: the loader's [0, 1] boxes (check_ava_boxes, on the device) to FP32 pixels of
    the crop.Hr x crop.Wr frames in `out` (K, 5)."""
    K = boxes.shape[0]
    assert boxes.is_cuda and boxes.is_contiguous() and out.shape == (K, 5) and out.dtype == torch.float32
    rt.check(rt.lib().esf_ava_boxes(boxes.data_ptr(), int(boxes.dtype == torch.float64), K, crop.H0, crop.W0, crop.Hr,
                                    crop.Wr, crop.S, out.data_ptr(), rt.current_stream_ptr()), "esf_ava_boxes")
