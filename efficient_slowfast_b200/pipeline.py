"""Host -> device -> host streaming of clip batches around the forward path.

The reference's test loop (SlowFast/tools/test_net.py:58-110) is strictly serial per batch: `inputs[i].cuda()`,
`model(inputs)`, `all_gather`, `.cpu()`.  A batch of 64 clips is 1.5 GB of FP32 pixels, i.e. ~30 ms of PCIe time next to
a ~45 ms forward, so serialising the two wastes 40 % of the wall clock.  `ClipStream` keeps the same per-batch contract
(every batch is copied from pinned host memory, run through `model.forward`, and its predictions copied back to the
host) but double-buffers the device staging tensors and issues the H2D copy of batch i+1 on a copy stream while batch i
computes.  Results are returned in submission order.

    stream = ClipStream(model, shapes)            # shapes of [slow, fast]
    for host_inputs in loader:                    # pinned FP32 tensors
        done = stream.submit(host_inputs)         # -> (index, preds) of an EARLIER batch, or None while filling
    for index, preds in stream.flush(): ...
"""
import math

import torch

from . import distributed as esf_dist
from . import runtime as rt


class ClipStream:
    def __init__(self, model, shapes, device=None, depth=2, gather=False, frames=False, slow_from_fast=False,
                 crop_size=None, spatial_idx=None, num_clips=None):
        """`depth` staging slots (>= 2 overlaps copy and compute); `gather=True` all-gathers the predictions over the
        process group before the D2H copy, like the reference's test loop.  `frames=True`: every batch is ONE pinned
        uint8 tensor of decoded frames (B, T, H, W, C) (`shapes` = [that shape]) and goes through
        `model.forward_frames` -- normalisation and pathway packing on the device, 1/5 of the H2D bytes.
        With `crop_size` / `spatial_idx` (test-time crops of frames at decode size) a batch may also be a list of at
        most B pinned uint8 clips (T, H_b, W_b, C) of mixed decode sizes: they are copied to 16-byte aligned offsets
        of the same staging slot (frames.arena_layout; its B * T * H * W * C bytes are the capacity) and run as
        `model.forward_frames(list)`.
        Video mode, `num_clips` given (frames=True, `shapes` = [(n_max, N_max, H, W, C)]): every batch is a list of at
        most n_max pinned uint8 videos (N_v, H_v, W_v, C), copied one `copy_` each to 16-byte aligned offsets of a
        staging slot of n_max * N_max * H * W * C bytes (frames.arena_layout), and run as `model.forward_videos` with
        `num_clips` temporal views (e.g. TEST.NUM_ENSEMBLE_VIEWS) and the crops of `crop_size` / `spatial_idx`
        (defaults as there); `submit(videos, fps=...)` gives the frame rates.
        `slow_from_fast=True`: the caller vouches that every batch is what the reference's loader produces,
        `[slow, fast] = pack_pathway_output(cfg, fast)` (datasets/utils.py:93-102: slow = the linspace frame subset of
        fast).  Only the fast clip is then copied to the device and the slow pathway's stem reads its frames out of it
        (`model.forward_fast`): 1/(1 + 1/ALPHA) of the H2D bytes.  The first batch is verified on the host."""
        if getattr(model, "enable_detection", False):
            raise NotImplementedError("ClipStream streams clip batches into classification models; call a detection "
                                      "model (cfg.DETECTION.ENABLE) as model(inputs, bboxes)")
        device = torch.device(device) if device is not None else next(model.parameters()).device
        if device.type != "cuda":
            raise rt.EsfError("ClipStream needs a CUDA device; there is no CPU fallback")
        assert depth >= 1
        self.model, self.device, self.depth, self.gather = model, device, depth, gather
        self.copy_stream = torch.cuda.Stream(device=device)
        self.frames = bool(frames)
        assert not self.frames or len(shapes) == 1
        self.crop = None
        self.videos = None
        if num_clips is not None:
            if not self.frames:
                raise ValueError("ClipStream: num_clips (video mode) needs frames=True")
            from . import frames as esf_frames
            cfg = model._cfg
            esf_frames.check_videos([], 1.0, num_clips)
            views = esf_frames.spatial_views(esf_frames.ensemble_spatial_views(cfg.TEST.NUM_SPATIAL_CROPS)
                                             if spatial_idx is None else spatial_idx)
            size = int(cfg.DATA.TEST_CROP_SIZE if crop_size is None else crop_size)
            esf_frames.view_shapes(tuple(shapes[0]), size, views)    # ValueError now rather than at the first batch
            self.videos = {"num_clips": int(num_clips), "spatial_idx": views, "crop_size": size}
        elif crop_size is not None or spatial_idx is not None:
            if not self.frames:
                raise ValueError("ClipStream: crop_size / spatial_idx need frames=True")
            from . import frames as esf_frames
            views = esf_frames.spatial_views(1 if spatial_idx is None else spatial_idx)
            size = int(model._cfg.DATA.TEST_CROP_SIZE if crop_size is None else crop_size)
            esf_frames.view_shapes(tuple(shapes[0]), size, views)    # ValueError now rather than at the first batch
            self.crop = {"crop_size": size, "spatial_idx": views}
        self.slow_from_fast = bool(slow_from_fast) and not self.frames and len(shapes) == 2
        self._sff_checked = False
        if self.slow_from_fast:
            shapes = [shapes[1]]            # staging holds the fast clip only
        dt = torch.uint8 if self.frames else torch.float32
        self.stage = [[torch.empty(tuple(s), dtype=dt, device=device) for s in shapes] for _ in range(depth)]
        self.ready = [torch.cuda.Event() for _ in range(depth)]     # H2D of the slot finished
        self.consumed = [torch.cuda.Event() for _ in range(depth)]  # forward no longer reads the slot
        self.done = [torch.cuda.Event() for _ in range(depth)]      # predictions of the slot are on the host
        self.host_out = [None] * depth
        self.pending = []   # (index, slot) in flight, oldest first
        self.n = 0
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.stage[0])

    def submit(self, host_inputs, fps=None):
        """Queue one batch (list of pinned host tensors, reference order [slow, fast]; in video mode a list of videos
        and their `fps`).  Never blocks on the batch just queued; when all staging slots are busy it first waits for
        the oldest batch and returns its (index, preds)."""
        if fps is not None and self.videos is None:
            raise ValueError("ClipStream.submit: fps is for video mode (ClipStream(..., num_clips=...))")
        if self.videos is not None:     # every check before a slot is waited for or a copy is queued
            video_views = self._video_views(host_inputs, fps)
        finished = None
        if len(self.pending) == self.depth:
            finished = self._pop()
        slot = self.n % self.depth
        cur = torch.cuda.current_stream(self.device)
        # A loader with drop_last=False (the reference's test loader, datasets/loader.py) ends on a SHORT batch: it is
        # copied into the leading rows of the staging slot (a leading-dim slice of a contiguous tensor is contiguous)
        # and the forward runs on those views -- the model compiles a second plan for that batch size and keeps both
        # (with cfg.ESF.MAX_BATCH, a variant of the same plan family, on the same arena).
        if self.slow_from_fast:
            if len(host_inputs) == 2:
                if not self._sff_checked:   # once: the promise the flag makes
                    T = host_inputs[1].shape[2]
                    idx = torch.linspace(0, T - 1, host_inputs[0].shape[2]).long()
                    if not torch.equal(host_inputs[0], host_inputs[1].index_select(2, idx)):
                        raise rt.EsfError("ClipStream(slow_from_fast=True): the slow clip is not the linspace frame "
                                          "subset of the fast clip (pack_pathway_output)")
                    self._sff_checked = True
                host_inputs = host_inputs[1:]
        if self.videos is not None:
            clips = video_views(self.stage[slot][0])
            copies, views = list(zip(host_inputs, clips)), [clips]
        elif self.crop is not None and host_inputs and all(h.dim() == 4 for h in host_inputs):
            clips = self._clip_views(host_inputs, self.stage[slot][0])   # clips of mixed decode sizes
            copies, views = list(zip(host_inputs, clips)), [clips]
        else:
            views = []
            for h, d in zip(host_inputs, self.stage[slot]):
                if tuple(h.shape[1:]) != tuple(d.shape[1:]) or h.shape[0] > d.shape[0] or h.shape[0] == 0:
                    raise rt.EsfError("ClipStream was built for batches of shape <= %s, got %s"
                                      % (tuple(d.shape), tuple(h.shape)))
                views.append(d if h.shape[0] == d.shape[0] else d[:h.shape[0]])
            copies = list(zip(host_inputs, views))
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.consumed[slot])
            for h, d in copies:
                d.copy_(h, non_blocking=True)
            self.ready[slot].record(self.copy_stream)
        cur.wait_event(self.ready[slot])
        if self.videos is not None:
            out = self.model.forward_videos(views[0], fps=fps, **self.videos)
        elif self.frames:
            out = self.model.forward_frames(views[0], **(self.crop or {}))
        elif self.slow_from_fast:
            out = self.model.forward_fast(views[0])
        else:
            out = self.model(views)
        self.consumed[slot].record(cur)
        if self.gather:
            out = esf_dist.all_gather([out])[0]
        if self.host_out[slot] is None or self.host_out[slot].shape[0] < out.shape[0] \
                or self.host_out[slot].shape[1:] != out.shape[1:]:
            self.host_out[slot] = torch.empty(out.shape, dtype=out.dtype).pin_memory()
        self.host_out[slot][:out.shape[0]].copy_(out, non_blocking=True)
        self.done[slot].record(cur)
        self.pending.append((self.n, slot, out.shape[0]))
        self.n += 1
        return finished

    def _clip_views(self, clips, stage):
        """Views of the staging slot `stage` (B, T, H, W, C) that a list of clips (T, H_b, W_b, C) is copied to, at the
        offsets of frames.arena_layout.  ValueError / EsfError before any copy when the clips are not a valid list
        (frames.check_clips, crops that do not fit) or exceed the slot's B clips or its bytes."""
        from . import frames as esf_frames
        if len(clips) > stage.shape[0]:
            raise rt.EsfError("ClipStream was built for batches of at most %d clips, got %d" % (stage.shape[0], len(clips)))
        sizes = esf_frames.check_clips(clips)
        esf_frames.view_shapes(sizes, self.crop["crop_size"], self.crop["spatial_idx"])
        flat = stage.view(-1)
        offsets, _ = esf_frames.arena_layout(sizes, flat.numel())
        return [flat[o:o + math.prod(sh)].view(sh) for o, sh in zip(offsets, sizes)]

    def _video_views(self, videos, fps):
        """Checks a list of videos (N, H, W, C) for video mode and returns the function that gives, for a staging
        slot, the views they are copied to at the offsets of frames.arena_layout.  ValueError / EsfError before any
        copy when the list is not valid for forward_videos or exceeds the slot's n_max videos or its bytes."""
        from . import frames as esf_frames
        stage = self.stage[0][0]
        videos = list(videos)
        if len(videos) > stage.shape[0]:
            raise rt.EsfError("ClipStream was built for batches of at most %d videos, got %d"
                              % (stage.shape[0], len(videos)))
        cfg = self.model._cfg
        sizes, _ = esf_frames.check_videos(videos, 1.0 if fps is None else fps, self.videos["num_clips"])
        if sizes:
            esf_frames.view_shapes([(cfg.DATA.NUM_FRAMES,) + sh[1:] for sh in sizes], self.videos["crop_size"],
                                   self.videos["spatial_idx"])
        offsets, _ = esf_frames.arena_layout(sizes, stage.numel())
        return lambda slot_stage: [slot_stage.view(-1)[o:o + math.prod(sh)].view(sh) for o, sh in zip(offsets, sizes)]

    def _pop(self):
        index, slot, rows = self.pending.pop(0)
        self.done[slot].synchronize()
        return index, self.host_out[slot][:rows].clone()

    def flush(self):
        """Wait for every batch still in flight; returns their (index, preds) in submission order."""
        out = []
        while self.pending:
            out.append(self._pop())
        return out
