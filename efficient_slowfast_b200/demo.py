"""Sliding-window inference over a frame stream -- the loop of the reference's `tools/demo_net.py:153-305` without its
per-window host work.

The reference keeps the last `NUM_FRAMES * SAMPLING_RATE` frames in a Python list and, once it is full, for EVERY new
frame: stacks the list into one tensor, normalises it on the host (`tensor_normalize`), permutes, picks the fast
pathway's frames with `linspace(0, L-1, NUM_FRAMES).long()` and the slow pathway's with a second `linspace` over those
(demo_net.py:198-224), copies both pathways to the GPU and runs the model; then it drops the oldest frame.

Here the window is a ring of uint8 frames that lives on the device: a new frame costs one H2D copy of H*W*C bytes into
its slot, and the two pathway selections are index arrays into the ring (`model.forward_frames(frame_index=...)`), so
normalisation, layout change and both gathers happen inside the stem-pack kernel and nothing is re-assembled.

A deployment watches many cameras.  `CameraWindows` keeps one such ring per camera in a bank (N, L, H, W, C) and runs
one batched forward per tick for every camera whose window is ready; the kernels read each row's frames out of its
camera's ring (esf_*_rings), so a tick uploads the pushed frames and an 8-byte (camera, oldest slot) pair per row.
"""
import ctypes
import numbers

import torch

from . import frames as esf_frames
from . import runtime as rt


def window_indices(seq_len, num_frames, alpha=None):
    """demo_net.py:203-224: positions (inside the window, oldest frame = 0) of the fast / single pathway's frames, and of
    the slow pathway's frames when `alpha` is given."""
    fast = torch.linspace(0, seq_len - 1, num_frames).long()
    if alpha is None:
        return [fast]
    slow = fast.index_select(0, torch.linspace(0, fast.shape[0] - 1, fast.shape[0] // alpha).long())
    return [slow, fast]


class SlidingWindow:
    def __init__(self, model, cfg, height, width, channels=3, device=None):
        device = torch.device(device) if device is not None else next(model.parameters()).device
        if device.type != "cuda":
            raise rt.EsfError("SlidingWindow needs a CUDA device; there is no CPU fallback")
        self.model, self.device = model, device
        self.seq_len = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.get("SAMPLING_RATE", 1) if hasattr(cfg.DATA, "get")
                                                      else cfg.DATA.SAMPLING_RATE)
        alpha = int(cfg.SLOWFAST.ALPHA) if model.num_pathways > 1 else None
        self.positions = window_indices(self.seq_len, int(cfg.DATA.NUM_FRAMES), alpha)
        self.ring = torch.zeros((1, self.seq_len, height, width, channels), dtype=torch.uint8, device=device)
        self.count = 0          # frames pushed so far

    def push(self, frame):
        """frame: uint8 (H, W, C) tensor, host (pinned for an asynchronous copy) or device.  Returns the model output
        (1, num_classes) for the window that ends with this frame, or None while the window is filling."""
        assert frame.dtype == torch.uint8 and tuple(frame.shape) == tuple(self.ring.shape[2:])
        self.ring[0, self.count % self.seq_len].copy_(frame, non_blocking=True)
        self.count += 1
        if self.count < self.seq_len:
            return None
        oldest = self.count % self.seq_len          # ring slot of window position 0
        index = [((p + oldest) % self.seq_len).to(torch.int32).to(self.device) for p in self.positions]
        return self.model.forward_frames(self.ring, frame_index=index)


class CameraClock:
    """Host bookkeeping of CameraWindows: the push count of every camera, the ring slot its next frame goes to, and the
    cameras that become rows.  A camera's window holds its last `seq_len` frames; once full, the camera is a row after
    every `stride`-th push (stride 1: a prediction for every frame, as the reference demo)."""

    def __init__(self, cameras, seq_len, stride):
        self.seq_len, self.stride = seq_len, stride
        self.count = [0] * cameras

    def slot(self, camera):
        """Ring slot of the camera's next frame."""
        return self.count[camera] % self.seq_len

    def ready_after_push(self, camera):
        c = self.count[camera] + 1
        return c >= self.seq_len and (c - self.seq_len) % self.stride == 0

    def advance(self, cameras):
        """Count one push of each of `cameras` (ascending ids); returns the rows [(camera, oldest slot)] they make."""
        rows = []
        for c in cameras:
            ready = self.ready_after_push(c)
            self.count[c] += 1
            if ready:
                rows.append((c, self.count[c] % self.seq_len))
        return rows


def _is_int(v):
    return isinstance(v, numbers.Integral) and not isinstance(v, bool)


def check_push(frames, boxes, clock, frame_shape, device, detection):
    """Validate the arguments of CameraWindows.push before anything is copied or launched (ValueError otherwise).
    Returns the pushed camera ids (ascending), the ids that become rows, and for detection models the (K, 5) boxes of
    those rows (batch index = row) with the box count of every row."""
    if not isinstance(frames, dict):
        raise ValueError("push takes a dict {camera id: uint8 (H, W, C) frame}, got %s" % type(frames).__name__)
    n = len(clock.count)
    for cid, f in frames.items():
        if not _is_int(cid) or not 0 <= cid < n:
            raise ValueError("unknown camera id %r (cameras are 0 .. %d)" % (cid, n - 1))
        if not isinstance(f, torch.Tensor) or f.dtype != torch.uint8 or tuple(f.shape) != tuple(frame_shape) \
                or not f.is_contiguous():
            raise ValueError("camera %d: frames are contiguous uint8 tensors of shape %s, got %s" % (
                cid, tuple(frame_shape), ("%s %s" % (f.dtype, tuple(f.shape))) if isinstance(f, torch.Tensor)
                else type(f).__name__))
        if f.device.type != "cpu" and f.device != device:
            raise ValueError("camera %d: frame on %s; frames are on the host or on the bank's device %s"
                             % (cid, f.device, device))
    ids = sorted(int(c) for c in frames)
    ready = [c for c in ids if clock.ready_after_push(c)]
    if not detection:
        if boxes is not None:
            raise ValueError("boxes are for detection models (cfg.DETECTION.ENABLE)")
        return ids, ready, None, None
    if not isinstance(boxes, dict):
        raise ValueError("a detection model's push needs boxes={camera id: (K, 4) boxes} for every ready camera")
    for cid, b in boxes.items():
        if not _is_int(cid) or int(cid) not in frames:
            raise ValueError("boxes for camera %r, which this push gives no frame" % (cid,))
        if not torch.is_tensor(b) or not b.is_floating_point() or b.dim() != 2 or b.shape[1] != 4:
            raise ValueError("camera %d: boxes are a floating-point (K, 4) tensor [x1, y1, x2, y2] in frame pixels, got "
                             "%s" % (cid, (tuple(b.shape), b.dtype) if torch.is_tensor(b) else type(b).__name__))
        if b.device.type != "cpu" and b.device != device:
            raise ValueError("camera %d: boxes on %s; boxes are on the host or on %s" % (cid, b.device, device))
    missing = [c for c in ready if c not in boxes]
    if missing:
        raise ValueError("cameras %s have a full window and no boxes" % missing)
    on_host = all(boxes[c].device.type == "cpu" for c in ready)
    where = torch.device("cpu") if on_host else device
    parts = [torch.cat([torch.full((boxes[c].shape[0], 1), float(r), device=where),
                        boxes[c].detach().to(device=where, dtype=torch.float32)], 1) for r, c in enumerate(ready)]
    counts = [int(boxes[c].shape[0]) for c in ready]
    return ids, ready, (torch.cat(parts) if parts else None), counts


class CameraWindows:
    """The reference demo's sliding window (tools/demo_net.py) over many cameras with one batched forward per tick.

    The bank `(cameras, L, height, width, channels)` uint8 on the device holds every camera's ring of its last
    L = NUM_FRAMES * SAMPLING_RATE frames.  `push({camera id: frame})` copies each frame into its camera's slot (one
    cudaMemcpyAsync per frame; host frames should be pinned), and every pushed camera whose window is full and whose
    pushes since it filled are a multiple of `stride` becomes a row.  The rows, in ascending camera id, run through one
    forward whose stem kernels read each row's frames out of its ring on the device (esf_stem_pack_u8_rings /
    esf_frames_to_clip_rings): row r holds what `SlidingWindow` of that camera would give for the same frames.

    The plan for R rows is the plan of `forward_frames(frames, frame_index=...)` on R stacked clips, so the bank,
    SlidingWindow and forward_frames share plans.  With cfg.ESF.MAX_BATCH >= cameras, R rows run the family's variant
    for R (one arena and one weight pack for every R).  Without it every tick is padded to `cameras` rows so that one
    plan serves all ticks: padding rows repeat row 0 and are dropped from the result, which costs a forward of
    `cameras` rows when fewer are ready (the whole bank's compute on every tick of a partly ready bank).
    0 < MAX_BATCH < cameras is refused.

    Detection models (cfg.DETECTION.ENABLE): `push(frames, boxes={camera id: (K, 4) boxes})`, the person boxes the
    reference demo's detector gives for the window, in pixels of the frames; every camera that becomes a row needs an
    entry (K may be 0).  They run through the detection head as forward(clips, bboxes) does and come back per camera."""

    def __init__(self, model, cfg, cameras, height, width, channels=3, stride=1, device=None):
        for name, v in (("cameras", cameras), ("height", height), ("width", width), ("channels", channels),
                        ("stride", stride)):
            if not _is_int(v) or v < 1:
                raise ValueError("%s must be an int >= 1, got %r" % (name, v))
        if channels > 4:
            raise ValueError("the frame kernels take up to 4 channels, got %d" % channels)
        device = torch.device(device) if device is not None else next(model.parameters()).device
        if device.type != "cuda":
            raise rt.EsfError("CameraWindows needs a CUDA device; there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        cap = int(getattr(model, "_max_batch", 0) or 0)
        if 0 < cap < cameras:
            raise ValueError("cfg.ESF.MAX_BATCH = %d is less than the %d cameras of the bank" % (cap, cameras))
        self.model, self.device, self.cameras = model, device, int(cameras)
        self.padded = cap == 0
        self.detection = bool(getattr(model, "enable_detection", False))
        self.seq_len = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.get("SAMPLING_RATE", 1) if hasattr(cfg.DATA, "get")
                                                      else cfg.DATA.SAMPLING_RATE)
        alpha = int(cfg.SLOWFAST.ALPHA) if model.num_pathways > 1 else None
        self.positions = window_indices(self.seq_len, int(cfg.DATA.NUM_FRAMES), alpha)
        self.frame_shape = (int(height), int(width), int(channels))
        self.bank = torch.zeros((self.cameras, self.seq_len) + self.frame_shape, dtype=torch.uint8, device=device)
        self.clock = CameraClock(self.cameras, self.seq_len, int(stride))
        self._pos = [(p.to(torch.int32).to(device), (ctypes.c_int32 * p.numel())(*p.tolist())) for p in self.positions]
        # two pinned staging tables: one is filled while the other's copy may still be queued; each is refilled only
        # after the event recorded behind its copy
        self._staging = [torch.empty((self.cameras, 2), dtype=torch.int32, pin_memory=True) for _ in range(2)]
        self._copied = [None, None]
        self._tick = 0

    def push(self, frames, boxes=None):
        """frames: {camera id: uint8 (H, W, C) frame}, host (pinned for asynchronous copies) or on the bank's device.
        Returns (camera_ids, scores) for the cameras that became rows: scores (R, num_classes), row r for
        camera_ids[r]; for detection models a list of (K_r, num_classes) per camera.  None when no camera is ready.
        Every argument is checked before anything is copied or launched."""
        if self.model.training:
            raise NotImplementedError("eval-mode forward path only")
        ids, ready, box_rows, counts = check_push(frames, boxes, self.clock, self.frame_shape, self.device,
                                                  self.detection)
        dev = self.device
        with torch.cuda.device(dev):
            for cid in ids:
                self.bank[cid, self.clock.slot(cid)].copy_(frames[cid], non_blocking=True)
            rows = self.clock.advance(ids)
            assert [c for c, _ in rows] == ready
            if not rows:
                return None
            R = len(rows)
            if self.detection and sum(counts) == 0:
                empty = self.model._empty(dev)
                return ready, [empty for _ in ready]
            table = rows + [rows[0]] * ((self.cameras if self.padded else R) - R)
            shapes = [(len(table), self.frame_shape[2], int(p.numel())) + self.frame_shape[:2] for p in self.positions]
            plan, fin = self.model._frame_plan(shapes, dev, self.frame_shape[2])
            host, dev_rows = self._stage_rows(plan, table)
            out = plan.run_frames(lambda: esf_frames.launch_rings(plan, fin, self.bank, (dev_rows, host), self._pos))
            if not self.detection:
                return ready, self.model._finish(plan, out[:R], None)
            out = self.model._finish(plan, out, self.model._boxes(box_rows, len(table), dev))
            return ready, list(torch.split(out, counts))

    def _stage_rows(self, plan, table):
        """Copy the (camera, oldest slot) table through pinned staging to the family's device buffer on the current
        stream; returns the filled staging table and the device buffer."""
        k = self._tick % 2
        self._tick += 1
        if self._copied[k] is not None:
            self._copied[k].synchronize()       # recorded a tick ago: normally complete
        host = self._staging[k][:len(table)]
        host.copy_(torch.tensor(table, dtype=torch.int32))
        dev_rows = getattr(plan.shared, "camera_rows", None)
        if dev_rows is None or dev_rows.shape[0] < len(table):
            dev_rows = plan.shared.camera_rows = torch.empty((self.cameras, 2), dtype=torch.int32, device=self.device)
        dev_rows[:len(table)].copy_(host, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._copied[k] = ev
        return host, dev_rows
