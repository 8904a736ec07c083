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

Frames at capture size (`scale_to=S`): the demo converts every captured frame with cv2.cvtColor(BGR2RGB) and resizes it
with datasets/cv2_transform.scale (cv2.resize INTER_LINEAR to short side S) before it enters the buffer.  Here the raw
frame is copied to a device staging area and esf_resize_u8_cv2 writes the resized frame, bit-identical to OpenCV's, into
its ring slot; the BGR order stays in the ring and the stem kernels read it through their channel table (`bgr=True`).
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
    """One camera's window.  With `scale_to=S` or `bgr=True` the frames are the camera's captures (height x width) and
    the window is a one-camera CameraWindows, which resizes them as the demo does (see CameraWindows)."""

    def __init__(self, model, cfg, height, width, channels=3, device=None, scale_to=None, bgr=False):
        self._bank = None
        if scale_to is not None or bgr:
            self._bank = CameraWindows(model, cfg, 1, height, width, channels, device=device, scale_to=scale_to,
                                       bgr=bgr)
            return
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
        if self._bank is not None:
            res = self._bank.push({0: frame})
            return None if res is None else res[1]
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


def box_rows(boxes, cameras, device):
    """(K, 5) FP32 rows [row, x1, y1, x2, y2] of the boxes of `cameras` (row r: cameras[r]) on the host when all of
    them are there, else on `device`, and the box count of every row."""
    on_host = all(boxes[c].device.type == "cpu" for c in cameras)
    where = torch.device("cpu") if on_host else device
    parts = [torch.cat([torch.full((boxes[c].shape[0], 1), float(r), device=where),
                        boxes[c].detach().to(device=where, dtype=torch.float32)], 1) for r, c in enumerate(cameras)]
    counts = [int(boxes[c].shape[0]) for c in cameras]
    return (torch.cat(parts) if parts else None), counts


def check_push(frames, boxes, clock, frame_shape, device, detection):
    """Validate the arguments of CameraWindows.push before anything is copied or launched (ValueError otherwise).
    `frame_shape`: the (H, W, C) of every camera's frames, or a list of one such shape per camera.  Returns the pushed
    camera ids (ascending), the ids that become rows, and for detection models the (K, 5) boxes of those rows (batch
    index = row) with the box count of every row."""
    if not isinstance(frames, dict):
        raise ValueError("push takes a dict {camera id: uint8 (H, W, C) frame}, got %s" % type(frames).__name__)
    n = len(clock.count)
    per_camera = isinstance(frame_shape, list)
    for cid, f in frames.items():
        if not _is_int(cid) or not 0 <= cid < n:
            raise ValueError("unknown camera id %r (cameras are 0 .. %d)" % (cid, n - 1))
        shape = tuple(frame_shape[cid] if per_camera else frame_shape)
        if not isinstance(f, torch.Tensor) or f.dtype != torch.uint8 or tuple(f.shape) != shape \
                or not f.is_contiguous():
            raise ValueError("camera %d: frames are contiguous uint8 tensors of shape %s, got %s" % (
                cid, shape, ("%s %s" % (f.dtype, tuple(f.shape))) if isinstance(f, torch.Tensor)
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
    rows, counts = box_rows(boxes, ready, device)
    return ids, ready, rows, counts


def _sizes(name, v, cameras, scaled):
    """`height` / `width` of CameraWindows as one int per camera."""
    if _is_int(v) and v >= 1:
        return [int(v)] * cameras
    if isinstance(v, (list, tuple)):
        if not scaled:
            raise ValueError("per-camera %s needs scale_to (cameras of one frame size share one bank)" % name)
        if len(v) != cameras or not all(_is_int(n) and n >= 1 for n in v):
            raise ValueError("%s: %d ints >= 1, one per camera, got %r" % (name, cameras, v))
        return [int(n) for n in v]
    raise ValueError("%s must be an int >= 1%s, got %r" % (name, " or one per camera" if scaled else "", v))


class _Bank:
    """The rings (n, L, H, W, C) of the cameras that share one frame size (ring i is cameras[i]'s), and the two pinned
    staging tables of their (ring, oldest slot) rows: one is filled while the other's copy may still be queued; each is
    refilled only after the event recorded behind its copy."""

    def __init__(self, cameras, seq_len, frame_shape, device):
        self.cameras, self.frame_shape, self.device = cameras, frame_shape, device
        self.ring = {c: i for i, c in enumerate(cameras)}
        self.bank = torch.zeros((len(cameras), seq_len) + frame_shape, dtype=torch.uint8, device=device)
        self._staging = [torch.empty((len(cameras), 2), dtype=torch.int32, pin_memory=True) for _ in range(2)]
        self._copied = [None, None]
        self._tick = 0

    def stage_rows(self, plan, table):
        """Copy the (ring, oldest slot) table through pinned staging to the family's device buffer on the current
        stream; returns the filled staging table and the device buffer."""
        k = self._tick % 2
        self._tick += 1
        if self._copied[k] is not None:
            self._copied[k].synchronize()       # recorded a tick ago: normally complete
        host = self._staging[k][:len(table)]
        host.copy_(torch.tensor(table, dtype=torch.int32))
        dev_rows = getattr(plan.shared, "camera_rows", None)
        if dev_rows is None or dev_rows.shape[0] < len(table):
            dev_rows = plan.shared.camera_rows = torch.empty((len(self.cameras), 2), dtype=torch.int32,
                                                             device=self.device)
        dev_rows[:len(table)].copy_(host, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._copied[k] = ev
        return host, dev_rows


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
    entry (K may be 0).  They run through the detection head as forward(clips, bboxes) does and come back per camera.

    Frames at capture size (`scale_to=S`, the demo's cfg.DATA.TEST_CROP_SIZE): `height` / `width` are the cameras'
    capture size, an int for every camera or a sequence of one int per camera.  Each pushed frame is resized as the demo's
    datasets/cv2_transform.scale does (cv2.resize INTER_LINEAR to short side S, bit for bit) when it enters its ring, so
    the rings hold what the demo's frame buffer holds.  Cameras of one scaled size share one bank (n_g, L, Hs, Ws, C);
    a push copies the host frames to a device staging area (one frame per camera), makes one resize launch
    (esf_resize_u8_cv2) for all of them, then runs one forward per bank that has rows, as above (without MAX_BATCH a bank
    pads to its own n_g rows, and 0 < MAX_BATCH < n_g is refused).  The results are merged in ascending camera id.
    Detection boxes are in capture pixels and are scaled as cv2_transform.scale_boxes does.  Every scaled size needs its
    plan, so more distinct scaled sizes than cfg.ESF.MAX_PLANS are refused; so are C = 2 and per-camera sizes without
    scale_to.  `bgr=True`: the frames are BGR (cv2.VideoCapture's order, which the demo converts with
    cv2.cvtColor(BGR2RGB)); the stem kernels read them in RGB order through their channel table, with no extra pass."""

    def __init__(self, model, cfg, cameras, height, width, channels=3, stride=1, device=None, scale_to=None,
                 bgr=False):
        for name, v in (("cameras", cameras), ("channels", channels), ("stride", stride)):
            if not _is_int(v) or v < 1:
                raise ValueError("%s must be an int >= 1, got %r" % (name, v))
        scaled = scale_to is not None
        if scaled and (not _is_int(scale_to) or scale_to < 1):
            raise ValueError("scale_to must be an int >= 1 (the demo's DATA.TEST_CROP_SIZE), got %r" % (scale_to,))
        heights, widths = _sizes("height", height, cameras, scaled), _sizes("width", width, cameras, scaled)
        if channels > 4:
            raise ValueError("the frame kernels take up to 4 channels, got %d" % channels)
        if scaled and channels == 2:
            raise ValueError("scale_to takes frames of 1, 3 or 4 channels: OpenCV resizes an exact 2x downscale of 2 "
                             "channels with INTER_AREA, which the resize kernel does not restate")
        if scaled and max(widths) * channels > esf_frames.MAX_ROW_BYTES:
            raise ValueError("capture rows of %d x %d bytes exceed the resize kernel's %d"
                             % (max(widths), channels, esf_frames.MAX_ROW_BYTES))
        if bgr and channels != 3:
            raise ValueError("bgr=True swaps the channels of 3-channel frames, got %d channels" % channels)
        capture = [(h, w, int(channels)) for h, w in zip(heights, widths)]
        shapes = [esf_frames.resized_size(h, w, int(scale_to)) + (c,) for h, w, c in capture] if scaled else capture
        distinct = list(dict.fromkeys(shapes))
        max_plans = int(getattr(model, "_max_plans", 1))
        if len(distinct) > max_plans:
            raise ValueError("the cameras scale to %d frame sizes %s, each with its own plan, and cfg.ESF.MAX_PLANS = %d "
                             "keeps %d: every tick would evict and recompile a plan" % (len(distinct), distinct,
                                                                                       max_plans, max_plans))
        largest = max(shapes.count(sh) for sh in distinct)
        cap = int(getattr(model, "_max_batch", 0) or 0)
        if 0 < cap < largest:
            raise ValueError("cfg.ESF.MAX_BATCH = %d is less than the %d cameras of the bank" % (cap, largest))
        device = torch.device(device) if device is not None else next(model.parameters()).device
        if device.type != "cuda":
            raise rt.EsfError("CameraWindows needs a CUDA device; there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.model, self.device, self.cameras = model, device, int(cameras)
        self.padded = cap == 0
        self.detection = bool(getattr(model, "enable_detection", False))
        self.scale_to, self.bgr = (int(scale_to) if scaled else None), bool(bgr)
        self.seq_len = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.get("SAMPLING_RATE", 1) if hasattr(cfg.DATA, "get")
                                                      else cfg.DATA.SAMPLING_RATE)
        alpha = int(cfg.SLOWFAST.ALPHA) if model.num_pathways > 1 else None
        self.positions = window_indices(self.seq_len, int(cfg.DATA.NUM_FRAMES), alpha)
        self.banks = [_Bank([c for c in range(self.cameras) if shapes[c] == sh], self.seq_len, sh, device)
                      for sh in distinct]
        self._bank_of = [next(b for b in self.banks if c in b.ring) for c in range(self.cameras)]
        if scaled:
            self.frame_shape = capture           # what push takes: one capture shape per camera
            tables = {hw: esf_frames.Cv2Resize(hw[0], hw[1], self.scale_to, device) for hw in dict.fromkeys(
                (h, w) for h, w, _ in capture)}
            self._resize = [tables[(h, w)] for h, w, _ in capture]
            self._offsets, size = esf_frames.arena_layout(capture)
            self._staged = torch.empty(size, dtype=torch.uint8, device=device)
        else:
            self.frame_shape = capture[0]
            self.bank = self.banks[0].bank
        self.clock = CameraClock(self.cameras, self.seq_len, int(stride))
        self._pos = [(p.to(torch.int32).to(device), (ctypes.c_int32 * p.numel())(*p.tolist())) for p in self.positions]

    def push(self, frames, boxes=None):
        """frames: {camera id: uint8 (H, W, C) frame}, host (pinned for asynchronous copies) or on the bank's device.
        Returns (camera_ids, scores) for the cameras that became rows: scores (R, num_classes), row r for
        camera_ids[r]; for detection models a list of (K_r, num_classes) per camera.  None when no camera is ready.
        Every argument is checked before anything is copied or launched."""
        if self.model.training:
            raise NotImplementedError("eval-mode forward path only")
        ids, ready, box_rows_all, counts_all = check_push(frames, boxes, self.clock, self.frame_shape, self.device,
                                                          self.detection)
        dev = self.device
        with torch.cuda.device(dev):
            if self.scale_to is None:
                for cid in ids:
                    self.bank[cid, self.clock.slot(cid)].copy_(frames[cid], non_blocking=True)
            elif ids:
                self._resize_into_rings(frames, ids)
            rows = self.clock.advance(ids)
            assert [c for c, _ in rows] == ready
            if not rows:
                return None
            if self.scale_to is None:
                return ready, self._forward(self.banks[0], rows, box_rows_all, counts_all)
            oldest = dict(rows)
            order, parts = [], []
            for bank in self.banks:
                cams = [c for c in ready if c in bank.ring]
                if not cams:
                    continue
                br = counts = None
                if self.detection:
                    scaled = {c: esf_frames.scale_boxes(self.scale_to, boxes[c], *self.frame_shape[c][:2]) for c in cams}
                    br, counts = box_rows(scaled, cams, dev)
                parts.append(self._forward(bank, [(bank.ring[c], oldest[c]) for c in cams], br, counts))
                order += cams
            if self.detection:
                by_camera = dict(zip(order, [s for p in parts for s in p]))
                return ready, [by_camera[c] for c in ready]
            scores = torch.cat(parts) if len(parts) > 1 else parts[0]
            if order != ready:
                scores = scores[torch.tensor([order.index(c) for c in ready], device=dev)]
            return ready, scores

    def _resize_into_rings(self, frames, ids):
        """Stage the host frames of `ids` on the device (one cudaMemcpyAsync each; device frames are read in place) and
        resize all of them into their ring slots with one esf_resize_u8_cv2 call."""
        sources, destinations = [], []
        for cid in ids:
            f = frames[cid]
            if f.device.type == "cpu":
                staged = self._staged[self._offsets[cid]:self._offsets[cid] + f.numel()]
                staged.copy_(f.view(-1), non_blocking=True)
                f = staged
            sources.append(f.data_ptr())
            bank = self._bank_of[cid]
            destinations.append(bank.bank[bank.ring[cid], self.clock.slot(cid)].data_ptr())
        esf_frames.launch_resize_cv2(sources, destinations, [self._resize[c] for c in ids], self.banks[0].frame_shape[2])

    def _forward(self, bank, rows, box_rows_, counts):
        """One forward of `bank`'s (ring, oldest slot) rows: scores (R, num_classes), or per-row lists for detection."""
        dev = self.device
        R = len(rows)
        if self.detection and sum(counts) == 0:
            empty = self.model._empty(dev)
            return [empty for _ in rows]
        table = rows + [rows[0]] * ((len(bank.cameras) if self.padded else R) - R)
        H, W, C = bank.frame_shape
        shapes = [(len(table), C, int(p.numel()), H, W) for p in self.positions]
        plan, fin = self.model._frame_plan(shapes, dev, C)
        host, dev_rows = bank.stage_rows(plan, table)
        out = plan.run_frames(lambda: esf_frames.launch_rings(plan, fin, bank.bank, (dev_rows, host), self._pos,
                                                              self.bgr))
        if not self.detection:
            return self.model._finish(plan, out[:R], None)
        out = self.model._finish(plan, out, self.model._boxes(box_rows_, len(table), dev))
        return list(torch.split(out, counts))
