"""The caller of the forward path: multi-view test loop and view ensembling (SURVEY.md section 8(f) row 1).

Mirrors the interface of the reference's `TestMeter` (SlowFast/slowfast/utils/meters.py:216-372) and `perform_test`
(SlowFast/tools/test_net.py:21-123) for the classification case, re-designed for this path:
  * the ensemble update is vectorised (`index_add_` / `scatter_reduce_(amax)` over the whole batch) instead of a
    Python loop over clips;
  * the loop feeds `ClipStream`, so the H2D copy of batch i+1 overlaps the forward of batch i and the meter is updated
    with the predictions of an EARLIER batch while the GPU keeps running (results come back in submission order, so
    labels / video indices are queued alongside);
  * multi-GPU: predictions are all-gathered on the device inside ClipStream, labels and clip indices with the same
    collective (`distributed.all_gather`), as `du.all_gather([preds, labels, video_idx])` does in the reference.
Detection (cfg.DETECTION.ENABLE) follows the reference's branch: `model(inputs, meta["boxes"])` per batch, the caller's
meter (the reference's AVAMeter) gets `update_stats(preds, ori_boxes, metadata)`; the AVA mAP evaluation is the meter's
own business.  Multi-label mAP of TestMeter is out of scope (SURVEY.md section 8)."""
import time

import torch

from . import distributed as esf_dist
from .pipeline import ClipStream


def topks_correct(preds, labels, ks):
    """Number of samples whose label is among the top-k predictions, for every k (utils/metrics.py:9-42)."""
    assert preds.size(0) == labels.size(0), "Batch dim of predictions and labels must match"
    top = torch.topk(preds, max(ks), dim=1, largest=True, sorted=True).indices   # (N, max_k)
    hit = top.eq(labels.view(-1, 1))
    return [hit[:, :k].float().sum() for k in ks]


class TestMeter:
    """Multi-view ensemble: every video is sampled as `num_clips` clips (ids video * num_clips + view); their
    predictions are summed (or max-ed) into one video-level prediction and scored against the label."""

    __test__ = False   # not a pytest class

    def __init__(self, num_videos, num_clips, num_cls, overall_iters, multi_label=False, ensemble_method="sum"):
        if multi_label:
            raise NotImplementedError("multi-label (mAP) testing is out of scope")
        if ensemble_method not in ("sum", "max"):
            raise NotImplementedError("Ensemble Method {} is not supported".format(ensemble_method))
        self.num_clips, self.overall_iters, self.ensemble_method = num_clips, overall_iters, ensemble_method
        self.multi_label = False
        self.video_preds = torch.zeros((num_videos, num_cls))
        self.video_labels = torch.zeros((num_videos,)).long()
        self.clip_count = torch.zeros((num_videos,)).long()
        self._tic = time.perf_counter()
        self._elapsed = 0.0
        self.stats = None

    def reset(self):
        self.clip_count.zero_()
        self.video_preds.zero_()
        self.video_labels.zero_()

    def update_stats(self, preds, labels, clip_ids):
        """preds (N, C), labels (N,), clip_ids (N,): whole-batch ensemble update."""
        preds, labels = preds.detach().cpu().float(), labels.detach().cpu().long()
        vid = torch.div(clip_ids.detach().cpu().long(), self.num_clips, rounding_mode="floor")
        seen = self.video_labels[vid]
        assert bool(((seen == 0) | (seen == labels)).all()), "clips of one video disagree on its label"
        self.video_labels[vid] = labels
        if self.ensemble_method == "sum":
            self.video_preds.index_add_(0, vid, preds)
        else:
            self.video_preds.scatter_reduce_(0, vid.view(-1, 1).expand_as(preds), preds, reduce="amax",
                                             include_self=True)
        self.clip_count.index_add_(0, vid, torch.ones_like(vid))

    def iter_tic(self):
        self._tic = time.perf_counter()

    def iter_toc(self):
        self._elapsed = time.perf_counter() - self._tic

    def log_iter_stats(self, cur_iter):
        return {"split": "test_iter", "cur_iter": str(cur_iter + 1), "time_diff": self._elapsed,
                "eta_sec": self._elapsed * (self.overall_iters - cur_iter)}

    def finalize_metrics(self, ks=(1, 5)):
        stats = {"split": "test_final", "complete": bool((self.clip_count == self.num_clips).all())}
        correct = topks_correct(self.video_preds, self.video_labels, ks)
        for k, c in zip(ks, correct):
            stats["top{}_acc".format(k)] = "{:.2f}".format(float(c) / self.video_preds.size(0) * 100.0)
        self.stats = stats
        return stats


def _slow_is_subset_of_fast(inputs):
    """True when [slow, fast] is what pack_pathway_output (datasets/utils.py:93-102) makes of the fast clip."""
    if len(inputs) != 2 or inputs[0].dim() != 5 or inputs[0].shape[2] > inputs[1].shape[2]:
        return False
    idx = torch.linspace(0, inputs[1].shape[2] - 1, inputs[0].shape[2]).long()
    return bool(torch.equal(inputs[0], inputs[1].index_select(2, idx)))


@torch.no_grad()
def perform_test(test_loader, model, test_meter, cfg, depth=2, slow_from_fast=None):
    """Classification branch of tools/test_net.py:21-123 over `(inputs, labels, video_idx, meta)` batches.  `inputs` is
    the reference's list [slow, fast] of FP32 host tensors (pinned memory makes the copies asynchronous); the last
    batch may be shorter (the reference's test loader has drop_last=False).  `slow_from_fast`: upload only the fast
    clip and let the slow pathway read its frames out of it (ClipStream); None = decide from the first batch."""
    if cfg.DETECTION.ENABLE:
        return perform_detection_test(test_loader, model, test_meter, cfg)
    model.eval()
    multi = cfg.NUM_GPUS > 1 and esf_dist.dist.is_available() and esf_dist.dist.is_initialized()
    device = next(model.parameters()).device
    stream, queued = None, []
    ks = (1, cfg.TRAIN.TOPK) if hasattr(cfg, "TRAIN") and "TOPK" in cfg.TRAIN else (1, 5)

    def consume(done):
        index, preds = done
        labels, video_idx = queued.pop(0)
        test_meter.iter_toc()
        test_meter.update_stats(preds, labels, video_idx)
        test_meter.log_iter_stats(index)
        test_meter.iter_tic()

    test_meter.iter_tic()
    for inputs, labels, video_idx, _meta in test_loader:
        if not isinstance(inputs, (list, tuple)):
            inputs = [inputs]
        if stream is None:
            if slow_from_fast is None:
                slow_from_fast = hasattr(model, "forward_fast") and _slow_is_subset_of_fast(inputs)
            stream = ClipStream(model, [tuple(t.shape) for t in inputs], device=device, depth=depth, gather=multi,
                                slow_from_fast=slow_from_fast)
        if multi:
            labels, video_idx = [t.cpu() for t in esf_dist.all_gather([labels.to(device), video_idx.to(device)])]
        queued.append((labels, video_idx))
        done = stream.submit(inputs)
        if done is not None:
            consume(done)
    if stream is not None:
        for done in stream.flush():
            consume(done)
    stats = test_meter.finalize_metrics(ks=ks)
    test_meter.reset()
    return stats


def _host(t):
    return t.detach().cpu() if torch.is_tensor(t) else t


@torch.no_grad()
def perform_detection_test(test_loader, model, test_meter, cfg):
    """Detection branch of tools/test_net.py:21-123 over `(inputs, labels, video_idx, meta)` batches: the clips go to the
    model's device, `preds = model(inputs, meta["boxes"])` (boxes (K, 5) [batch index, x1, y1, x2, y2] in input pixels,
    copied to the device once by the model), then `test_meter.update_stats(preds, meta["ori_boxes"], meta["metadata"])`
    on the host and `log_iter_stats(None, cur_iter)`.  `test_meter` is duck-typed (the reference's AVAMeter);
    returns what its finalize_metrics() returns.  One process: sharding boxes over GPUs is not implemented."""
    if cfg.NUM_GPUS > 1:
        raise NotImplementedError("multi-GPU detection testing (box sharding and all_gather_unaligned of the "
                                  "predictions) is not implemented; run detection with NUM_GPUS = 1")
    model.eval()
    device = next(model.parameters()).device
    test_meter.iter_tic()
    for cur_iter, (inputs, _labels, _video_idx, meta) in enumerate(test_loader):
        if not isinstance(inputs, (list, tuple)):
            inputs = [inputs]
        inputs = [t.to(device, non_blocking=True) for t in inputs]
        preds = model(inputs, meta["boxes"])
        test_meter.iter_toc()
        test_meter.update_stats(_host(preds), _host(meta["ori_boxes"]), _host(meta["metadata"]))
        test_meter.log_iter_stats(None, cur_iter)
        test_meter.iter_tic()
    return test_meter.finalize_metrics()
