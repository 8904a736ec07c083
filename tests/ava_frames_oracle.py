"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the test split of the reference's AVA loader, PyTorch image backend
(upstream PySlowFast slowfast/datasets/ava_dataset.py: Ava.__getitem__ and Ava._images_and_boxes_preprocessing with
split "test"; slowfast/datasets/transform.py: clip_boxes_to_image, random_short_side_scale_jitter,
color_normalization; slowfast/datasets/utils.py: pack_pathway_output; slowfast/datasets/loader.py: detection_collate).
The product path (efficient_slowfast_b200.frames + csrc/esf_crop.cu) never imports it.

Pinned against the reference's own transform functions in tests/test_frames_ava.py wherever ESF_REFERENCE_ROOT points to
the reference tree.
"""
import math

import numpy as np
import torch

from oracle import input_oracle as IO


def clip_boxes_to_image(boxes, height, width):
    """transform.clip_boxes_to_image: numpy, x clipped to [0, width - 1], y to [0, height - 1]."""
    clipped_boxes = boxes.copy()
    clipped_boxes[:, [0, 2]] = np.minimum(width - 1.0, np.maximum(0.0, boxes[:, [0, 2]]))
    clipped_boxes[:, [1, 3]] = np.minimum(height - 1.0, np.maximum(0.0, boxes[:, [1, 3]]))
    return clipped_boxes


def random_short_side_scale_jitter(images, size, boxes=None):
    """transform.random_short_side_scale_jitter(images, min_size=size, max_size=size, boxes=boxes): the size is not
    random when min = max; images (T, C, H, W), boxes numpy (N, 4) scaled by new / old of the long side's resize."""
    height, width = images.shape[2], images.shape[3]
    if (width <= height and width == size) or (height <= width and height == size):
        return images, boxes
    new_width, new_height = size, size
    if width < height:
        new_height = int(math.floor((float(height) / width) * size))
        if boxes is not None:
            boxes = boxes * float(new_height) / height
    else:
        new_width = int(math.floor((float(width) / height) * size))
        if boxes is not None:
            boxes = boxes * float(new_width) / width
    return (torch.nn.functional.interpolate(images, size=(new_height, new_width), mode="bilinear",
                                            align_corners=False), boxes)


def color_normalization(images, mean, stddev):
    """transform.color_normalization for images (T, C, H, W): channel by channel, (x - mean[c]) / stddev[c]."""
    assert len(mean) == images.shape[1], "channel mean not computed properly"
    assert len(stddev) == images.shape[1], "channel stddev not computed properly"
    out_images = torch.zeros_like(images)
    for idx in range(len(mean)):
        out_images[:, idx] = (images[:, idx] - mean[idx]) / stddev[idx]
    return out_images


def images_and_boxes_preprocessing(imgs, boxes, crop_size, data_mean, data_std, use_bgr=False):
    """Ava._images_and_boxes_preprocessing, split "test": imgs uint8 (T, C, H, W), boxes float64 numpy (N, 4) in [0, 1].
    Returns FP32 (T, C, H', W') and float64 boxes in pixels of the resized frame."""
    # Image [0, 255] -> [0, 1].
    imgs = imgs.float()
    imgs = imgs / 255.0
    height, width = imgs.shape[2], imgs.shape[3]
    # The format of boxes is [x1, y1, x2, y2]. The input boxes are in the range of [0, 1].
    boxes = boxes.copy()
    boxes[:, [0, 2]] *= width
    boxes[:, [1, 3]] *= height
    boxes = clip_boxes_to_image(boxes, height, width)
    # split == "test": short side to the test scale, no crop (TEST_FORCE_FLIP off)
    imgs, boxes = random_short_side_scale_jitter(imgs, crop_size, boxes=boxes)
    # Normalize images by mean and std.
    imgs = color_normalization(imgs, np.array(data_mean, dtype=np.float32), np.array(data_std, dtype=np.float32))
    if not use_bgr:
        # Convert image format from BGR to RGB.
        imgs = imgs[:, [2, 1, 0], ...]
    boxes = clip_boxes_to_image(boxes, crop_size, crop_size)
    return imgs, boxes


def prepare(frames_u8, boxes, crop_size, mean, std, alpha, single_pathway=False, use_bgr=False,
            reverse_input_channel=False):
    """uint8 frames (B, T, H, W, C) and the loader's boxes (K, 5) [batch index, x1, y1, x2, y2] in [0, 1] -> the
    model's input list and the FP32 (K, 5) boxes in pixels, clip by clip as Ava.__getitem__ and detection_collate make
    them.  Row k of the boxes keeps its position (the collate concatenates clip by clip; here the rows of every clip
    are put back where they came from)."""
    boxes = boxes.detach().cpu().to(torch.float64).numpy()
    per_clip, out = [], np.zeros((boxes.shape[0], 5), dtype=np.float64)
    out[:, 0] = boxes[:, 0]
    for b in range(frames_u8.shape[0]):
        # T H W C -> T C H W.
        imgs = frames_u8[b].permute(0, 3, 1, 2)
        rows = np.nonzero(boxes[:, 0] == b)[0]
        imgs, bx = images_and_boxes_preprocessing(imgs, boxes[rows, 1:5].copy(), crop_size, mean, std, use_bgr)
        out[rows, 1:5] = bx
        # T C H W -> C T H W.
        imgs = imgs.permute(1, 0, 2, 3)
        per_clip.append(IO.pack_pathway_output(imgs, alpha, single_pathway, reverse_input_channel))
    xs = [torch.stack([c[i] for c in per_clip]).contiguous() for i in range(len(per_clip[0]))]
    # detection_collate: torch.tensor(np.concatenate(...)).float()
    return xs, torch.tensor(out).float()
