"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's test-mode spatial sampling (upstream PySlowFast
slowfast/datasets/utils.py spatial_sampling with spatial_idx in {0, 1, 2}, and transform.py
random_short_side_scale_jitter / uniform_crop), and the Kinetics test branch around it (datasets/kinetics.py:
tensor_normalize -> permute(3, 0, 1, 2) -> spatial_sampling(min_scale = max_scale = crop_size = DATA.TEST_CROP_SIZE) ->
pack_pathway_output).  The product path (efficient_slowfast_b200.frames + csrc/esf_crop.cu) never imports it.

Pinned against the reference's own functions in tests/test_frames_spatial.py wherever ESF_REFERENCE_ROOT points to it.
"""
import math

import torch

from oracle import input_oracle as IO


def random_short_side_scale_jitter(images, size):
    """transform.random_short_side_scale_jitter(images, size, size): test mode, the size is not random."""
    height, width = images.shape[2], images.shape[3]
    if (width <= height and width == size) or (height <= width and height == size):
        return images
    new_width, new_height = size, size
    if width < height:
        new_height = int(math.floor((float(height) / width) * size))
    else:
        new_width = int(math.floor((float(width) / height) * size))
    return torch.nn.functional.interpolate(images, size=(new_height, new_width), mode="bilinear", align_corners=False)


def uniform_crop(images, size, spatial_idx):
    """transform.uniform_crop without boxes or scale_size."""
    assert spatial_idx in [0, 1, 2]
    height, width = images.shape[2], images.shape[3]
    y_offset = int(math.ceil((height - size) / 2))
    x_offset = int(math.ceil((width - size) / 2))
    if height > width:
        if spatial_idx == 0:
            y_offset = 0
        elif spatial_idx == 2:
            y_offset = height - size
    else:
        if spatial_idx == 0:
            x_offset = 0
        elif spatial_idx == 2:
            x_offset = width - size
    return images[:, :, y_offset:y_offset + size, x_offset:x_offset + size]


def spatial_sampling(frames, spatial_idx, crop_size):
    """utils.spatial_sampling(frames, spatial_idx, min_scale = max_scale = crop_size = crop_size), frames (C, T, H, W)."""
    return uniform_crop(random_short_side_scale_jitter(frames, crop_size), crop_size, spatial_idx)


def frames_to_crop_inputs(frames_u8, mean, std, alpha, crop_size, spatial_idx, single_pathway=False,
                          reverse_input_channel=False):
    """uint8 (B, T, H, W, C) at decode size -> the model's input list for the V views `spatial_idx`, clip by clip like the
    test loader (clip k of a video: temporal window k // V, view k % V), stacked by the collate function: row b * V + v."""
    per_clip = []
    for b in range(frames_u8.shape[0]):
        f = IO.tensor_normalize(frames_u8[b], list(mean), list(std))
        f = f.permute(3, 0, 1, 2)
        for v in spatial_idx:
            c = spatial_sampling(f, v, crop_size)
            per_clip.append(IO.pack_pathway_output(c, alpha, single_pathway, reverse_input_channel))
    return [torch.stack([c[i] for c in per_clip]).contiguous() for i in range(len(per_clip[0]))]
