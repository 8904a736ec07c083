"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's test-time temporal sampling (upstream PySlowFast
slowfast/datasets/decoder.py at the fork's age: the clip size of `decode`, `get_start_end_idx` with a given clip index
and `temporal_sampling`), for the branch where the whole video is decoded (`decode_all_video`: the clip index and the
number of clips are used as given; the uniform split, which later upstream versions keep as the default of
DATA.USE_OFFSET_SAMPLING = False).  The Kinetics test dataset (datasets/kinetics.py) numbers the clips of a video
`temporal_idx * NUM_SPATIAL_CROPS + spatial_idx` and calls `decode(..., clip_idx=temporal_idx,
num_clips=NUM_ENSEMBLE_VIEWS, target_fps=DATA.TARGET_FPS)`.  The product path (efficient_slowfast_b200.frames
temporal_index + csrc/esf_crop.cu) never imports it.

Pinned against the reference's own functions in tests/test_frames_videos.py wherever ESF_REFERENCE_ROOT points to it.
"""
import torch


def temporal_sampling(frames, start_idx, end_idx, num_samples):
    """decoder.temporal_sampling: num_samples frames between start_idx and end_idx at equal intervals."""
    index = torch.linspace(start_idx, end_idx, num_samples)
    index = torch.clamp(index, 0, frames.shape[0] - 1).long()
    frames = torch.index_select(frames, 0, index)
    return frames


def get_start_end_idx(video_size, clip_size, clip_idx, num_clips):
    """decoder.get_start_end_idx for clip_idx >= 0 (test mode: uniform split into num_clips clips)."""
    delta = max(video_size - clip_size, 0)
    start_idx = delta * clip_idx / num_clips
    end_idx = start_idx + clip_size - 1
    return start_idx, end_idx


def decode_all_video(frames, sampling_rate, num_frames, clip_idx, num_clips, fps, target_fps=30):
    """decoder.decode after the decoder returned every frame of the video (decode_all_video = True)."""
    clip_sz = sampling_rate * num_frames / target_fps * fps
    start_idx, end_idx = get_start_end_idx(frames.shape[0], clip_sz, clip_idx, num_clips)
    return temporal_sampling(frames, start_idx, end_idx, num_frames)


def sampled_index(video_size, sampling_rate, num_frames, clip_idx, num_clips, fps, target_fps=30):
    """The frame numbers decode_all_video picks: temporal_sampling applied to the frame numbers themselves."""
    return decode_all_video(torch.arange(video_size), sampling_rate, num_frames, clip_idx, num_clips, fps, target_fps)


def view_clips(video_u8, sampling_rate, num_frames, num_clips, fps, target_fps=30):
    """The uint8 clips (T, H, W, C) of the num_clips temporal views of one decoded video (N, H, W, C), in order."""
    return [decode_all_video(video_u8, sampling_rate, num_frames, j, num_clips, fps, target_fps)
            for j in range(num_clips)]
