"""CPU oracle for the segment-index rules of the reference's feature loader -- TEST INFRASTRUCTURE.

SURVEY 8f row n3: `dataset.py` of cmhungsteve/TA3N decides which pre-extracted frame features of a video
feed the path.  This file restates those rules (plain Python / numpy), each function citing the reference
lines it follows; `tests/test_dataset.py` pins it against `tests/golden/dataset_indices.npz`, which
`oracle/gen_golden_dataset.py` produced by running the reference itself.  Only tests may import this module.
"""
from __future__ import annotations

from typing import List

import numpy as np


def val_indices(num_frames: int, num_segments: int, new_length: int = 1) -> np.ndarray:
    """dataset.py:92-101 (`_get_val_indices`): centre frame of each of num_segments equal ticks, 1-based;
    all ones when the video is shorter than num_segments + new_length - 1."""
    num_min = num_segments + new_length - 1
    num_select = num_frames - new_length + 1
    if num_frames >= num_min:
        tick = float(num_select) / float(num_segments)
        offsets = np.array([int(tick / 2.0 + tick * float(x)) for x in range(num_segments)])
    else:
        offsets = np.zeros((num_segments,))
    return offsets + 1


def test_indices(num_frames: int, num_segments: int, new_length: int = 1) -> np.ndarray:
    """dataset.py:103-116 (`_get_test_indices`) -- the rule main.py uses for EVERY split, training included
    (main.py:171-196 build all three sets with random_shift=False, test_mode=True).
    Long enough: as val_indices.  Too short: frames 0..num_select-1 followed by copies of
    `id_select[id_select[0]-1]`; id_select[0] is 0, so that is id_select[-1], the last selectable frame."""
    num_min = num_segments + new_length - 1
    num_select = num_frames - new_length + 1
    if num_frames >= num_min:
        tick = float(num_select) / float(num_segments)
        offsets = np.array([int(tick / 2.0 + tick * float(x)) for x in range(num_segments)])
    else:
        id_select = np.array([x for x in range(num_select)])
        id_expand = np.ones(num_segments - num_select, dtype=int) * id_select[id_select[0] - 1]
        offsets = np.append(id_select, id_expand)
    return offsets + 1


def sample_indices(num_frames: int, num_segments: int, new_length: int = 1) -> np.ndarray:
    """dataset.py:77-90 (`_sample_indices`, random_shift=True): one uniformly random frame per segment, drawn
    from numpy's GLOBAL RandomState exactly as the reference does (numpy.random.randint), so that seeding
    numpy reproduces the reference's draws."""
    from numpy.random import randint
    average_duration = (num_frames - new_length + 1) // num_segments
    if average_duration > 0:
        offsets = np.multiply(list(range(num_segments)), average_duration) + randint(average_duration, size=num_segments)
    elif num_frames > num_segments:
        offsets = np.sort(randint(num_frames - new_length + 1, size=num_segments))
    else:
        offsets = np.zeros((num_segments,))
    return offsets + 1


def frames_to_load(indices, num_frames: int, new_length: int = 1) -> List[int]:
    """dataset.py:128-140 (`get`): new_length consecutive frames from each start index, clamped at the end of
    the video (the frame counter only advances while p < num_frames)."""
    out = []
    for seg_ind in indices:
        p = int(seg_ind)
        for _ in range(new_length):
            out.append(p)
            if p < num_frames:
                p += 1
    return out


def repeat_list(n_items: int, num_dataload: int) -> List[int]:
    """dataset.py:70-75 (`_parse_list`): the list is tiled to exactly num_dataload entries."""
    n_repeat, n_left = num_dataload // n_items, num_dataload % n_items
    base = list(range(n_items))
    return base * n_repeat + base[:n_left]
