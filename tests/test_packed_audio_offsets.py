"""Offsets of a packed PCM call (PathConfig.packed_audio_offsets): per utterance the kaldi frame count of its samples
(snip_edges), then the encoder and adapter rows of those frames as prefix sums; CPU only."""
import dataclasses

import numpy as np
import pytest

from freeze_omni_b200.config import load_path_config, load_yaml, path_config_from_dict


def fork_cfg():
    y = load_yaml("tiny")
    y["frontend"] = dict(y["frontend"], frame_length_ms=16, frame_shift_ms=8, frames_per_chunk=28, context_frames=4)
    return path_config_from_dict(y)


@pytest.mark.parametrize("cfg", [load_path_config("tiny"), fork_cfg(), dataclasses.replace(load_path_config("tiny"), adapter_type="cnn")],
                         ids=["shipped_frontend", "fork_frontend", "cnn_adapter"])
def test_offsets_match_a_direct_loop(cfg):
    L, S = cfg.frame_len, cfg.frame_shift
    # seven frames exactly, one sample short of the eighth, one sample into it, remainders, several seconds
    n = [L + 6 * S, L + 7 * S - 1, L + 7 * S, L + 7 * S + 1, L + 100 * S + S // 2, 3 * cfg.sample_rate + 17, 10 * cfg.sample_rate]
    frames, eo, ao = cfg.packed_audio_offsets(n)
    fl, el, al = [], [0], [0]
    for s in n:
        m, k = 0, 0
        while k + L <= s:             # kaldi snip_edges: a frame every frame_shift samples while it fits
            m, k = m + 1, k + S
        t2 = ((m - 1) // 2 - 1) // 2
        fl.append(m)
        el.append(el[-1] + t2)
        al.append(al[-1] + cfg.adapter_len(t2))
    assert list(frames) == fl and list(eo) == el and list(ao) == al
    assert fl[:4] == [7, 7, 8, 8]
    assert frames.dtype == eo.dtype == ao.dtype == np.int64 and len(eo) == len(ao) == len(n) + 1
    e2, a2 = cfg.packed_offsets(frames)
    assert np.array_equal(e2, eo) and np.array_equal(a2, ao)


def test_short_or_empty_refused():
    cfg = load_path_config("tiny")
    L, S = cfg.frame_len, cfg.frame_shift
    with pytest.raises(ValueError):
        cfg.packed_audio_offsets([L + 6 * S, L + 6 * S - 1])     # six frames
    with pytest.raises(ValueError):
        cfg.packed_audio_offsets([L - 1])                        # not one frame
    with pytest.raises(ValueError):
        cfg.packed_audio_offsets([])
