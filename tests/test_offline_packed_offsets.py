"""Row offsets of a packed offline call (PathConfig.packed_offsets): per utterance the encoder rows of Conv2dSubsampling4 and the
adapter rows of the configured adapter, as prefix sums; CPU only."""
import dataclasses

import numpy as np
import pytest

from freeze_omni_b200.config import load_path_config


def test_offsets_match_per_utterance_lengths():
    cfg = load_path_config("tiny")
    lens = [7, 8, 10, 11, 19, 67, 203, 1003]
    eo, ao = cfg.packed_offsets(lens)
    t2 = [((t - 1) // 2 - 1) // 2 for t in lens]
    assert t2[:4] == [1, 1, 1, 2]
    assert list(np.diff(eo)) == t2 and eo[0] == 0
    assert list(np.diff(ao)) == [(t - 1) // 2 + 1 for t in t2]
    assert [cfg.sub_len(t) for t in lens] == t2 and [cfg.adapter_len(t) for t in t2] == list(np.diff(ao))
    assert eo.dtype == np.int64 and len(eo) == len(ao) == len(lens) + 1


@pytest.mark.parametrize("kind", ["linear", "cnn"])
def test_rate_keeping_adapters(kind):
    cfg = dataclasses.replace(load_path_config("tiny"), adapter_type=kind)
    eo, ao = cfg.packed_offsets(np.array([7, 100, 2999], dtype=np.int32))
    assert np.array_equal(eo, ao)


def test_short_or_empty_refused():
    cfg = load_path_config("tiny")
    with pytest.raises(ValueError):
        cfg.packed_offsets([7, 6])
    with pytest.raises(ValueError):
        cfg.packed_offsets([])
