import hashlib
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu under gpurun)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def synth_audio(seed, n):
    """SURVEY 8d config 2: 0.1*N(0,1) band-limited, 200 ms silent gaps, int16-quantised."""
    g = torch.Generator().manual_seed(seed)
    x = 0.1 * torch.randn(n + 8, generator=g)
    x = torch.nn.functional.avg_pool1d(x.view(1, 1, -1), 5, 1).view(-1)[:n] * 2.0
    t = torch.arange(n)
    x = x * ((t // 3200) % 5 != 4).float()
    return torch.clamp((x * 32768.0).round(), -32768, 32767).to(torch.int16)


def stream_feats(pcm):
    """(chunks, sessions, 19, 80) fbank blocks of int16 pcm (sessions, samples), 2560-sample chunks at scale 32768: what
    bin/inference.py feeds the encoder, computed by the oracle's streaming frontend."""
    from oracle import freeze_omni_oracle as O
    fronts = [O.StreamingFrontend() for _ in pcm]
    return np.stack([np.concatenate([f.process(torch.from_numpy(p[i:i + 2560].astype(np.float32) / 32768.0), 32768.0).numpy()
                                     for f, p in zip(fronts, pcm)]) for i in range(0, pcm.shape[1] - 2559, 2560)])


def _rebuild_inputs(name, g):
    """The inputs tests/golden/make_golden.py does not store: seeded audio and features rebuilt with the seeds it used,
    streaming features from that audio, checked bit for bit against the SHA-256 of the reference's own features."""
    if name == "tiny":
        g["stream_pcm"] = np.stack([synth_audio(2000 + b, 2560 * 24).numpy() for b in range(3)])
        gen = torch.Generator().manual_seed(5)
        g["t7_feats"] = torch.stack([9.0 + 3.0 * torch.randn(1, 32, 80, generator=gen) for _ in range(12)]).numpy()
        g["off_feats"] = (9.0 + 3.0 * torch.randn(3, 150, 80, generator=gen)).numpy()
        feats, pcm = "stream_feats", g["stream_pcm"]
    elif name == "shipped_b2":
        feats, pcm = "feats", np.stack([synth_audio(1000 + b, 2560 * 20).numpy() for b in range(2)])
    elif name == "shipped_question":
        feats, pcm = "feats", g["pcm"][None]
    else:
        return g
    g[feats] = stream_feats(pcm)
    digest = hashlib.sha256(g[feats].tobytes()).hexdigest()
    assert digest == str(g[feats + "_sha256"]), "%s: rebuilt %s differ from the reference's" % (name, feats)
    return g


def load_golden(name):
    return _rebuild_inputs(name, dict(np.load(os.path.join(GOLDEN, name + ".npz"))))


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = load_golden(name)
        return cache[name]
    return get
