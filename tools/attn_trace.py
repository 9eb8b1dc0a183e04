#!/usr/bin/env python
"""Timeline of one CTA of the fp16 streaming attention kernel (library built with FO_TC_TRACE_BUILD=1).
t1 after the dependency wait, t2 session state read, t3 bulk copies issued, t4 registers staged to smem, t5 all rows
landed, t9 output stored (ns from kernel entry).  t9 - t5 is the shared chunk core (scores, softmax, PV, store:
attn_chunk_mma in csrc/fo_attn_core.cuh)."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["FO_TC_TRACE"] = "1"
from freeze_omni_b200.config import load_path_config  # noqa: E402
from freeze_omni_b200.engine import Engine  # noqa: E402
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state  # noqa: E402

cfg = load_path_config("shipped")
S = 64
eng = Engine(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0), dtype=torch.bfloat16, max_sessions=S,
             max_stream_frames=cfg.chunk_feat_frames)
eng.set_option("use_graph", 0)
ids = eng.alloc(S)
pcm = (0.05 * torch.randn(S, cfg.samples_per_chunk) * 32768).round().to(torch.int16).cuda()
for i in range(19):
    if i == 18:
        sys.stderr.write("---- step %d (windows full)\n" % i)
    eng.stream_step(ids, pcm, 1.0)
torch.cuda.synchronize()
eng.close()
