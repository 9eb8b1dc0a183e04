import os, sys, torch, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from freeze_omni_b200.config import load_path_config
from freeze_omni_b200.engine import Engine
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state
cfg = load_path_config("shipped")
eng = Engine(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0), dtype=torch.bfloat16, max_sessions=8)
g = torch.Generator().manual_seed(99)
ia, ib = eng.alloc(2), eng.alloc(2)
worst = 0.0
pcm_bank = (0.05 * torch.randn(16, 2, cfg.samples_per_chunk, generator=g) * 32768).round().clamp(-32768, 32767).to(torch.int16).cuda()
N = int(sys.argv[1]) if len(sys.argv) > 1 else 4000
for i in range(N):
    pcm = pcm_bank[i % 16]
    n = 1 + (i % 3 == 0)            # alternate 1 and 2 sessions per call (different graphs, different barrier targets)
    eng.set_option("stack_rows", 8)
    e1, y1 = eng.stream_step(ia[:n], pcm[:n], 1.0)
    eng.set_option("stack_rows", 0)
    e0, y0 = eng.stream_step(ib[:n], pcm[:n], 1.0)
    if i % 97 == 0 or i > N - 5:
        d = max(float((e1 - e0).abs().max()), float((y1 - y0).abs().max()))
        worst = max(worst, d)
        assert torch.isfinite(e1).all() and d < 5e-3, (i, d)
print("soak ok: %d steps, worst sampled max-abs stack vs chain %.3g, states %s %s, stack launches %d" % (N, worst, eng.state(int(ia[0])), eng.state(int(ib[0])), eng.get_option("stack_launches")))
