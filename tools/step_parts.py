import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from freeze_omni_b200.config import load_path_config
from freeze_omni_b200.engine import Engine
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state
cfg = load_path_config("shipped")
eng = Engine(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0), dtype=torch.bfloat16, max_sessions=8)
st = torch.cuda.current_stream()
for n in (1, 2):
    ids = eng.alloc(n)
    pcm = (0.05 * torch.randn(n, cfg.samples_per_chunk) * 32768).round().clamp(-32768, 32767).to(torch.int16).cuda()
    for part in (0, 1, 2):
        eng.set_option("step_part", part)
        for _ in range(10):
            eng.stream_step(ids, pcm, 1.0)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for _ in range(200):
            eng.stream_step(ids, pcm, 1.0, want_enc=False)
        b.record(st)
        torch.cuda.synchronize()
        print("n=%d step_part=%d: %.4f ms, launches per step %d" % (n, part, a.elapsed_time(b) / 200, 0), flush=True)
    eng.set_option("step_part", 0)
    eng.free(ids)
