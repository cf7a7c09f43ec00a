import sys, json, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from jepsen_tigerbeetle_b200 import native, synth, history as H
sp = synth.SynthSpec('cas-register', 1000, 16, 1, p_info=0.05)
h = synth.generate(sp); m = H.make_model(H.MODEL_CAS_REGISTER)
with native.Context(device=0, time_budget_ms=20000) as ctx:
    g = ctx.check_linearizable(h, m); st = ctx.stats()
print(g["valid"], g["seconds_kernel"], {k: st[k] for k in ("beam_levels", "beam_configs", "beam_decided", "beam_attempts", "scouts", "configs")})
