"""One eager step of BASELINE configs[2] (cfg3) or configs[4] (cfg5) on B pairs, for ncu captures of the
P = 12 patch kernel and the cluster SOR:
   ncu --set full -k regex:sor_wave -c 3 ... python tools/one_step_big.py cfg5 1"""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
from of_dis_b200 import api, synth
import big_configs

name = [k for k in big_configs.CFGS if sys.argv[1] in k][0]
B = int(sys.argv[2]) if len(sys.argv) > 2 else 1
c = big_configs.CFGS[name]
prm = c["prm"]()
h, w = c["size"]
i0, i1, _ = synth.synthetic_pair(h, w, c["ch"], seed=1, stereo=(c["nop"] == 1), amp=6.0)
scf = 1 << prm.sc_f
W, H = (w + scf - 1) // scf * scf, (h + scf - 1) // scf * scf
ctx = api.Context(prm, W, H, prm.p_samp_s, B)
for o in sys.argv[3:]:
    k, v = o.split("=")
    ctx.set_option(k, int(v))
frames = np.ascontiguousarray(np.stack([np.stack([i0, i1])] * B))
ctx.upload_frames_u8(0, B, frames, w, h)
ctx.run(B)
ctx.sync()
print('launches', ctx.launch_count)
