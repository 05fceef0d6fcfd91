"""1920x1080 gray at operating point 2 (levels 6..4, finest 240x135... see level_info): lane step time."""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from of_dis_b200 import api, params, preprocess, synth
B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
prm = params.operating_point(2, 1920)
i0, i1, _ = synth.synthetic_pair(1080, 1920, 1, seed=2)
scf = 1 << prm.sc_f
W, H = (1920 + scf - 1) // scf * scf, (1080 + scf - 1) // scf * scf
st = torch.cuda.Stream(); torch.cuda.set_stream(st)
ctx = api.Context(prm, W, H, prm.p_samp_s, B, stream=st.cuda_stream)
print('levels', [(lv, ctx.level_info(lv)['w'], ctx.level_info(lv)['h']) for lv in range(prm.sc_l, prm.sc_f + 1)])
ctx.upload_frames_u8(0, B, np.ascontiguousarray(np.stack([np.stack([i0, i1])] * B)), 1920, 1080)
ctx.set_graph_mode(True)
for _ in range(3): ctx.run(B)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record(st)
for _ in range(10): ctx.run(B)
b.record(st); torch.cuda.synchronize()
ms = a.elapsed_time(b) / 10
ctx.set_graph_mode(False)
prof = ctx.profile_kernels(B, steps=3)
print('B %d: %.3f ms/step  %.1f Gpix/s   sor %.3f ms' % (B, ms, B * 1920 * 1080 / ms / 1e6, prof['sor']['ms_per_step']))
