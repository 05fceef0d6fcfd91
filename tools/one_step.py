"""One eager step (48 launches at operating point 2) of a B-pair batch, for ncu launch lists:
   ncu --metrics gpu__time_duration.sum,smsp__inst_executed.sum --clock-control none --csv \
       --log-file gpurun_out/x.csv python tools/one_step.py [B] [steps]"""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from of_dis_b200 import api, params, preprocess, synth
B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 1
prm = params.operating_point(2, 1024)
pyrs = []
for s in range(min(B, 8)):
    i0, i1, _ = synth.synthetic_pair(436, 1024, 1, seed=s)
    pyrs.append(preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s))
ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, B)
packed = np.stack([ctx.pack_frame(pyrs[f % len(pyrs)]) for f in range(B)])
ctx.upload_packed(0, B, packed)
for _ in range(steps):
    ctx.run(B)
ctx.sync()
print('launches', ctx.launch_count)
