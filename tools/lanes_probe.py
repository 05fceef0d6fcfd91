"""Resident throughput of NL lanes (graph replay), for A/B experiments driven by env knobs."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from of_dis_b200 import api, params, preprocess, synth
import dataclasses, os
prm = params.operating_point(2, 1024)
FB = int(os.environ.get('FB', '0'))  # 1: forward-backward consistency (usefbcon)
prm = dataclasses.replace(prm, usefbcon=FB)
i0, i1, _ = synth.synthetic_pair(436, 1024, 1, seed=0)
pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
B = int(os.environ.get('B', '64')); NL = int(sys.argv[1]) if len(sys.argv) > 1 else 8
lanes = []
for _ in range(NL):
    st = torch.cuda.Stream()
    c = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, B, stream=st.cuda_stream)
    lanes.append((c, st))
import numpy as np
packed = np.stack([lanes[0][0].pack_frame(pyr)] * B)
ni = lanes[0][0].packed_images_frame_floats
imgs = np.ascontiguousarray(packed[:, :ni])
for c, st in lanes:
    c.upload_packed_images(0, B, imgs); c.set_graph_mode(True); c.run(B)
torch.cuda.synchronize()
def pipelined(steps=80):
    for i in range(2 * NL): lanes[i % NL][0].run(B)
    torch.cuda.synchronize()
    s0 = lanes[0][1]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s0)
    for _, s in lanes[1:]: s.wait_event(e0)
    for i in range(steps): lanes[i % NL][0].run(B)
    for _, s in lanes[1:]: s0.wait_stream(s)
    e1.record(s0); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps
r = [pipelined() for _ in range(3)]
print('B %d' % B, 'usefbcon %d' % FB, 'lanes %d: ms/step %s -> %.1f Gpix/s' % (NL, ['%.4f' % x for x in r], B * 436 * 1024 / min(r) / 1e6))
