"""Which part of the e2e step breaks the overlap between lanes?  A/B variants on one box."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from of_dis_b200 import api, params, preprocess, synth
prm = params.operating_point(2, 1024)
i0, i1, _ = synth.synthetic_pair(436, 1024, 1, seed=0)
pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
B = 64; NL = int(sys.argv[1]) if len(sys.argv) > 1 else 4
lanes = []
for _ in range(NL):
    st = torch.cuda.Stream()
    c = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, B, stream=st.cuda_stream)
    lanes.append((c, st))
ctx = lanes[0][0]
ff = ctx.packed_frame_floats; ni = ctx.packed_images_frame_floats
li = ctx.level_info(prm.sc_l); fl = li['w'] * li['h'] * prm.nop
hin = torch.empty((B, ff), dtype=torch.float32, pin_memory=True)
for f in range(B): ctx.pack_frame(pyr, hin[f].numpy())
himg = torch.empty((B, ni), dtype=torch.float32, pin_memory=True); himg.copy_(hin[:, :ni])
houts = [torch.empty((B, fl), dtype=torch.float32, pin_memory=True) for _ in range(NL)]
dfull = [torch.empty((B, ff), dtype=torch.float32, device='cuda') for _ in range(NL)]
dimg = [torch.empty((B, ni), dtype=torch.float32, device='cuda') for _ in range(NL)]
dfl = [torch.empty((B, fl), dtype=torch.float32, device='cuda') for _ in range(NL)]
small = [torch.zeros(4096, device='cuda') for _ in range(NL)]
for c, st in lanes:
    c.upload_packed(0, B, hin.data_ptr()); c.set_graph_mode(True); c.run(B)
torch.cuda.synchronize()
def pipelined(step, steps=40):
    for i in range(2 * NL): step(i)
    torch.cuda.synchronize()
    s0 = lanes[0][1]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s0)
    for _, s in lanes[1:]: s.wait_event(e0)
    w = time.perf_counter()
    for i in range(steps): step(i)
    wq = (time.perf_counter() - w) / steps * 1e3
    for _, s in lanes[1:]: s0.wait_stream(s)
    e1.record(s0); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, wq
def mk(h2d, extra, d2h):
    def step(i):
        k = i % NL; c, s = lanes[k]
        with torch.cuda.stream(s):
            if h2d == 'full': dfull[k].copy_(hin, non_blocking=True)
            elif h2d == 'img': dimg[k].copy_(himg, non_blocking=True)
            elif h2d == 'api_img': c.upload_packed_images(0, B, himg.data_ptr())
            elif h2d == 'api_pyr': c.upload_packed(0, B, hin.data_ptr())
            for _ in range(extra): small[k].add_(1.0)
            c.run(B)
            if d2h == 'api': c.get_flow_batch(0, B, houts[k].data_ptr())
            elif d2h == 'torch': houts[k].copy_(dfl[k], non_blocking=True)
    return step
variants = [('resident only', mk(None, 0, None)), ('run + D2H(api)', mk(None, 0, 'api')), ('run + D2H(torch)', mk(None, 0, 'torch')),
            ('H2D full(torch) + run', mk('full', 0, None)), ('H2D img(torch) + run', mk('img', 0, None)),
            ('H2D full(torch) + run + D2H', mk('full', 0, 'api')), ('H2D img(torch) + run + D2H', mk('img', 0, 'api')),
            ('H2D img(torch) + 3 tiny kernels + run + D2H', mk('img', 3, 'api')),
            ('3 tiny kernels + run', mk(None, 3, None)),
            ('api images + run + D2H', mk('api_img', 0, 'api')), ('api pyramids + run + D2H', mk('api_pyr', 0, 'api'))]
for rep in range(2):
    for name, fn in variants:
        ms, wq = pipelined(fn)
        print('%-46s %.4f ms/step  (host enqueue %.4f)  %.1f Gpix/s' % (name, ms, wq, B * 436 * 1024 / ms / 1e6))
