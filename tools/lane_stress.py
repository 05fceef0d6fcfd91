"""Stress run of sor_lane_kernel's flag protocol and of programmatic dependent launch: many graph replays of the same
inputs, every flow compared bit for bit with the first one (a memory-ordering bug would be a rare event, not a
deterministic one).  python tools/lane_stress.py [replays]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from of_dis_b200 import api, params, preprocess, synth

N = int(sys.argv[1]) if len(sys.argv) > 1 else 300
CASES = [
    ("bench_1024x436_op2", (436, 1024), 1, 2, lambda: params.operating_point(2, 1024), (1, 8, 16)),
    ("rows100_5sweeps_4bands", (200, 320), 1, 2, lambda: params.from_cli_numbers("3 1 8 8 0.05 0.95 0 6 0.5 0 0 0 1 10 10 5 2 5 1.5 0".split()), (3,)),
    ("stereo_rows125_4bands", (250, 360), 1, 1, lambda: params.from_cli_numbers("3 1 32 32 0.05 0.95 0 12 0.75 0 1 0 1 10 10 5 1 3 1.6 0".split(), noc=1, nop=1), (2,)),
    ("rgb_rows135_5bands", (270, 480), 3, 2, lambda: params.from_cli_numbers("4 1 16 16 0.05 0.95 0 12 0.75 0 1 1 1 10 10 5 1 3 1.6 0".split(), noc=3), (2,)),
]
bad = 0
for name, (h, w), ch, nop, mk, batches in CASES:
    prm = mk()
    i0, i1, _ = synth.synthetic_pair(h, w, ch, seed=7, stereo=(nop == 1), amp=5.0)
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    for B in batches:
        ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, B)
        ctx.set_option("sor_lane", 1)  # also on the levels the auto rule would leave to sor_wave_kernel
        ctx.set_option("pdl", 1)
        for f in range(B):
            ctx.upload_pyramids(f, pyr)
        ctx.set_graph_mode(True)
        ctx.run(B)
        ref = [ctx.get_flow(f, prm.sc_l).copy() for f in range(B)]
        diff = 0
        for r in range(N):
            ctx.run(B)
            f = r % B
            if not np.array_equal(ctx.get_flow(f, prm.sc_l).view(np.uint32), ref[f].view(np.uint32)):
                diff += 1
        ctx.close()
        bad += diff
        print(json.dumps({"case": name, "pairs": B, "replays": N, "replays_that_differ": diff}), flush=True)
sys.exit(1 if bad else 0)
