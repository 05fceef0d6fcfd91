"""A/B of programmatic dependent launch (ofdis_set_option("pdl", 0 | 1)) on the bench workload: graph-replayed step time
of 1 / 8 / 64 pairs on one stream, flows compared bit for bit; a second pass runs 20 replays each and compares all.
python tools/pdl_ab.py [B ...]"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from of_dis_b200 import api, params, synth

prm = params.operating_point(2, 1024)
h, w = 436, 1024
i0, i1, _ = synth.synthetic_pair(h, w, 1, seed=1, amp=6.0)
scf = 1 << prm.sc_f
W, H = (w + scf - 1) // scf * scf, (h + scf - 1) // scf * scf
for B in [int(a) for a in sys.argv[1:]] or [1, 8, 64]:
    res, flows = {}, {}
    for pdl in (0, 1):
        ctx = api.Context(prm, W, H, prm.p_samp_s, B)
        ctx.set_option("pdl", pdl)
        frames = np.ascontiguousarray(np.stack([np.stack([i0, i1])] * B))
        ctx.upload_frames_u8(0, B, frames, w, h)
        ctx.set_graph_mode(True)
        for _ in range(5):
            ctx.run(B)
        ctx.sync()
        best = 1e9
        for rep in range(5):
            t0 = time.perf_counter()
            for _ in range(50):
                ctx.run(B)
            ctx.sync()
            best = min(best, (time.perf_counter() - t0) * 1e3 / 50)
        res[pdl] = best
        fl = []
        for _ in range(20):  # races would show up as run-to-run differences
            ctx.run(B)
            fl.append(ctx.get_flow(B - 1, prm.sc_l).copy())
        flows[pdl] = fl
        ctx.close()
    same = all(np.array_equal(f.view(np.uint32), flows[0][0].view(np.uint32)) for f in flows[0] + flows[1])
    print(json.dumps({"pairs": B, "ms_per_step_pdl0": round(res[0], 4), "ms_per_step_pdl1": round(res[1], 4),
                      "all_40_flows_bitwise_equal": bool(same)}), flush=True)
