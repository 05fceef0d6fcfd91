"""A/B of the two exact SOR kernels on the bench workload (1024x436 gray, operating point 2) and on
configs[2] (1920x1080 RGB): ofdis_set_option("sor_lane", 0 | 1); per pyramid level the SOR and assemble time of
one eager pass, and the graph-replayed step time.  python tools/lane_ab.py [B ...]  -> one JSON line per (config, B, lane)."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from of_dis_b200 import api, params, synth

CFGS = {
    "cfg2_1024x436_gray_op2": dict(size=(436, 1024), ch=1, nop=2, prm=lambda: params.operating_point(2, 1024)),
    "cfg3_1920x1080_rgb_l1": dict(size=(1080, 1920), ch=3, nop=2, prm=lambda: params.from_cli_numbers(
        "6 2 16 16 0.05 0.95 0 12 0.75 0 1 1 1 10 10 5 1 3 1.6 0".split(), noc=3)),
}


def measure(name, c, B, lane):
    prm = c["prm"]()
    h, w = c["size"]
    st = torch.cuda.current_stream()
    i0, i1, _ = synth.synthetic_pair(h, w, c["ch"], seed=1, amp=6.0)
    scf = 1 << prm.sc_f
    W, H = (w + scf - 1) // scf * scf, (h + scf - 1) // scf * scf
    ctx = api.Context(prm, W, H, prm.p_samp_s, B, stream=st.cuda_stream)
    ctx.set_option("sor_lane", lane)
    frames = np.ascontiguousarray(np.stack([np.stack([i0, i1])] * B))
    ctx.upload_frames_u8(0, B, frames, w, h)
    ctx.set_graph_mode(True)
    for _ in range(3):
        ctx.run(B)
    torch.cuda.synchronize()
    flow = ctx.get_flow(0, prm.sc_l).copy()
    import time
    n = 50
    ctx.sync()
    t0 = time.perf_counter()
    for _ in range(n):
        ctx.run(B)
    ctx.sync()
    ms = (time.perf_counter() - t0) * 1e3 / n  # graph replays back to back on one stream, host clock around the batch
    ctx.set_graph_mode(False)
    lev = ctx.profile_levels(B, steps=3)
    row = {"config": name, "pairs": B, "sor_lane": lane, "ms_per_step": round(ms, 4),
           "levels": {str(lv): {"wxh": "%dx%d" % (ctx.level_info(lv)["w"], ctx.level_info(lv)["h"]),
                                "sor_ms": round(lev[lv]["sor"], 4), "assemble_ms": round(lev[lv]["assemble"], 4),
                                "sor_us_per_launch": round(lev[lv]["sor"] * 1e3 / (prm.tv_innerit * (lv + 1)), 2)}
                      for lv in range(prm.sc_l, prm.sc_f + 1)}}
    ctx.close()
    return row, flow


if __name__ == "__main__":
    batches = [int(a) for a in sys.argv[1:]] or [1, 64]
    for name, c in CFGS.items():
        for B in batches:
            if "cfg3" in name and B > 8:
                continue
            flows = []
            for lane in (0, 1):
                row, flow = measure(name, c, B, lane)
                flows.append(flow)
                print(json.dumps(row), flush=True)
            print(json.dumps({"config": name, "pairs": B, "flows_bitwise_equal": bool(np.array_equal(flows[0].view(np.uint32), flows[1].view(np.uint32)))}), flush=True)
