"""BASELINE configs[2] (1920x1080 RGB, op-3 geometry, L1 cost) and configs[4] (2880x1988 stereo, op 4) on
one GPU: step time and, per kernel class, the achieved algorithmic GB/s (SURVEY 8d formulas) -- the
levels of these configs are the ones that stream from HBM.  Also the SOR time per pyramid level.
python tools/big_configs.py [B ...] [--opt name=value ...] [--cfg substring]"""
import os, sys, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from of_dis_b200 import api, params, preprocess, synth

CFGS = {
    "cfg3_1920x1080_rgb_l1": dict(size=(1080, 1920), ch=3, nop=2, prm=lambda: params.from_cli_numbers(
        "6 2 16 16 0.05 0.95 0 12 0.75 0 1 1 1 10 10 5 1 3 1.6 0".split(), noc=3)),
    "cfg5_2880x1988_stereo_op4": dict(size=(1988, 2880), ch=1, nop=1, prm=lambda: params.operating_point(4, 2880, noc=1, nop=1)),
}


def measure(name, c, B, opts):
    prm = c["prm"]()
    h, w = c["size"]
    st = torch.cuda.current_stream()
    i0, i1, _ = synth.synthetic_pair(h, w, c["ch"], seed=1, stereo=(c["nop"] == 1), amp=6.0)
    scf = 1 << prm.sc_f
    W, H = (w + scf - 1) // scf * scf, (h + scf - 1) // scf * scf
    ctx = api.Context(prm, W, H, prm.p_samp_s, B, stream=st.cuda_stream)
    for k, v in opts.items():
        ctx.set_option(k, v)
    frames = np.ascontiguousarray(np.stack([np.stack([i0, i1])] * B))
    ctx.upload_frames_u8(0, B, frames, w, h)
    ctx.set_graph_mode(True)
    for _ in range(2): ctx.run(B)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 5
    a.record(st)
    for _ in range(n): ctx.run(B)
    b.record(st); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / n
    ctx.set_graph_mode(False)
    prof = ctx.profile_kernels(B, steps=2)
    lev = ctx.profile_levels(B, steps=2)
    # algorithmic bytes per step (SURVEY 8d)
    C, nop, P = prm.noc, prm.nop, prm.p_samp_s
    b_dis = b_sor = b_asm = b_setup = 0
    sor_lv = {}
    for lv in range(prm.sc_l, prm.sc_f + 1):
        g = ctx.level_info(lv)
        wl, hl = g["w"], g["h"]
        n_inner = prm.tv_innerit * (lv + 1)
        b_dis += 4 * (4 * C * (wl + 2 * P) * (hl + 2 * P) + nop * (wl // 2) * (hl // 2) * (lv < prm.sc_f) + nop * wl * hl)
        bs = n_inner * (44 if nop == 2 else 24) * wl * hl
        b_sor += bs
        b_asm += n_inner * 4 * wl * hl * (14 + 8 * C)
        b_setup += 4 * wl * hl * (2 * C + nop) + 4 * wl * hl * (8 * C + 1)
        steps = n_inner * ((wl + 3) // 4 + hl + 2 * prm.tv_solverit + 1)
        sor_lv[str(lv)] = {"wxh": "%dx%d" % (wl, hl), "ms": round(lev[lv]["sor"], 3),
                           "alg_GBps": round(bs * B / (lev[lv]["sor"] * 1e-3) / 1e9, 1),
                           "us_per_superstep": round(lev[lv]["sor"] * 1e3 / steps, 3),
                           "patch_ms": round(lev[lv]["patch"], 3)}
    alg = {"patch": b_dis, "densify": 0, "vr_setup": b_setup, "assemble": b_asm, "sor": b_sor}
    row = {"config": name, "pairs": B, "options": opts, "ms_per_step": round(ms, 3), "mpix_per_s": round(B * w * h / ms / 1e3, 1),
           "classes": {k: {"ms": round(v["ms_per_step"], 3), "launches": v["launches_per_step"],
                           "alg_GBps": round(alg[k] * B / (v["ms_per_step"] * 1e-3) / 1e9, 1) if alg.get(k) else None}
                       for k, v in prof.items()},
           "sor_levels": sor_lv}
    ctx.close()
    return row


if __name__ == "__main__":
    args = sys.argv[1:]
    opts, only, batches = {}, None, []
    while args:
        a = args.pop(0)
        if a == "--opt":
            k, v = args.pop(0).split("=")
            opts[k] = int(v)
        elif a == "--cfg":
            only = args.pop(0)
        else:
            batches.append(int(a))
    st = torch.cuda.Stream(); torch.cuda.set_stream(st)
    for name, c in CFGS.items():
        if only and only not in name:
            continue
        for B in batches or [1, 8]:
            print(json.dumps(measure(name, c, B, opts)), flush=True)
