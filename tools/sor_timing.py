"""Per-phase cycle stamps of the two exact SOR kernels on the bench level (1024x436, operating point 2, level 3 =
128x56, the last SOR launch of a run).  The stamps need a build with -DOFDIS_SOR_TIMING, which this tool makes
next to the product library; the product library carries none.
  python tools/sor_timing.py --build    # nvcc: the stamped library into of_dis_b200/lib/exp/
  python tools/sor_timing.py            # on the GPU: sor_wave_kernel's super-step phases, sor_lane_kernel's chunk timeline
Each readout runs in a child process that loads the stamped library through OFDIS_LIB."""
import ctypes, json, os, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
LIB = os.path.join(ROOT, "of_dis_b200", "lib", "exp", "libofdis_sor_timing.so")


def build():
    from of_dis_b200 import build as B
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    cmd = [B._nvcc()] + B.NVCC_FLAGS + ["-DOFDIS_SOR_TIMING"] + [os.path.join(B.CSRC, s) for s in B.SOURCES] + ["-ldl", "-o", LIB]
    subprocess.check_call(cmd)
    print(LIB)


def stamps(nframes, sor_lane):
    """Two runs of the bench pair with the given SOR kernel selection; the stamps of the last SOR launch."""
    import numpy as np
    from of_dis_b200 import api, params, preprocess, synth
    prm = params.operating_point(2, 1024)
    i0, i1, _ = synth.synthetic_pair(436, 1024, 1, seed=0)
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, nframes)
    ctx.set_option("sor_lane", sor_lane)
    for f in range(nframes):
        ctx.upload_pyramids(f, pyr)
    ctx.run(nframes)
    ctx.run(nframes)
    ctx.sync()
    buf = np.zeros(64 * 8 * 16, np.int64)
    assert api.lib().ofdis_debug_sor_times(buf.ctypes.data_as(ctypes.c_void_p)) == 0
    ctx.close()
    return buf


def wave():
    import numpy as np
    t = stamps(8, 0).reshape(64, 8, 16)[:7, :, :7]  # 6 compute warps + the producer, super-steps 40..47
    # compute warps stamp slots 0 (step start), 2 (operands loaded), 4 (arithmetic done), 5 (stores issued), 6 (barrier passed);
    # the producer 0 (start), 1 (bulk copies issued), 2 (stage mbarrier passed), 5 (halo mbarriers passed), 6 (barrier passed)
    for wp in range(7):
        slots = [0, 1, 2, 5, 6] if wp == 6 else [0, 2, 4, 5, 6]
        names = ["issue", "stage wait", "halo wait", "barrier"] if wp == 6 else ["loads", "arithmetic", "stores+prefetch", "barrier"]
        d = np.diff(t[wp][:, slots], axis=1).mean(0).round(0)
        role = "producer" if wp == 6 else "k=%d rows %d.." % (wp // 2, 32 * (wp % 2))
        print("warp %d %-14s %s | step %.0f cycles" % (wp, role, dict(zip(names, d.tolist())), (t[wp, 1:, 0] - t[wp, :-1, 0]).mean()))


def lane():
    t = stamps(1, 1)[:16 * 32 * 4].reshape(16, 32, 4)  # [warp][chunk of 8 steps][slot 0 = start, 3 = end]
    t0 = t[0, 0, 0]
    for wi in range(6):  # 2 bands x 3 sweeps
        chunks = [c for c in range(32) if t[wi, c, 3]]
        print(json.dumps({"timeline": "warp%d(b=%d,k=%d)" % (wi, wi % 2, wi // 2),
                          "first_chunk_start_cycle": int(t[wi, chunks[0], 0] - t0),
                          "last_chunk_end_cycle": int(t[wi, chunks[-1], 3] - t0),
                          "cycles_per_chunk_of_8_steps": [int(t[wi, c, 3] - t[wi, c, 0]) for c in chunks]}))


if __name__ == "__main__":
    if "--build" in sys.argv:
        build()
    elif "--child" in sys.argv:
        {"wave": wave, "lane": lane}[sys.argv[-1]]()
    else:
        if not os.path.exists(LIB):
            sys.exit("%s not found: run `python tools/sor_timing.py --build` first" % LIB)
        for which in ("wave", "lane"):
            print("# sor_%s_kernel" % which, flush=True)
            subprocess.run([sys.executable, os.path.abspath(__file__), "--child", which], env=dict(os.environ, OFDIS_LIB=LIB),
                           check=True, timeout=600)
