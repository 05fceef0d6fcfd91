"""Generates tests/golden/*.npz from the REFERENCE build (oracle/_ref, i.e. the
reference's own sources compiled in place by oracle/Makefile).  Run in the
container that has /root/reference:

    make -C oracle ref && python tests/golden/make_golden.py

Each fixture holds the uint8 input pair, the parameters (20 CLI numbers + noc +
nop) and the reference flow at level sc_l, plus the patch-stage outputs of the
finest level (p, conv, cnt) for a fixed seeded coarser flow.  reference/runs.npz
keeps, for the larger cases tests/test_oracle.py compares with the reference, the
shape, SHA-256 and a seeded sample of each reference output.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from of_dis_b200 import params, preprocess, synth  # noqa: E402
from oracle import ref_driver  # noqa: E402

CASES = {
    # name: (h, w, channels, cli numbers, nop, amp, stereo)
    "gray_flow_l2": (128, 256, 1, "3 1 12 12 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0", 2, 5.0, False),
    "gray_flow_l1cost": (96, 200, 1, "3 1 16 16 0.05 0.95 0 8 0.4 0 1 1 1 10 10 5 1 3 1.6 0", 2, 5.0, False),
    "gray_flow_huber_p12": (120, 216, 1, "3 1 16 16 0.05 0.95 0 12 0.75 0 1 2 1 10 10 5 1 3 1.6 0", 2, 4.0, False),
    "rgb_flow_l1cost": (104, 184, 3, "3 1 16 16 0.05 0.95 0 12 0.75 0 1 1 1 10 10 5 1 3 1.6 0", 2, 4.0, False),
    "gray_stereo": (96, 224, 1, "3 1 24 24 0.05 0.95 0 12 0.75 0 1 0 1 10 10 5 1 3 1.6 0", 1, 4.0, True),
    "gray_flow_earlyexit": (100, 168, 1, "3 1 16 2 0.05 0.95 0.5 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0", 2, 5.0, False),
    "gray_flow_big_motion": (128, 256, 1, "3 1 12 12 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0", 2, 40.0, False),
    # forward-backward consistency (README parameter 10 = 1): second grid on the swapped images
    "gray_flow_fbcon": (120, 200, 1, "3 1 8 8 0.05 0.95 0 8 0.4 1 1 0 1 10 10 5 1 3 1.6 0", 2, 6.0, False),
    "rgb_flow_fbcon_l1cost": (104, 184, 3, "3 1 8 8 0.05 0.95 0 12 0.75 1 1 1 1 10 10 5 1 3 1.6 0", 2, 4.0, False),
    "gray_stereo_fbcon": (96, 224, 1, "3 1 12 12 0.05 0.95 0 8 0.4 1 1 0 1 10 10 5 1 3 1.6 0", 1, 4.0, True),
}


def reference_runs(out_dir):
    """reference/runs.npz: digests and samples of what the reference build computes for the cases
    tests/test_oracle.py compares the port with (test_oracle.REFERENCE_CASES)."""
    sys.path.insert(0, os.path.dirname(out_dir))
    import test_oracle

    out = {}
    for name in test_oracle.REFERENCE_CASES:
        case = test_oracle.reference_case(name)
        out.update(test_oracle.summarize(case, test_oracle.reference_outputs(case)))
        print(name)
    os.makedirs(os.path.join(out_dir, "reference"), exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, "reference", "runs.npz"), **out)


def main():
    out_dir = os.path.dirname(os.path.abspath(__file__))
    only = sys.argv[1:]  # optional: generate just these fixtures ("reference" = reference/runs.npz)
    if not only or "reference" in only:
        reference_runs(out_dir)
    for name, (h, w, ch, cli, nop, amp, stereo) in CASES.items():
        if only and name not in only:
            continue
        prm = params.from_cli_numbers(cli.split(), noc=ch, nop=nop)
        i0, i1, _ = synth.synthetic_pair(h, w, ch, seed=len(name), amp=amp, stereo=stereo)
        pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
        flow = ref_driver.ref_run(pyr, prm)
        lv = prm.sc_l
        hh, ww = pyr.level_shape(lv + 1)
        rng = np.random.default_rng(7)
        fp = (rng.standard_normal((hh, ww, nop)) * 1.5).astype(np.float32)
        if stereo:
            fp = -np.abs(fp)
        lvl = ref_driver.ref_level_patches(pyr, prm, lv, fp)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), img0=i0, img1=i1,
                            cli=np.array([float(x) for x in cli.split()]), noc=ch, nop=nop, flow=flow,
                            flow_prev=fp, p=lvl["p"], conv=lvl["conv"], cnt=lvl["cnt"], dense=lvl["dense"])
        print(name, flow.shape, float(np.abs(flow).max()))


if __name__ == "__main__":
    main()
