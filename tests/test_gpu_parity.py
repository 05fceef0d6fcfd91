"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through
the C-ABI (of_dis_b200/lib/libofdis_b200.so); the oracle (C restatement, pinned
bitwise to the reference build) is only the checker.  Integer/bit-exact bar:
all float outputs must be BITWISE equal, which is stronger than the 1e-3
max-abs bar north_star states for the final .flo."""
import glob
import os

import numpy as np
import pytest

from of_dis_b200 import params, preprocess, synth

pytestmark = pytest.mark.gpu
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_bits(got, exp, name):
    got, exp = np.asarray(got), np.asarray(exp)
    assert got.shape == exp.shape, (name, got.shape, exp.shape)
    if got.dtype.kind == "f":
        bad = bits(got) != bits(exp)
        # +0/-0 and NaN payloads count as different on purpose
        if bad.any():
            d = np.abs(got.astype(np.float64) - exp.astype(np.float64))
            raise AssertionError("%s: %d of %d values differ bitwise, max-abs %.3e, first at %s" %
                                 (name, int(bad.sum()), bad.size, float(np.nanmax(d)), np.argwhere(bad)[0]))
    else:
        assert np.array_equal(got, exp), name


@pytest.fixture(scope="module")
def api():
    from of_dis_b200 import api as _api

    _api.lib()
    return _api


def _golden(path):
    z = np.load(path)
    prm = params.from_cli_numbers(z["cli"], noc=int(z["noc"]), nop=int(z["nop"]))
    pyr = preprocess.PairPyramids(z["img0"], z["img1"], prm.sc_f, prm.p_samp_s)
    return z, prm, pyr


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_golden_fixtures_whole_run_and_patch_stage(path, api):
    """Committed outputs of the reference build (tests/golden/make_golden.py)."""
    z, prm, pyr = _golden(path)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    assert_bits(ctx.get_flow(0, prm.sc_l), z["flow"], "flow")
    # patch stage of the finest level from a prescribed coarser flow (the stage fixture is the plain
    # grid: without the forward-backward merge)
    if prm.usefbcon:
        ctx.close()
        import dataclasses
        prm = dataclasses.replace(prm, usefbcon=0)
        ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
        ctx.upload_pyramids(0, pyr)
    lv = prm.sc_l
    ctx.set_flow(0, lv + 1, z["flow_prev"])
    ctx.patgrid_optimize(lv, 0, 1, True)
    ctx.patgrid_aggregate(lv, 0, 1)
    got = ctx.get_patches(0, lv)
    assert_bits(got["p"], z["p"], "p")
    assert_bits(got["conv"], z["conv"], "conv")
    assert_bits(got["cnt"], z["cnt"], "cnt")
    assert_bits(ctx.get_flow(0, lv), z["dense"], "dense")
    ctx.close()


CASES = {
    # name: (h, w, ch, params, amp, stereo)
    "cfg2_1024x436_gray_op2": (436, 1024, 1, lambda: params.operating_point(2, 1024), 6.0, False),
    "cfg1_640x480_gray_op2": (480, 640, 1, lambda: params.operating_point(2, 640), 6.0, False),
    "gray_op2_motion40": (436, 1024, 1, lambda: params.operating_point(2, 1024), 40.0, False),
    "gray_op1_no_tv": (436, 1024, 1, lambda: params.operating_point(1, 1024), 6.0, False),
    "rgb_op3_l1cost_small": (270, 480, 3, lambda: params.from_cli_numbers(
        "4 1 16 16 0.05 0.95 0 12 0.75 0 1 1 1 10 10 5 1 3 1.6 0".split(), noc=3), 6.0, False),
    "stereo_op4_small": (250, 360, 1, lambda: params.from_cli_numbers(
        "3 1 32 32 0.05 0.95 0 12 0.75 0 1 0 1 10 10 5 1 3 1.6 0".split(), noc=1, nop=1), 6.0, True),
    "gray_p6_nopatnorm_sor5": (200, 320, 1, lambda: params.from_cli_numbers(
        "3 1 8 8 0.05 0.95 0 6 0.5 0 0 0 1 10 10 5 2 5 1.5 0".split()), 6.0, False),
    "gray_early_exit": (200, 320, 1, lambda: params.from_cli_numbers(
        "3 1 16 2 0.05 0.95 0.5 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split()), 6.0, False),
    # 2 SOR sweeps on a 70-row level: rows padded to 128, so one warp of every sweep holds shadow
    # lanes only (the TMA kernel with HPAD = 128)
    "gray_sor2_rows70": (140, 352, 1, lambda: params.from_cli_numbers(
        "2 1 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 2 2 1.6 0".split()), 6.0, False),
    # 1 sweep, 100 rows, wide
    "stereo_sor1_rows100": (200, 416, 1, lambda: params.from_cli_numbers(
        "2 1 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 1 1.8 0".split(), noc=1, nop=1), 6.0, True),
}


@pytest.mark.parametrize("name", list(CASES))
def test_stages_and_whole_run_vs_oracle(name, api, oracle_port):
    h, w, ch, mk, amp, stereo = CASES[name]
    prm = mk()
    i0, i1, _ = synth.synthetic_pair(h, w, ch, seed=1, amp=amp, stereo=stereo)
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    ctx.upload_pyramids(0, pyr)
    lv = prm.sc_l
    hh, ww = pyr.level_shape(lv + 1)
    rng = np.random.default_rng(2)
    fp = (rng.standard_normal((hh, ww, prm.nop)) * 2).astype(np.float32)
    if stereo:
        fp = -np.abs(fp)
    # --- patch stage (K1-K4)
    exp = oracle_port.port_level_patches(pyr, prm, lv, fp)
    ctx.set_flow(0, lv + 1, fp)
    ctx.patgrid_optimize(lv, 0, 1, True)
    ctx.patgrid_aggregate(lv, 0, 1)
    got = ctx.get_patches(0, lv)
    for k in ("p", "pweight", "conv", "cnt"):
        assert_bits(got[k], exp[k], "patch." + k)
    dense = ctx.get_flow(0, lv)
    assert_bits(dense, exp["dense"], "dense")
    # --- refinement (K5-K12), stage by stage then end to end
    if prm.usetvref:
        st = oracle_port.varref_stages(pyr, prm, lv, dense, n_iters=2)
        ctx.varref_refine(lv, 0, 1, n_inner=2)
        for k in ("Ix", "Iy", "Iz", "Ixx", "Ixy", "Iyy", "Ixz", "Iyz"):
            assert_bits(ctx.debug_get(k, 0, lv), st[k], "deriv." + k)
        assert_bits(ctx.debug_get("mask", 0, lv)[0], st["mask"], "mask")
        rec = ctx.debug_get("rec", 0, lv)
        it = st["iters"][1]
        if prm.nop == 2:
            for idx, key in enumerate(("a11_inv", "a12_inv", "a22_inv", "b1", "b2", "sh", "sv")):
                assert_bits(rec[..., idx], it[key], "rec." + key)
        else:
            assert_bits(rec[..., 1], it["b1"], "rec.b1")
            assert_bits(rec[..., 2], it["sh"], "rec.sh")
            assert_bits(rec[..., 3], it["sv"], "rec.sv")
        dudv = ctx.debug_get("dudv", 0, lv)
        assert_bits(dudv[..., 0], it["du"], "du")
        if prm.nop == 2:
            assert_bits(dudv[..., 1], it["dv"], "dv")
        ctx.set_flow(0, lv, dense)
        ctx.varref_refine(lv, 0, 1)
        assert_bits(ctx.get_flow(0, lv), oracle_port.port_level_varref(pyr, prm, lv, dense), "varref")
    # --- whole run
    ctx.run(1)
    assert_bits(ctx.get_flow(0, prm.sc_l), oracle_port.port_run(pyr, prm), "run")
    ctx.close()


def test_batch_of_frames_and_graph_replay(api, oracle_port):
    """cfg 4 in miniature: 8 distinct pairs in one launch == 8 single runs; graph replay == eager."""
    prm = params.operating_point(2, 1024)
    nfr = 8
    pyrs = []
    for s in range(nfr):
        i0, i1, _ = synth.synthetic_pair(436, 1024, 1, seed=100 + s)
        pyrs.append(preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s))
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, nfr)
    packed = np.stack([ctx.pack_frame(p) for p in pyrs])
    ctx.upload_packed(0, nfr, packed)
    ctx.run(nfr)
    eager = [ctx.get_flow(f, prm.sc_l) for f in range(nfr)]
    for f in (0, 3, 7):
        assert_bits(eager[f], oracle_port.port_run(pyrs[f], prm), "frame %d" % f)
    before = ctx.launch_count
    ctx.set_graph_mode(True)
    ctx.run(nfr)
    ctx.run(nfr)
    for f in range(nfr):
        assert_bits(ctx.get_flow(f, prm.sc_l), eager[f], "graph frame %d" % f)
    assert ctx.launch_count > before
    ctx.close()


def test_bench_batch_of_64_pairs_vs_oracle(api, oracle_port):
    """The bench workload itself (bench.py: 64 pairs per launch, 16 distinct, graph replay): every frame of the batch
    equals the oracle's flow of its pair -- six distinct pairs against the oracle, all 64 slots against those."""
    prm = params.operating_point(2, 1024)
    nfr, ndist = 64, 16
    pyrs = []
    for s in range(ndist):
        i0, i1, _ = synth.synthetic_pair(436, 1024, 1, seed=s)
        pyrs.append(preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s))
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, nfr)
    packed = np.stack([ctx.pack_frame(pyrs[f % ndist]) for f in range(nfr)])
    ctx.upload_packed(0, nfr, packed)
    ctx.set_graph_mode(True)
    ctx.run(nfr)
    ctx.run(nfr)
    flows = [ctx.get_flow(f, prm.sc_l) for f in range(nfr)]
    ctx.close()
    for d in (0, 3, 6, 9, 12, 15):
        assert_bits(flows[d], oracle_port.port_run(pyrs[d], prm), "pair %d" % d)
    for f in range(nfr):
        assert_bits(flows[f], flows[f % ndist], "slot %d" % f)


def test_properties_at_full_size(api):
    """Size-independent properties at BASELINE cfg 2 size: identical images -> exactly zero flow;
    the reference-shaped OFClass wrapper gives the same result as the batch engine."""
    prm = params.operating_point(2, 1024)
    i0, i1, gt = synth.synthetic_pair(436, 1024, 1, seed=5)
    pyr = preprocess.PairPyramids(i0, i0, prm.sc_f, prm.p_samp_s)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    assert np.abs(ctx.get_flow(0, prm.sc_l)).max() == 0.0
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    a = ctx.get_flow(0, prm.sc_l)
    ctx.close()
    out = np.zeros_like(a)
    api.OFClass(pyr.i0, pyr.i0x, pyr.i0y, pyr.i1, pyr.i1x, pyr.i1y, pyr.imgpadding, out, None, pyr.width, pyr.height,
                prm.sc_f, prm.sc_l, prm.max_iter, prm.min_iter, prm.dp_thresh, prm.dr_thresh, prm.res_thresh,
                prm.p_samp_s, prm.patove, prm.usefbcon, prm.costfct, prm.noc, prm.patnorm, prm.usetvref, prm.tv_alpha,
                prm.tv_gamma, prm.tv_delta, prm.tv_innerit, prm.tv_solverit, prm.tv_sor, 0)
    assert_bits(out, a, "OFClass wrapper")
    full = preprocess.postprocess(a, prm.sc_l, pyr.padw, pyr.padh, pyr.width_org, pyr.height_org)
    epe = np.sqrt(((full - gt) ** 2).sum(-1)).mean()
    assert epe < 0.5, epe


@pytest.mark.parametrize("rt", [1, 2, 4])
def test_tall_level_1024_rows_runs_as_a_cluster_of_bands(rt, api, oracle_port):
    """Refinement level with exactly 1024 rows (as in BASELINE configs[4]'s level 1; 8 bands of 128 rows,
    one CTA of a thread-block cluster each, tiles of 1, 2 or 4 rows per thread): narrow stereo pair so the
    oracle stays fast."""
    prm = params.from_cli_numbers("2 1 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split(), noc=1, nop=1)
    i0, i1, _ = synth.synthetic_pair(2048, 96, 1, seed=9, amp=3.0, stereo=True)
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    ctx.set_option("sor_rows_per_thread", rt)
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    assert_bits(ctx.get_flow(0, prm.sc_l), oracle_port.port_run(pyr, prm), "run h=1024")
    ctx.close()


@pytest.mark.parametrize("nop,rows,sweeps,rt", [(2, 1100, 3, 2), (1, 2048, 2, 2), (2, 1101, 3, 4), (2, 1100, 3, 1), (1, 4090, 1, 4)])  # 4090 rows need a 16-CTA cluster
def test_levels_taller_than_1024_rows(nop, rows, sweeps, rt, api, oracle_port):
    """Levels beyond 8 x 128 rows (the round-1 kernel refused these): more rows per band, fewer sweeps per
    launch when the stage ring no longer fits; odd heights; 4090 rows = 8 bands of 512 rows, 4 rows per thread."""
    prm = params.from_cli_numbers(("1 0 6 6 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 %d 1.6 0" % sweeps).split(), noc=1, nop=nop)
    i0, i1, _ = synth.synthetic_pair(rows, 72, 1, seed=11, amp=2.0, stereo=(nop == 1))
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    try:
        ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    except api.OfdisError:
        if rows > 2048:
            pytest.skip("device grants no 16-CTA clusters")
        raise
    ctx.set_option("sor_rows_per_thread", rt)
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    assert_bits(ctx.get_flow(0, prm.sc_l), oracle_port.port_run(pyr, prm), "run h=%d" % rows)
    ctx.close()


CLUSTER_CASES = ["cfg2_1024x436_gray_op2", "rgb_op3_l1cost_small", "stereo_op4_small", "gray_p6_nopatnorm_sor5",
                 "gray_sor2_rows70", "stereo_sor1_rows100"]


@pytest.mark.parametrize("single_max,rt", [(32, 1), (64, 1), (32, 2)])
@pytest.mark.parametrize("name", CLUSTER_CASES)
def test_cluster_sor_on_small_levels_vs_oracle(name, single_max, rt, api, oracle_port):
    """ofdis_set_option("sor_single_max" / "sor_rows_per_thread"): the same levels solved by a cluster of bands of
    32 or 64 lanes (1 or 2 rows each) instead of one CTA (2..5 bands, partial last bands, odd heights, 1..5
    sweeps, flow and stereo) -- dudv after two inner iterations and the whole run, bitwise; two frames per
    launch so that consecutive clusters share the grid."""
    h, w, ch, mk, amp, stereo = CASES[name]
    prm = mk()
    pyrs = []
    for s in range(2):
        i0, i1, _ = synth.synthetic_pair(h, w, ch, seed=1 + s, amp=amp, stereo=stereo)
        pyrs.append(preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s))
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, 2)
    ctx.set_option("sor_lane", 0)  # this test is about the block wavefront (sor_wave_kernel)
    ctx.set_option("sor_single_max", single_max)
    ctx.set_option("sor_rows_per_thread", rt)
    for f, p in enumerate(pyrs):
        ctx.upload_pyramids(f, p)
    lv = prm.sc_l
    hh, ww = pyrs[0].level_shape(lv)
    rng = np.random.default_rng(3)
    dense = (rng.standard_normal((hh, ww, prm.nop)) * 1.5).astype(np.float32)
    if stereo:
        dense = -np.abs(dense)
    st = oracle_port.varref_stages(pyrs[1], prm, lv, dense, n_iters=2)
    ctx.set_flow(1, lv, dense)
    ctx.varref_refine(lv, 0, 2, n_inner=2)
    dudv = ctx.debug_get("dudv", 1, lv)
    assert_bits(dudv[..., 0], st["iters"][1]["du"], "du")
    if prm.nop == 2:
        assert_bits(dudv[..., 1], st["iters"][1]["dv"], "dv")
    ctx.set_graph_mode(True)
    ctx.run(2)
    for f, p in enumerate(pyrs):
        assert_bits(ctx.get_flow(f, prm.sc_l), oracle_port.port_run(p, prm), "run, frame %d" % f)
    ctx.close()


@pytest.mark.parametrize("rt", [1, 4])
@pytest.mark.parametrize("name", ["cfg2_1024x436_gray_op2", "stereo_op4_small", "gray_p6_nopatnorm_sor5", "gray_sor2_rows70"])
def test_sor_tile_heights_vs_oracle(name, rt, api, oracle_port):
    """Tiles of 1 and 4 rows per SOR thread (the default is 2) give the same bits."""
    h, w, ch, mk, amp, stereo = CASES[name]
    prm = mk()
    i0, i1, _ = synth.synthetic_pair(h, w, ch, seed=3, amp=amp, stereo=stereo)
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    ctx.set_option("sor_lane", 0)
    ctx.set_option("sor_rows_per_thread", rt)
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    assert_bits(ctx.get_flow(0, prm.sc_l), oracle_port.port_run(pyr, prm), "run rt=%d" % rt)
    ctx.close()


@pytest.mark.parametrize("pdl", [0, 1])
@pytest.mark.parametrize("name", ["cfg2_1024x436_gray_op2", "rgb_op3_l1cost_small", "stereo_op4_small"])
def test_programmatic_dependent_launch_vs_oracle(name, pdl, api, oracle_port):
    """ofdis_set_option("pdl"): every kernel starts with griddepcontrol.wait; with the launch attribute the next kernel
    is scheduled while the current one drains.  Eager and graph replay, four frames per launch, several replays:
    the reference's bits every time."""
    h, w, ch, mk, amp, stereo = CASES[name]
    prm = mk()
    pyrs = []
    for s in range(4):
        i0, i1, _ = synth.synthetic_pair(h, w, ch, seed=21 + s, amp=amp, stereo=stereo)
        pyrs.append(preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s))
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, 4)
    ctx.set_option("pdl", pdl)
    for f, p in enumerate(pyrs):
        ctx.upload_pyramids(f, p)
    exp = [oracle_port.port_run(p, prm) for p in pyrs]
    for graph in (False, True):
        ctx.set_graph_mode(graph)
        for rep in range(3):
            ctx.run(4)
            for f in range(4):
                assert_bits(ctx.get_flow(f, prm.sc_l), exp[f], "pdl=%d graph=%s replay %d frame %d" % (pdl, graph, rep, f))
    ctx.close()


LANE_CASES = ["cfg2_1024x436_gray_op2", "cfg1_640x480_gray_op2", "rgb_op3_l1cost_small", "stereo_op4_small",
              "gray_p6_nopatnorm_sor5", "gray_sor2_rows70", "stereo_sor1_rows100"]


@pytest.mark.parametrize("lane", [1, 0])
@pytest.mark.parametrize("name", LANE_CASES)
def test_lane_sor_and_block_sor_vs_oracle(name, lane, api, oracle_port):
    """ofdis_set_option("sor_lane"): the pixel wavefront (sor_lane_kernel: warps synchronised through shared-memory
    flags; 1..5 bands of 32 rows, partial last bands, 1..5 sweeps -- more than fit one launch included --, flow and
    stereo) and the block wavefront (sor_wave_kernel) give the reference's bits: (du,dv) after two inner
    iterations and the whole run, three frames per launch, graph replay."""
    h, w, ch, mk, amp, stereo = CASES[name]
    prm = mk()
    pyrs = []
    for s in range(3):
        i0, i1, _ = synth.synthetic_pair(h, w, ch, seed=11 + s, amp=amp, stereo=stereo)
        pyrs.append(preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s))
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, 3)
    ctx.set_option("sor_lane", lane)
    for f, p in enumerate(pyrs):
        ctx.upload_pyramids(f, p)
    lv = prm.sc_l
    hh, ww = pyrs[0].level_shape(lv)
    rng = np.random.default_rng(5)
    dense = (rng.standard_normal((hh, ww, prm.nop)) * 1.5).astype(np.float32)
    if stereo:
        dense = -np.abs(dense)
    st = oracle_port.varref_stages(pyrs[2], prm, lv, dense, n_iters=2)
    ctx.set_flow(2, lv, dense)
    ctx.varref_refine(lv, 0, 3, n_inner=2)
    rec = ctx.debug_get("rec", 2, lv)
    it = st["iters"][1]
    assert_bits(rec[..., 1 if prm.nop == 1 else 3], it["b1"], "rec.b1")
    dudv = ctx.debug_get("dudv", 2, lv)
    assert_bits(dudv[..., 0], it["du"], "du")
    if prm.nop == 2:
        assert_bits(dudv[..., 1], it["dv"], "dv")
    ctx.set_graph_mode(True)
    for _ in range(2):
        ctx.run(3)
    for f, p in enumerate(pyrs):
        assert_bits(ctx.get_flow(f, prm.sc_l), oracle_port.port_run(p, prm), "run, frame %d" % f)
    ctx.close()


def test_cluster_of_sixteen_bands_where_the_device_grants_it(api, oracle_port):
    """Non-portable cluster size 16: 1100-row level as 9 bands of 64 lanes x 2 rows (all sweeps in flight)."""
    prm = params.from_cli_numbers("1 0 6 6 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split(), noc=1, nop=2)
    i0, i1, _ = synth.synthetic_pair(1100, 72, 1, seed=11, amp=2.0)
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    try:
        ctx.set_option("sor_max_cluster", 16)
    except api.OfdisError:
        ctx.close()
        pytest.skip("device grants no 16-CTA clusters")
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    assert_bits(ctx.get_flow(0, prm.sc_l), oracle_port.port_run(pyr, prm), "run h=1100, cluster 16")
    ctx.close()


def test_full_size_rgb_op3_l1_cost_vs_oracle(api, oracle_port):
    """BASELINE configs[2]: run_OF_RGB geometry, 1920x1080, op-point-3 parameters with L1 cost."""
    prm = params.from_cli_numbers("6 2 16 16 0.05 0.95 0 12 0.75 0 1 1 1 10 10 5 1 3 1.6 0".split(), noc=3)
    i0, i1, _ = synth.synthetic_pair(1080, 1920, 3, seed=2)
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    assert_bits(ctx.get_flow(0, prm.sc_l), oracle_port.port_run(pyr, prm), "cfg3 run")
    ctx.close()


@pytest.mark.parametrize("ch", [1, 3])
def test_images_only_upload_derives_the_same_gradients_on_device(ch, api):
    """ofdis_upload_packed_images (I0,I1 only; Sobel/8 on the device) == full upload, bit for bit."""
    prm = params.from_cli_numbers("3 1 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split(), noc=ch)
    nfr = 3
    pyrs = []
    for s in range(nfr):
        i0, i1, _ = synth.synthetic_pair(120, 200, ch, seed=60 + s)  # odd level sizes: 15x25 at level 3
        pyrs.append(preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s))
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, nfr)
    full = np.stack([ctx.pack_frame(p) for p in pyrs])
    ctx.upload_packed(0, nfr, full)
    ctx.run(nfr)
    ref = [ctx.get_flow(f, prm.sc_l) for f in range(nfr)]
    ni = ctx.packed_images_frame_floats
    assert 0 < ni < ctx.packed_frame_floats
    ctx.upload_packed(0, nfr, np.zeros_like(full))          # wipe, then images only
    ctx.upload_packed_images(0, nfr, np.ascontiguousarray(full[:, :ni]))
    ctx.run(nfr)
    for f in range(nfr):
        assert_bits(ctx.get_flow(f, prm.sc_l), ref[f], "frame %d" % f)
    ctx.close()


def _frames_u8(pairs):
    """[frame][2][h][w][C] uint8 block as ofdis_upload_frames_u8 takes it."""
    return np.ascontiguousarray(np.stack([np.stack([a, b]) for a, b in pairs]))


@pytest.mark.parametrize("ch,size", [(1, (436, 1024)), (3, (121, 203)), (1, (128, 256))])
def test_device_pyramid_from_8bit_frames_equals_the_host_pyramid(ch, size, api):
    """ofdis_upload_frames_u8 (divisibility padding, box-mean levels, Sobel/8, border padding on the
    device; run_dense.cpp:130-178,298-311) reproduces preprocess.PairPyramids bit for bit -- every
    padded array of every level -- and therefore the same flow."""
    prm = params.operating_point(2, size[1], noc=ch) if size[1] >= 256 else \
        params.from_cli_numbers("3 1 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split(), noc=ch)
    nfr = 2
    pairs = [synth.synthetic_pair(size[0], size[1], ch, seed=70 + s)[:2] for s in range(nfr)]
    pyrs = [preprocess.PairPyramids(a, b, prm.sc_f, prm.p_samp_s) for a, b in pairs]
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, nfr)
    ctx.upload_frames_u8(0, nfr, _frames_u8(pairs), size[1], size[0])
    for f, p in enumerate(pyrs):
        for lv in range(prm.sc_l, prm.sc_f + 1):
            for which, exp in enumerate((p.i0[lv], p.i0x[lv], p.i0y[lv], p.i1[lv])):
                assert_bits(ctx.get_level(f, lv, which), exp, "frame %d level %d array %d" % (f, lv, which))
    ctx.run(nfr)
    got = [ctx.get_flow(f, prm.sc_l) for f in range(nfr)]
    for f, p in enumerate(pyrs):
        ctx.upload_pyramids(f, p)
    ctx.run(nfr)
    for f in range(nfr):
        assert_bits(got[f], ctx.get_flow(f, prm.sc_l), "flow of frame %d" % f)
    ctx.close()


@pytest.mark.parametrize("ch", [1, 3])
def test_finest_level_upload_derives_the_rest_on_device(ch, api):
    """ofdis_upload_finest_level: un-padded I0,I1 of level sc_l in, everything else derived."""
    prm = params.from_cli_numbers("4 2 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split(), noc=ch)
    nfr = 3
    pairs = [synth.synthetic_pair(144, 208, ch, seed=80 + s)[:2] for s in range(nfr)]
    pyrs = [preprocess.PairPyramids(a, b, prm.sc_f, prm.p_samp_s) for a, b in pairs]
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, nfr)
    P, l = pyrs[0].imgpadding, prm.sc_l
    packed = np.ascontiguousarray(np.stack([np.stack([p.i0[l][P:-P, P:-P], p.i1[l][P:-P, P:-P]]) for p in pyrs]))
    assert packed[0].size == ctx.finest_level_frame_floats
    ctx.upload_finest_level(0, nfr, packed)
    for f, p in enumerate(pyrs):
        for lv in range(prm.sc_l, prm.sc_f + 1):
            for which, exp in enumerate((p.i0[lv], p.i0x[lv], p.i0y[lv], p.i1[lv])):
                assert_bits(ctx.get_level(f, lv, which), exp, "frame %d level %d array %d" % (f, lv, which))
    ctx.close()


@pytest.mark.parametrize("nop,size,op", [(2, (436, 1024), 2), (1, (121, 203), None), (2, (64, 128), 0)])
def test_fullres_output_stage_equals_postprocess(nop, size, op, api):
    """ofdis_get_flow_fullres (x2^lv_l, bilinear x2^lv_l, crop; run_dense.cpp:407-414) ==
    preprocess.postprocess of the level flow, bit for bit."""
    if op == 2:
        prm = params.operating_point(2, size[1], nop=nop)
    elif op == 0:  # lv_l = 0: plain crop
        prm = params.from_cli_numbers("2 0 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split(), nop=nop)
    else:
        prm = params.from_cli_numbers("3 1 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split(), nop=nop)
    nfr = 2
    pairs = [synth.synthetic_pair(size[0], size[1], 1, seed=90 + s)[:2] for s in range(nfr)]
    pyrs = [preprocess.PairPyramids(a, b, prm.sc_f, prm.p_samp_s) for a, b in pairs]
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, nfr)
    for f, p in enumerate(pyrs):
        ctx.upload_pyramids(f, p)
    ctx.run(nfr)
    out = np.empty((nfr, size[0], size[1], nop), np.float32)
    ctx.get_flow_fullres(0, nfr, out, size[1], size[0])
    ctx.sync()
    for f, p in enumerate(pyrs):
        exp = preprocess.postprocess(ctx.get_flow(f, prm.sc_l), prm.sc_l, p.padw, p.padh, size[1], size[0])
        assert_bits(out[f], exp.reshape(out[f].shape), "frame %d" % f)
    ctx.close()


def test_full_size_stereo_op4_vs_oracle(api, oracle_port):
    """BASELINE configs[4]: run_DE_INT geometry, 2880x1988 (Middlebury shape), operating point 4
    (P=12, 128 iterations, levels 6..1; level 1 has 994 rows -- the tall-level SOR variant)."""
    prm = params.operating_point(4, 2880, noc=1, nop=1)
    i0, i1, _ = synth.synthetic_pair(1988, 2880, 1, seed=4, amp=6.0, stereo=True)
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    assert_bits(ctx.get_flow(0, prm.sc_l), oracle_port.port_run(pyr, prm), "cfg5 run")
    ctx.close()


FB_CASES = [
    (2, 1, "3 1 8 8 0.05 0.95 0 8 0.4 1 1 0 1 10 10 5 1 3 1.6 0", (120, 200), 3.0),
    (1, 1, "3 1 8 8 0.05 0.95 0 8 0.4 1 1 0 1 10 10 5 1 3 1.6 0", (120, 200), 3.0),
    (2, 3, "4 2 6 4 0.05 0.95 0 12 0.75 1 1 1 1 10 10 5 1 3 1.6 0", (144, 208), 3.0),
    (1, 3, "3 0 6 4 0.05 0.95 0 8 0.5 1 0 2 0 10 10 5 1 3 1.6 0", (64, 96), 3.0),
    (2, 1, "3 1 8 8 0.05 0.95 0 8 0.4 1 1 0 1 10 10 5 1 3 1.6 0", (120, 200), 14.0),
    (2, 1, "2 2 8 8 0.05 0.95 0 8 0.4 1 1 0 1 10 10 5 1 3 1.6 0", (64, 96), 2.0),   # one level only
    (2, 1, "5 3 12 12 0.05 0.95 0 8 0.4 1 1 0 1 10 10 5 1 3 1.6 0", (436, 1024), 6.0),  # operating point 2 of cfg 2 + fbcon
]


@pytest.mark.parametrize("nop,ch,numbers,size,amp", FB_CASES)
def test_forward_backward_consistency_vs_oracle(nop, ch, numbers, size, amp, api, oracle_port):
    """usefbcon = 1 (README parameter 10): second grid on the swapped images, merged densification
    (patchgrid.cpp:278-375), backward refinement on all but the last level -- bitwise against the oracle,
    for a batch of pairs and through the image-only upload (backward gradients derived on the device)."""
    prm = params.from_cli_numbers(numbers.split(), noc=ch, nop=nop)
    nfr = 2
    pyrs = []
    for s in range(nfr):
        i0, i1, _ = synth.synthetic_pair(size[0], size[1], ch, seed=50 + s, stereo=(nop == 1), amp=amp)
        pyrs.append(preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s))
    exp = [oracle_port.port_run(p, prm) for p in pyrs]
    ctx = api.Context(prm, pyrs[0].width, pyrs[0].height, pyrs[0].imgpadding, nfr)
    for f, p in enumerate(pyrs):
        ctx.upload_pyramids(f, p)
    ctx.run(nfr)
    for f in range(nfr):
        assert_bits(ctx.get_flow(f, prm.sc_l), exp[f], "frame %d" % f)
    # graph replay + finest-level upload: the device builds both directions' pyramids and gradients
    P, l = pyrs[0].imgpadding, prm.sc_l
    packed = np.ascontiguousarray(np.stack([np.stack([p.i0[l][P:-P, P:-P], p.i1[l][P:-P, P:-P]]) for p in pyrs]))
    ctx.upload_finest_level(0, nfr, packed)
    ctx.set_graph_mode(True)
    ctx.run(nfr)
    ctx.run(nfr)
    out = np.empty((nfr,) + exp[0].shape, np.float32)
    ctx.get_flow_batch(0, nfr, out)
    ctx.sync()
    for f in range(nfr):
        assert_bits(out[f], exp[f], "graph + finest-level upload, frame %d" % f)
    ctx.close()


def _random_config(rng):
    """A valid parameter set / image size drawn from the ranges the reference's CLI accepts."""
    P = int(rng.choice([4, 6, 8, 10, 12, 16]))
    ch = int(rng.choice([1, 3]))
    nop = int(rng.choice([1, 2]))
    nlev = int(rng.integers(1, 4))
    sc_l = int(rng.integers(0, 3))
    sc_f = sc_l + nlev - 1
    # coarsest level 6..24 x 8..30 pixels (the reference's 5-tap vertical filter reads out of bounds
    # below 4 rows, image.c:401-434); the finest level stays below ~100 x 120
    h = int(rng.integers(6, 25 >> (nlev - 1)) + 1) << sc_f if (25 >> (nlev - 1)) > 6 else 6 << sc_f
    w = int(rng.integers(8, max(9, 31 >> (nlev - 1)) + 1)) << sc_f
    max_iter = int(rng.integers(1, 20))
    min_iter = int(rng.integers(0, max_iter + 1))
    numbers = [sc_f, sc_l, max_iter, min_iter, float(rng.choice([0.05, 0.2, 0.5])), float(rng.choice([0.95, 0.8, 0.5])),
               float(rng.choice([0.0, 0.5, 2.0])), P, float(rng.choice([0.0, 0.3, 0.4, 0.5, 0.75, 0.9])),
               int(rng.integers(0, 2)), int(rng.integers(0, 2)), int(rng.integers(0, 3)), int(rng.integers(0, 2)),
               float(rng.choice([10.0, 3.0, 30.0])), float(rng.choice([10.0, 0.0, 5.0])), float(rng.choice([5.0, 0.0, 12.0])),
               int(rng.integers(1, 3)), int(rng.integers(1, 6)), float(rng.choice([1.6, 1.0, 1.9])), 0]
    return numbers, ch, nop, (h, w), float(rng.choice([1.0, 4.0, 12.0]))


@pytest.mark.parametrize("seed", range(40))
def test_random_configurations_vs_oracle(seed, api, oracle_port):
    """Seeded sweep over the parameter space (patch sizes 4..16, overlaps 0..0.9, 1..3 levels, early
    exit thresholds, all three costs, patnorm on/off, refinement on/off with varied weights and sweep
    counts, gray/RGB, flow/stereo, forward-backward on/off): whole run, bitwise against the oracle."""
    rng = np.random.default_rng(1000 + seed)
    numbers, ch, nop, size, amp = _random_config(rng)
    prm = params.from_cli_numbers(numbers, noc=ch, nop=nop)
    i0, i1, _ = synth.synthetic_pair(size[0], size[1], ch, seed=200 + seed, stereo=(nop == 1), amp=amp)
    pyr = preprocess.PairPyramids(i0, i1, prm.sc_f, prm.p_samp_s)
    exp = oracle_port.port_run(pyr, prm)
    ctx = api.Context(prm, pyr.width, pyr.height, pyr.imgpadding, 1)
    ctx.upload_pyramids(0, pyr)
    ctx.run(1)
    assert_bits(ctx.get_flow(0, prm.sc_l), exp, "config %s ch=%d nop=%d size=%s" % (numbers, ch, nop, size))
    ctx.close()
