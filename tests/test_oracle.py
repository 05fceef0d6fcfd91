"""CPU tests of the checker itself: the C restatement (oracle/dis_oracle.c) must
equal (a) the committed golden fixtures produced by the reference build and
(b) what the reference build computed on the inputs of the GPU suite (stored digests
under tests/golden/reference/; where oracle/_ref exists, the reference build itself
must reproduce them too) -- bit for bit."""
import glob
import hashlib
import os

import numpy as np
import pytest

from of_dis_b200 import params, preprocess, synth
from oracle import ref_driver

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))


def _load(path):
    z = np.load(path)
    prm = params.from_cli_numbers(z["cli"], noc=int(z["noc"]), nop=int(z["nop"]))
    pyr = preprocess.PairPyramids(z["img0"], z["img1"], prm.sc_f, prm.p_samp_s)
    return z, prm, pyr


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_port_matches_golden_bitwise(path, oracle_port):
    z, prm, pyr = _load(path)
    flow = oracle_port.port_run(pyr, prm)
    assert np.array_equal(bits(flow), bits(z["flow"]))
    lvl = oracle_port.port_level_patches(pyr, prm, prm.sc_l, z["flow_prev"])
    assert np.array_equal(bits(lvl["p"]), bits(z["p"]))
    assert np.array_equal(lvl["conv"], z["conv"]) and np.array_equal(lvl["cnt"], z["cnt"])
    assert np.array_equal(bits(lvl["dense"]), bits(z["dense"]))


@pytest.mark.skipif(not ref_driver.ref_available("m1c1"), reason="oracle/_ref not built")
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_reference_build_reproduces_golden(path):
    z, prm, pyr = _load(path)
    if not ref_driver.ref_available(prm.flavour()):
        pytest.skip("flavour not built")
    assert np.array_equal(bits(ref_driver.ref_run(pyr, prm)), bits(z["flow"]))


def test_port_vs_reference_cfg1_and_stages(oracle_port):
    """BASELINE config 1 (640x480 gray, op-point 2) whole run, plus per-stage checks."""
    case = reference_case("cfg1")
    _, prm, _, (pyr,) = case
    lv = prm.sc_l
    fl = _cfg1_flow(pyr, prm)  # variational refinement alone, on an arbitrary smooth-ish flow
    assert_reference(case, {"flow": oracle_port.port_run(pyr, prm), "varref": oracle_port.port_level_varref(pyr, prm, lv, fl)})
    st = oracle_port.varref_stages(pyr, prm, lv, fl)
    out = np.stack([st["uu"], st["vv"]], -1)
    assert np.array_equal(bits(out), bits(oracle_port.port_level_varref(pyr, prm, lv, fl)))


def test_packet_order_sum_is_the_documented_order(oracle_port):
    import ctypes

    rng = np.random.default_rng(5)
    for n in (1, 3, 4, 7, 8, 12, 36, 64, 100, 144, 432):
        v = (rng.standard_normal(n) * 100).astype(np.float32)
        got = np.float32(oracle_port.lib().dis_sum_packet_order(v.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), n))
        n4, n8 = n // 4 * 4, n // 8 * 8
        if n4:
            a = v[0:4].copy()
            if n4 > 4:
                b = v[4:8].copy()
                for i in range(8, n8, 8):
                    a = a + v[i:i + 4]
                    b = b + v[i + 4:i + 8]
                a = a + b
                if n4 > n8:
                    a = a + v[n8:n8 + 4]
            r = np.float32(np.float32(a[0] + a[2]) + np.float32(a[1] + a[3]))
            for i in range(n4, n):
                r = np.float32(r + v[i])
        else:
            r = v[0]
            for i in range(1, n):
                r = np.float32(r + v[i])
        assert got == r


def test_properties_zero_flow_and_translation(oracle_port):
    """SURVEY section 4(iii): identical images -> zero flow; integer shift recovered."""
    i0, _, _ = synth.synthetic_pair(128, 192, 1, seed=11)
    prm = params.from_cli_numbers("3 1 12 12 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split())
    pyr = preprocess.PairPyramids(i0, i0, prm.sc_f, prm.p_samp_s)
    assert np.abs(oracle_port.port_run(pyr, prm)).max() == 0.0
    big, _, _ = synth.synthetic_pair(128, 192 + 8, 1, seed=12)
    a, b = np.ascontiguousarray(big[:, 4:-4]), np.ascontiguousarray(big[:, 2:-6])  # I1(x+2) = I0(x)
    pyr = preprocess.PairPyramids(a, b, prm.sc_f, prm.p_samp_s)
    fl = preprocess.postprocess(oracle_port.port_run(pyr, prm), prm.sc_l, pyr.padw, pyr.padh, 192, 128)
    inner = fl[16:-16, 16:-16]
    assert abs(np.median(inner[..., 0]) - 2.0) < 0.1 and abs(np.median(inner[..., 1])) < 0.1


# ---- the port against the reference build on everything the GPU tests use it for ----------------
# What the reference build computed for the cases below is stored in tests/golden/reference/runs.npz
# (tests/golden/make_golden.py) as, per array, its shape, the SHA-256 of its float32 bits and a seeded
# sample of its values: the digest keeps the comparison bitwise over the whole array, the sample
# locates a difference.
REFERENCE_RUNS = os.path.join(os.path.dirname(__file__), "golden", "reference", "runs.npz")
SAMPLE = 512

BASELINE_CASES = {
    "cfg2_seed1": (436, 1024, 1, lambda: params.operating_point(2, 1024), 1, False),
    "cfg2_seed7": (436, 1024, 1, lambda: params.operating_point(2, 1024), 7, False),
    "cfg3_1920x1080_rgb_l1": (1080, 1920, 3, lambda: params.from_cli_numbers(
        "6 2 16 16 0.05 0.95 0 12 0.75 0 1 1 1 10 10 5 1 3 1.6 0".split(), noc=3), 2, False),
    "cfg5_2880x1988_stereo_op4": (1988, 2880, 1, lambda: params.operating_point(4, 2880, noc=1, nop=1), 4, True),
}
REFERENCE_CASES = ["cfg1", "thread_pool"] + ["random%d" % s for s in range(40)] + list(BASELINE_CASES)


def reference_case(name):
    """(name, prm, uint8 pairs, pyramids) of a case compared with the reference build."""
    if name == "cfg1":
        prm = params.operating_point(2, 640)
        pairs = [synth.synthetic_pair(480, 640, 1, seed=3)[:2]]
    elif name == "thread_pool":
        prm = params.from_cli_numbers("3 1 8 8 0.05 0.95 0 8 0.4 0 1 0 1 10 10 5 1 3 1.6 0".split())
        pairs = [synth.synthetic_pair(121, 203, 1, seed=30 + s)[:2] for s in range(3)]  # odd size: padding + crop
    elif name.startswith("random"):
        # the 40 seeded parameter sets of tests/test_gpu_parity.py::test_random_configurations_vs_oracle
        from test_gpu_parity import _random_config

        seed = int(name[len("random"):])
        numbers, ch, nop, size, amp = _random_config(np.random.default_rng(1000 + seed))
        prm = params.from_cli_numbers(numbers, noc=ch, nop=nop)
        pairs = [synth.synthetic_pair(size[0], size[1], ch, seed=200 + seed, stereo=(nop == 1), amp=amp)[:2]]
    else:
        h, w, ch, mk, seed, stereo = BASELINE_CASES[name]
        prm = mk()
        pairs = [synth.synthetic_pair(h, w, ch, seed=seed, stereo=stereo, amp=6.0)[:2]]
    return name, prm, pairs, [preprocess.PairPyramids(a, b, prm.sc_f, prm.p_samp_s) for a, b in pairs]


def _cfg1_flow(pyr, prm):
    h, w = pyr.level_shape(prm.sc_l)
    return (np.random.default_rng(0).standard_normal((h, w, 2)) * 0.7).astype(np.float32)


def _frames(pairs):
    return np.stack([np.stack([a, b]) for a, b in pairs])[..., None]


def reference_outputs(case):
    """The reference build's arrays for `case` (needs oracle/_ref)."""
    name, prm, pairs, pyrs = case
    if name == "cfg1":
        return {"flow": ref_driver.ref_run(pyrs[0], prm),
                "varref": ref_driver.ref_level_varref(pyrs[0], prm, prm.sc_l, _cfg1_flow(pyrs[0], prm))}
    if name == "thread_pool":
        # ofdis_ref_run_many / ofdis_ref_run_many_u8, the native thread-pool drivers of the CPU baseline
        return {"flows": ref_driver.ref_run_many(pyrs, prm, nrep=2, threads=3)[1],
                "full": ref_driver.ref_run_many_u8(_frames(pairs), prm, nrep=1, threads=2)[1]}
    return {"flow": ref_driver.ref_run(pyrs[0], prm)}


def _sha256(data):
    return hashlib.sha256(np.ascontiguousarray(data).tobytes()).hexdigest()


def summarize(case, arrays):
    """What tests/golden/reference/runs.npz keeps of the reference's `arrays` for `case`."""
    name, _, pairs, _ = case
    out = {name + "/inputs.sha256": np.array(_sha256(_frames(pairs)))}
    for key, a in arrays.items():
        flat = bits(a).reshape(-1)
        idx = np.sort(np.random.default_rng(0).permutation(flat.size)[:SAMPLE]).astype(np.int32)
        out.update({"%s/%s.shape" % (name, key): np.array(a.shape), "%s/%s.sha256" % (name, key): np.array(_sha256(flat)),
                    "%s/%s.idx" % (name, key): idx, "%s/%s.val" % (name, key): flat[idx].view(np.float32)})
    return out


_RUNS = {}


def _runs():
    if not _RUNS:
        _RUNS.update(np.load(REFERENCE_RUNS))
    return _RUNS


def _assert_stored(name, arrays, who):
    z = _runs()
    assert sorted(arrays) == sorted(k[len(name) + 1:-6] for k in z if k.startswith(name + "/") and k.endswith(".shape"))
    for key, a in arrays.items():
        k = "%s/%s" % (name, key)
        assert a.shape == tuple(z[k + ".shape"]), (who, name, key, a.shape)
        flat = bits(a).reshape(-1)
        bad = flat[z[k + ".idx"]] != z[k + ".val"].view(np.uint32)
        assert not bad.any(), "%s, %s %s: %d of %d sampled values differ from the reference build's" % (
            who, name, key, int(bad.sum()), bad.size)
        assert _sha256(flat) == str(z[k + ".sha256"]), "%s, %s %s: differs from the reference build outside the sample" % (
            who, name, key)


def assert_reference(case, got):
    """`got` (name -> array) is bitwise what the reference build computed for `case` (the stored digests); where
    oracle/_ref is built, the reference build must reproduce them as well."""
    name, prm, pairs, _ = case
    assert _sha256(_frames(pairs)) == str(_runs()[name + "/inputs.sha256"]), "%s: not the inputs the golden data was made from" % name
    _assert_stored(name, got, "port")
    if ref_driver.ref_available(prm.flavour()):
        _assert_stored(name, reference_outputs(case), "reference build")


@pytest.mark.parametrize("seed", range(40))
def test_port_vs_reference_on_the_random_configurations_of_the_gpu_suite(seed, oracle_port):
    """The 40 seeded parameter sets of tests/test_gpu_parity.py::test_random_configurations_vs_oracle:
    the port (the GPU tests' checker) must equal the reference build on each of them."""
    case = reference_case("random%d" % seed)
    _, prm, _, (pyr,) = case
    assert_reference(case, {"flow": oracle_port.port_run(pyr, prm)})


@pytest.mark.parametrize("name", list(BASELINE_CASES))
def test_port_vs_reference_at_baseline_sizes(name, oracle_port):
    """BASELINE configs[1], [2] and [4] at full size (the inputs of the GPU suite's full-size tests)."""
    case = reference_case(name)
    _, prm, _, (pyr,) = case
    assert_reference(case, {"flow": oracle_port.port_run(pyr, prm)})


def test_native_thread_pool_drivers_reproduce_single_runs(oracle_port):
    """ofdis_ref_run_many / ofdis_ref_run_many_u8 (the CPU baseline's drivers): same flows as one
    run per pair, and the restated pyramid / upsampling equal of_dis_b200/preprocess.py
    (which tests/test_preprocess.py pins to cv2), bit for bit."""
    case = reference_case("thread_pool")
    _, prm, pairs, pyrs = case
    flows = np.stack([oracle_port.port_run(p, prm) for p in pyrs])
    full = np.stack([preprocess.postprocess(f, prm.sc_l, p.padw, p.padh, 203, 121).reshape(121, 203, prm.nop)
                     for f, p in zip(flows, pyrs)])
    assert_reference(case, {"flows": flows, "full": full})
    if ref_driver.ref_available(prm.flavour()):
        for q, p in enumerate(pyrs):
            assert np.array_equal(bits(ref_driver.ref_run(p, prm)), bits(flows[q]))
