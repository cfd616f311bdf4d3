"""CPU tests of the oracle (oracle/gs_oracle.c): internal consistency, a finite-difference check of its backward
against its own forward (independent of any GPU), and the golden vectors produced by the compiled reference."""
import os

import numpy as np
import pytest

import util
from oracle import gs_oracle as O


def _run(inp, backward=True):
    return util.run_oracle(inp, backward)


def test_binning_invariants():
    inp = util.make_inputs(P=20000, W=200, H=120, F=0, seed=1)
    fw, _ = _run(inp, backward=False)
    keys, vals, R = fw["point_list_keys"], fw["point_list"], fw["num_rendered"]
    assert R == int(fw["tiles_touched"].sum()) > 0
    assert np.all(keys[1:] >= keys[:-1])
    same = keys[1:] == keys[:-1]
    assert np.all(vals[1:][same] > vals[:-1][same])  # stable: ties keep ascending Gaussian id
    tiles = (keys >> np.uint64(32)).astype(np.int64)
    T = fw["ranges"].shape[0]
    assert tiles.max() < T
    cnt = np.bincount(tiles, minlength=T)
    rg = fw["ranges"].astype(np.int64)
    assert np.array_equal(rg[:, 1] - rg[:, 0], cnt)
    assert np.array_equal(keys.astype(np.uint32), fw["depths"][vals].view(np.uint32))
    dead = fw["radii"] == 0
    assert np.all(fw["tiles_touched"][dead] == 0)


def test_get_higher_msb_matches_bit_length():
    for n in list(range(1, 70)) + [255, 256, 257, 1023, 1024, 4096, 65535, 65536]:
        assert O.get_higher_msb(n) == int(n).bit_length(), n


def test_empty_and_degenerate_inputs():
    inp = util.make_inputs(P=50, W=33, H=17, F=3, seed=2)
    inp["g"]["means3D"][:] = np.array([10.0, 0.0, 1.1], np.float32)  # all behind the camera
    fw, bw = _run(inp)
    assert fw["num_rendered"] == 0 and np.all(fw["radii"] == 0)
    assert np.allclose(fw["out_color"], inp["bg"][:, None, None]) and np.all(fw["final_T"] == 1)
    assert all(not np.any(v) for v in bw.values())
    inp2 = util.make_inputs(P=50, W=33, H=17, F=3, seed=2)
    inp2["g"]["opacities"][:] = 0.001  # below 1/255 everywhere: nothing may blend, gradients vanish
    fw2, bw2 = _run(inp2)
    assert fw2["num_rendered"] > 0 and np.all(fw2["n_contrib"] == 0) and not np.any(bw2["dL_dmeans3D"])


def _loss(inp):
    fw, _ = _run(inp, backward=False)
    l = float((fw["out_color"].astype(np.float64) * inp["ct"]["dL_dcolor"]).sum())
    if inp["F"]:
        l += float((fw["out_feature"].astype(np.float64) * inp["ct"]["dL_dfeature"]).sum())
    return l


@pytest.mark.parametrize("field,gname", [("means3D", "dL_dmeans3D"), ("scales", "dL_dscales"), ("rotations", "dL_drotations"),
                                         ("opacities", "dL_dopacity"), ("shs", "dL_dsh"), ("feature", "dL_dfeature")])
def test_backward_matches_finite_differences(field, gname):
    """Few large, faint splats (no alpha clamp, no early termination, nothing near the frustum clamp), so the
    reference's gradient conventions coincide with the true derivative and central differences apply."""
    inp = util.make_inputs(P=12, W=32, H=32, F=4, seed=5, scale0=0.06, sh_degree=2)
    inp["g"]["opacities"][:] = 0.35
    inp["g"]["scales"] = np.clip(inp["g"]["scales"], 0.04, 0.09).astype(np.float32)
    # smooth cotangents keep fp32 finite differences meaningful
    yy, xx = np.mgrid[0:32, 0:32].astype(np.float32) / 32
    inp["ct"]["dL_dcolor"] = np.stack([xx, yy, 1 - xx]).astype(np.float32)
    inp["ct"]["dL_dfeature"] = np.stack([yy, xx * yy, 1 - yy, xx]).astype(np.float32)
    _, bw = _run(inp)
    g = bw[gname].reshape(inp["g"][field].shape).astype(np.float64)
    rng = np.random.default_rng(0)
    num, ana = [], []
    base = inp["g"][field]
    for _ in range(12):
        idx = tuple(rng.integers(0, s) for s in base.shape)
        eps = 2e-3 * max(1.0, abs(float(base[idx])))
        if field == "scales":
            eps = 1e-3
        plus, minus = dict(inp), dict(inp)
        plus["g"], minus["g"] = dict(inp["g"]), dict(inp["g"])
        a, b = base.copy(), base.copy()
        a[idx] += eps
        b[idx] -= eps
        plus["g"][field], minus["g"][field] = a, b
        num.append((_loss(plus) - _loss(minus)) / (float(a[idx]) - float(b[idx])))
        ana.append(g[idx])
    num, ana = np.array(num), np.array(ana)
    # geometry moves the discontinuous alpha >= 1/255 footprint boundary, which central differences see and the
    # analytic gradient (by construction) does not: a few percent; appearance parameters are smooth
    tol = 0.10 if field in ("means3D", "scales", "rotations") else 0.02
    assert np.linalg.norm(num - ana) <= tol * max(np.linalg.norm(ana), 1e-3), (field, num, ana)


@pytest.mark.skipif(not util.REFERENCE_GOLDEN, reason="tests/golden/*.npz not generated yet (tests/golden/make_golden.py on a B200)")
@pytest.mark.parametrize("path", util.REFERENCE_GOLDEN, ids=[os.path.basename(p)[:-4] for p in util.REFERENCE_GOLDEN])
def test_oracle_against_reference_golden(path):
    """The restatement vs outputs of the unmodified reference run on a B200 (oracle/_ref)."""
    inp, ref, ref_bw = util.load_reference_golden(path)
    fw, bw = _run(inp)
    F = inp["F"]
    # integer / index outputs: bit-exact
    assert np.array_equal(fw["radii"], ref["radii"])
    assert np.array_equal(fw["tiles_touched"], ref["tiles_touched"])
    assert fw["num_rendered"] == ref["num_rendered"]
    assert np.array_equal(fw["point_list"], ref["point_list"])
    assert np.array_equal(fw["point_list_keys"] >> np.uint64(32), ref["point_list_keys"] >> np.uint64(32))  # tile ids
    assert np.array_equal(fw["ranges"], ref["ranges"])
    assert (fw["n_contrib"] != ref["n_contrib"]).mean() <= 1e-3
    live = ref["radii"] > 0
    # floating point: 1e-4 relative L2 (BASELINE.json north_star); depth key bits differ only by FMA contraction
    for k in ("depths", "means2D", "conic_opacity", "cov3D"):
        if k == "cov3D" and inp["g"]["cov3D_precomp"] is not None:
            continue
        assert util.rel_l2(fw[k][live], ref[k][live]) < 1e-5, k
    if inp["g"]["colors_precomp"] is None:
        assert util.rel_l2(fw["rgb"][live], ref["rgb"][live]) < 1e-5
        assert np.array_equal(fw["clamped"][live], ref["clamped"][live])
    assert util.rel_l2(fw["out_color"], ref["out_color"]) < 1e-4
    if F:
        assert util.rel_l2(fw["out_feature"], ref["out_feature"]) < 1e-4
    assert util.rel_l2(fw["final_T"], ref["final_T"]) < 1e-4
    for k, v in bw.items():
        if k == "dL_dconic" or (k == "dL_dfeature" and not F):
            continue
        assert util.rel_l2(v, ref_bw[k]) < 1e-4, (k, util.rel_l2(v, ref_bw[k]))
