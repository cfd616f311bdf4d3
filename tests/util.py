"""Shared helpers for the parity tests: run the CUDA product path, the CPU oracle (oracle/gs_oracle.c) and,
when its build travelled with the snapshot, the compiled reference (oracle/_ref) on the same seeded inputs and
return everything as numpy so tests compare stage by stage."""
import glob
import importlib.util
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from manigaussian_b200 import scenes  # noqa: E402


def rel_l2(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    d = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / d) if d > 0 else float(np.linalg.norm(a - b))


def have_cuda():
    import torch
    return torch.cuda.is_available()


# --------------------------------------------------------------------------- reference (oracle/_ref)
_REF = {}


def load_reference(F):
    """The unmodified reference rasterizer compiled with NUM_CHANNELS_language_feature == F (3 or 32), or None."""
    if F in _REF:
        return _REF[F]
    import torch  # noqa: F401  (the extension links against libtorch)
    name = f"dgr_ref_f{F}"
    path = os.path.join(ROOT, "oracle", "_ref", name, name + ".so")
    mod = None
    if os.path.exists(path):
        try:
            spec = importlib.util.spec_from_file_location(name, path)
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
        except Exception as ex:  # pragma: no cover
            print(f"[tests] could not load {path}: {ex}")
            mod = None
    _REF[F] = mod
    return mod


def load_reference_package(F):
    """The reference's OWN Python operator (diff_gaussian_rasterization/__init__.py, installed unmodified into
    oracle/_ref/python by oracle/build_ref.py) bound to the compiled reference of feature width F: its `from . import _C`
    resolves to that build.  Returns the package module (GaussianRasterizer, GaussianRasterizationSettings) or None."""
    mod = load_reference(F)
    init = os.path.join(ROOT, "oracle", "_ref", "python", "diff_gaussian_rasterization", "__init__.py")
    if mod is None or not os.path.exists(init):
        return None
    name = f"dgr_reference_pkg_f{F}"
    if name in sys.modules:
        return sys.modules[name]
    sys.modules[name + "._C"] = mod
    spec = importlib.util.spec_from_file_location(name, init, submodule_search_locations=[os.path.dirname(init)])
    pkg = importlib.util.module_from_spec(spec)
    sys.modules[name] = pkg
    spec.loader.exec_module(pkg)
    return pkg


# outputs of the unmodified reference rasterizer, run on a B200 by tests/golden/make_golden.py
REFERENCE_GOLDEN = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "g[0-9]*.npz")))


def load_reference_golden(path):
    """(inputs, forward dict, backward dict) of one stored reference run, in the layout of run_reference().  Entries of
    culled Gaussians in the per-Gaussian float state are zero (the reference leaves them uninitialised)."""
    z = np.load(path)
    kw = json.loads(bytes(z["recipe"]).decode())
    if "bg" in kw:
        kw["bg"] = tuple(kw["bg"])
    fw = {k[3:]: z[k] for k in z.files if k.startswith("fw_")}
    fw["num_rendered"] = int(fw["num_rendered"])
    bw = {k[3:]: z[k] for k in z.files if k.startswith("bw_")}
    return make_inputs(**kw), fw, bw


# --------------------------------------------------------------------------- recorded parity values
# Expected values of the reference comparisons at sizes whose outputs are far too large to store (tests/golden/
# make_parity_record.py): a SHA-256 digest of every array compared bit for bit, and of every tensor compared by relative
# L2 its exact norm plus a CountSketch, which is linear, so that ||sketch(a) - sketch(b)|| estimates ||a - b|| over the
# whole tensor (within about 25 % at 64 buckets, ample for a 1e-4 bar met at 1e-5; a single wrong entry is caught exactly).
PARITY_RECORD = os.path.join(ROOT, "tests", "golden", "parity_record.npz")
SKETCH_BUCKETS = 64
_RECORD = {}


def sketch(x, k=SKETCH_BUCKETS):
    x = np.asarray(x, np.float64).ravel()
    rng = np.random.default_rng(x.size)
    bucket = rng.integers(0, k, x.size, dtype=np.int32)
    sign = rng.integers(0, 2, x.size, dtype=np.int8) * 2 - 1
    return np.bincount(bucket, weights=x * sign, minlength=k)


def _sha(x):
    import hashlib
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(x).tobytes()).digest(), np.uint8)


def summarize(exact, close, values=None):
    """exact: arrays compared bit for bit; close: tensors compared by relative L2; values: scalars kept as they are."""
    s = {"sha_" + k: _sha(v) for k, v in exact.items()}
    for k, v in close.items():
        s["norm_" + k] = np.float64(np.linalg.norm(np.asarray(v, np.float64)))
        s["sketch_" + k] = sketch(v).astype(np.float32)
    s.update({"value_" + k: np.float64(v) for k, v in (values or {}).items()})
    return s


def parity_fields(fw, bw, F, depth=False):
    """What the reference comparisons look at (test_parity_gpu.check_vs_reference): (bit-exact arrays, rel-L2 tensors).
    n_contrib is bit-exact too: its mismatch bar (1e-5 of the pixels) admits no mismatch at these image sizes."""
    live = fw["radii"] > 0
    exact = {k: fw[k] for k in ("radii", "tiles_touched", "point_list_keys", "point_list", "ranges", "n_contrib")}
    exact.update({k: fw[k][live].view(np.uint32) for k in ("depths", "means2D", "conic_opacity")})
    exact["num_rendered"] = np.int64(fw["num_rendered"])
    close = {"out_color": fw["out_color"], "final_T": fw["final_T"]}
    if F:
        close["out_feature"] = fw["out_feature"]
    if depth:
        close["out_depth"] = fw["out_depth"]
    close.update({k: v for k, v in bw.items() if not (k == "dL_dfeature" and not F)})
    return exact, close


def load_record(name):
    if not _RECORD:
        z = np.load(PARITY_RECORD)
        for key in z.files:
            case, field = key.split("/", 1)
            _RECORD.setdefault(case, {})[field] = z[key]
    assert name in _RECORD, f"{name} is not in {PARITY_RECORD}"
    return _RECORD[name]


def compare_with_record(name, exact, close):
    """Asserts the digests of `exact` equal the recorded ones; returns the estimated relative L2 of every `close` tensor."""
    rec = load_record(name)
    assert sorted(exact) == sorted(k[4:] for k in rec if k.startswith("sha_")), name
    assert sorted(close) == sorted(k[5:] for k in rec if k.startswith("norm_")), name
    for k, v in exact.items():
        assert np.array_equal(_sha(v), rec["sha_" + k]), f"{name}: {k} differs from the recorded value"
    report = {}
    for k, v in close.items():
        d, n = float(np.linalg.norm(sketch(v) - rec["sketch_" + k])), float(rec["norm_" + k])
        report[k] = d / n if n > 0 else d
    return report


def _obtain(base_ptr, off, nbytes, align=128):
    a = (base_ptr + off + align - 1) & ~(align - 1)
    return a - base_ptr, a - base_ptr + nbytes


def parse_ref_geom(buf, P):
    """GeometryState layout of the reference up to (not including) its CUB scan space (rasterizer_impl.cu:155-171)."""
    import torch
    base, off, out = buf.data_ptr(), 0, {}
    for name, nbytes, dt in (("depths", 4 * P, torch.float32), ("clamped", 3 * P, torch.uint8),
                             ("internal_radii", 4 * P, torch.int32), ("means2D", 8 * P, torch.float32),
                             ("cov3D", 24 * P, torch.float32), ("conic_opacity", 16 * P, torch.float32),
                             ("rgb", 12 * P, torch.float32), ("tiles_touched", 4 * P, torch.int32)):
        s, off = _obtain(base, off, nbytes)
        out[name] = buf[s:off].view(dt)
    return out


def parse_ref_binning(buf, R):
    """BinningState layout of the reference up to its CUB sort space (rasterizer_impl.cu:182-195)."""
    import torch
    base, off, out = buf.data_ptr(), 0, {}
    for name, nbytes, dt in (("point_list", 4 * R, torch.int32), ("point_list_unsorted", 4 * R, torch.int32),
                             ("point_list_keys", 8 * R, torch.int64), ("point_list_keys_unsorted", 8 * R, torch.int64)):
        s, off = _obtain(base, off, nbytes)
        out[name] = buf[s:off].view(dt)
    return out


def parse_ref_image(buf, N):
    """ImageState layout of the reference (rasterizer_impl.cu:173-180); ranges over-allocated to N entries."""
    import torch
    base, off, out = buf.data_ptr(), 0, {}
    for name, nbytes, dt in (("final_T", 4 * N, torch.float32), ("n_contrib", 4 * N, torch.int32),
                             ("ranges", 8 * N, torch.int32)):
        s, off = _obtain(base, off, nbytes)
        out[name] = buf[s:off].view(dt)
    return out


# --------------------------------------------------------------------------- inputs
def make_inputs(P, W, H, F=0, seed=0, view=0, num_views=4, sh_degree=1, precomp_colors=False, precomp_cov=False,
                scale0=None, bg=(0.0, 0.0, 0.0), depth=False):
    cam = scenes.make_camera(W, H, view, num_views)
    g = scenes.make_gaussians(P, F=F, sh_degree=sh_degree, seed=seed, scale0=scale0, precomp_colors=precomp_colors)
    g["cov3D_precomp"] = None
    if precomp_cov:
        # world-space covariance from scale/rotation computed on the host in float64, upper triangle
        s, q = g["scales"].astype(np.float64), g["rotations"].astype(np.float64)
        r, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
        Rm = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                       2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                       2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], -1).reshape(-1, 3, 3)
        Sig = Rm @ (s[:, :, None] ** 2 * np.transpose(Rm, (0, 2, 1)))
        g["cov3D_precomp"] = np.stack([Sig[:, 0, 0], Sig[:, 0, 1], Sig[:, 0, 2], Sig[:, 1, 1], Sig[:, 1, 2], Sig[:, 2, 2]],
                                      -1).astype(np.float32)
        g["scales"], g["rotations"] = None, None
    ct = scenes.make_cotangents(W, H, F, seed=seed, depth=depth)
    return dict(cam=cam, g=g, ct=ct, bg=np.asarray(bg, np.float32), P=P, W=W, H=H, F=F)


def _t(x, dev="cuda"):
    import torch
    return torch.Tensor([]) if x is None else torch.from_numpy(np.ascontiguousarray(x)).to(dev)


# --------------------------------------------------------------------------- oracle
def run_oracle(inp, backward=True, scale_modifier=1.0):
    from oracle import gs_oracle as O
    cam, g, ct = inp["cam"], inp["g"], inp["ct"]
    kw = dict(scales=g["scales"], rotations=g["rotations"], cov3D_precomp=g["cov3D_precomp"], shs=g["shs"],
              sh_degree=g["sh_degree"], colors_precomp=g["colors_precomp"], feature=g["feature"], scale_modifier=scale_modifier)
    fw = O.forward(g["means3D"], g["opacities"], cam["viewmatrix"], cam["projmatrix"], cam["campos"], inp["W"], inp["H"],
                   cam["tanfovx"], cam["tanfovy"], inp["bg"], **kw)
    bw = None
    if backward:
        bw = O.backward(fw, ct["dL_dcolor"], ct["dL_dfeature"], g["means3D"], cam["viewmatrix"], cam["projmatrix"],
                        cam["campos"], cam["tanfovx"], cam["tanfovy"], inp["bg"], **kw)
    return fw, bw


# --------------------------------------------------------------------------- product path (CUDA)
def run_ours(inp, backward=True, debug=False, scale_modifier=1.0, prefiltered=False, depth=False):
    """depth=True renders the view-space depth plane too (fw['out_depth']) and feeds inp['ct']['dL_ddepth'] to the backward."""
    import torch
    from manigaussian_b200 import rasterizer as R
    cam, g, ct = inp["cam"], inp["g"], inp["ct"]
    P, W, H, F = inp["P"], inp["W"], inp["H"], inp["F"]
    include = F > 0
    feat = _t(g["feature"]) if include else torch.zeros((P, 3), device="cuda")
    args = (_t(inp["bg"]), _t(g["means3D"]), _t(g["colors_precomp"]), feat, _t(g["opacities"]), _t(g["scales"]),
            _t(g["rotations"]), scale_modifier, _t(g["cov3D_precomp"]), _t(cam["viewmatrix"]), _t(cam["projmatrix"]),
            cam["tanfovx"], cam["tanfovy"], H, W, _t(g["shs"]), g["sh_degree"], _t(cam["campos"]), prefiltered, debug, include)
    out = R.rasterize_gaussians_raw(*args, return_depth=depth)
    num_rendered, color, feature, radii, geomB, binB, imgB = out[:7]
    torch.cuda.synchronize()
    N, T = W * H, ((W + 15) // 16) * ((H + 15) // 16)

    def arr(which, name, state, a0, a1, dtype, count):
        addr = R.state_array(which, name, state, a0, a1)
        off = addr - state.data_ptr()
        nbytes = count * torch.empty((), dtype=dtype).element_size()
        return state[off:off + nbytes].view(dtype).cpu().numpy()

    fw = dict(P=P, W=W, H=H, F=F, M=0 if g["shs"] is None else g["shs"].shape[1], num_rendered=num_rendered,
              out_color=color.cpu().numpy(), out_feature=feature.cpu().numpy(), radii=radii.cpu().numpy())
    if depth:
        fw["out_depth"] = out[7].cpu().numpy()
    for name, dt, cnt in (("depths", torch.float32, P), ("means2D", torch.float32, 2 * P), ("cov3D", torch.float32, 6 * P),
                          ("conic_opacity", torch.float32, 4 * P), ("rgbd", torch.float32, 4 * P),
                          ("tiles_touched", torch.int32, P), ("point_offsets", torch.int32, P), ("clamped", torch.uint8, P),
                          ("extent", torch.float32, 2 * P)):
        fw[name] = arr("geometry", name, geomB, P, 0, dt, cnt)
    fw["means2D"] = fw["means2D"].reshape(P, 2)
    fw["cov3D"] = fw["cov3D"].reshape(P, 6)
    fw["conic_opacity"] = fw["conic_opacity"].reshape(P, 4)
    fw["rgb"] = np.ascontiguousarray(fw["rgbd"].reshape(P, 4)[:, :3])
    fw["tiles_touched"] = fw["tiles_touched"].astype(np.uint32)
    Rn = num_rendered
    fw["point_list"] = arr("binning", "point_list", binB, Rn, 0, torch.int32, Rn).astype(np.uint32)
    fw["tile_ids"] = arr("binning", "tile_ids", binB, Rn, 0, torch.int32, Rn).astype(np.uint32)
    fw["point_list_unsorted"] = arr("binning", "point_list_unsorted", binB, Rn, 0, torch.int32, Rn).astype(np.uint32)
    fw["depth_order"] = arr("geometry", "depth_order", geomB, P, 0, torch.int32, P).astype(np.uint32)
    # The library sorts (depth, id) then (tile) instead of one 64-bit key; the reference's key array is, by definition
    # (rasterizer_impl.cu:100-104), tile << 32 | depth bits of the instance's Gaussian -- rebuilt here for comparison.
    fw["point_list_keys"] = (fw["tile_ids"].astype(np.uint64) << np.uint64(32)) | \
        fw["depths"].view(np.uint32)[fw["point_list"]].astype(np.uint64)
    fw["final_T"] = arr("image", "final_T", imgB, W, H, torch.float32, N)
    fw["n_contrib"] = arr("image", "n_contrib", imgB, W, H, torch.int32, N).astype(np.uint32)
    fw["ranges"] = arr("image", "ranges", imgB, W, H, torch.int32, 2 * T).astype(np.uint32).reshape(T, 2)
    fw["tile_order"] = arr("image", "tile_order", imgB, W, H, torch.int32, T).astype(np.uint32)
    # expand the 3-bit clamp mask to the reference's bool[P,3] layout
    fw["clamped"] = ((fw["clamped"][:, None] >> np.arange(3)[None, :]) & 1).astype(np.uint8)
    bw = None
    if backward:
        grads = R.rasterize_gaussians_backward_raw(
            args[0], args[1], radii, args[2], feat, args[5], args[6], scale_modifier, args[8], args[9], args[10], cam["tanfovx"],
            cam["tanfovy"], _t(ct["dL_dcolor"]), _t(ct["dL_dfeature"]) if include else torch.zeros((1,), device="cuda"),
            args[15], g["sh_degree"], args[17], geomB, num_rendered, binB, imgB, debug, include,
            dL_dout_depth=_t(ct["dL_ddepth"]) if depth else None)
        torch.cuda.synchronize()
        names = ("dL_dmeans2D", "dL_dcolors", "dL_dfeature", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh",
                 "dL_dscales", "dL_drotations")
        bw = {n: t.cpu().numpy() for n, t in zip(names, grads)}
    return fw, bw


# --------------------------------------------------------------------------- compiled reference (CUDA)
def run_reference(inp, backward=True, scale_modifier=1.0, prefiltered=False, depth=False):
    """Runs oracle/_ref (the reference's own kernels).  Features are padded/truncated to the build's width.  The reference
    renders no depth: with depth=True view-space z rides in the spare feature channel F of the build (SURVEY.md finding 4),
    fw['out_depth'] is that channel's image and dL/dz is chained into dL_dmeans3D by hand (z = V[2,:3] . p + V[2,3])."""
    import torch
    P, W, H, F = inp["P"], inp["W"], inp["H"], inp["F"]
    Fb = 32 if F + (1 if depth else 0) > 3 else 3
    assert F + (1 if depth else 0) <= Fb
    mod = load_reference(Fb)
    if mod is None:
        return None, None
    cam, g, ct = inp["cam"], inp["g"], inp["ct"]
    include = F > 0 or depth
    feat = torch.zeros((P, Fb), device="cuda")
    if F > 0:
        feat[:, :F] = _t(g["feature"])
    vm = cam["viewmatrix"].reshape(-1)
    zrow = np.array([vm[2], vm[6], vm[10]], np.float32)
    if depth:
        feat[:, F] = _t(g["means3D"]) @ _t(zrow) + float(vm[14])
    args = (_t(inp["bg"]), _t(g["means3D"]), _t(g["colors_precomp"]), feat, _t(g["opacities"]), _t(g["scales"]),
            _t(g["rotations"]), scale_modifier, _t(g["cov3D_precomp"]), _t(cam["viewmatrix"]), _t(cam["projmatrix"]),
            cam["tanfovx"], cam["tanfovy"], H, W, _t(g["shs"]), g["sh_degree"], _t(cam["campos"]), prefiltered, False, include)
    num_rendered, color, feature, radii, geomB, binB, imgB = mod.rasterize_gaussians(*args)
    torch.cuda.synchronize()
    N, T = W * H, ((W + 15) // 16) * ((H + 15) // 16)
    gs, bs, ims = parse_ref_geom(geomB, P), parse_ref_binning(binB, num_rendered), parse_ref_image(imgB, N)
    fw = dict(P=P, W=W, H=H, F=F, num_rendered=num_rendered, out_color=color.cpu().numpy(), radii=radii.cpu().numpy(),
              out_feature=feature[:F].cpu().numpy() if include else feature.cpu().numpy())
    if depth:
        fw["out_depth"] = feature[F].cpu().numpy()
    fw["depths"] = gs["depths"].cpu().numpy()
    fw["means2D"] = gs["means2D"].cpu().numpy().reshape(P, 2)
    fw["cov3D"] = gs["cov3D"].cpu().numpy().reshape(P, 6)
    fw["conic_opacity"] = gs["conic_opacity"].cpu().numpy().reshape(P, 4)
    fw["rgb"] = gs["rgb"].cpu().numpy().reshape(P, 3)
    fw["clamped"] = gs["clamped"].cpu().numpy().reshape(P, 3)
    fw["tiles_touched"] = gs["tiles_touched"].cpu().numpy().astype(np.uint32)
    fw["point_list"] = bs["point_list"].cpu().numpy().astype(np.uint32)
    fw["point_list_keys"] = bs["point_list_keys"].cpu().numpy().astype(np.uint64)
    fw["final_T"] = ims["final_T"].cpu().numpy()
    fw["n_contrib"] = ims["n_contrib"].cpu().numpy().astype(np.uint32)
    fw["ranges"] = ims["ranges"].cpu().numpy().astype(np.uint32)[:2 * T].reshape(T, 2)
    bw = None
    if backward:
        dF = torch.zeros((Fb, H, W), device="cuda")
        if F > 0:
            dF[:F] = _t(ct["dL_dfeature"])
        if depth:
            dF[F] = _t(ct["dL_ddepth"])
        grads = mod.rasterize_gaussians_backward(
            args[0], args[1], radii, args[2], feat, args[5], args[6], scale_modifier, args[8], args[9], args[10], cam["tanfovx"],
            cam["tanfovy"], _t(ct["dL_dcolor"]), dF if include else torch.zeros((1,), device="cuda"), args[15],
            g["sh_degree"], args[17], geomB, num_rendered, binB, imgB, False, include)
        torch.cuda.synchronize()
        names = ("dL_dmeans2D", "dL_dcolors", "dL_dfeature", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh",
                 "dL_dscales", "dL_drotations")
        bw = {n: t.cpu().numpy() for n, t in zip(names, grads)}
        if depth:
            bw["dL_dmeans3D"] = bw["dL_dmeans3D"] + bw["dL_dfeature"][:, F:F + 1] * zrow[None, :]
        if include:
            bw["dL_dfeature"] = bw["dL_dfeature"][:, :F]
    return fw, bw
