#!/usr/bin/env python
"""bench.py -- Gaussians/s fwd+bwd of the rasterizer hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|cpu] [--workload c1|c2|c3|c4|c5|mg]
                    [--dump-outputs DIR]

A "step" = forward + backward of every view of the workload over one synthetic Gaussian cloud (SURVEY.md 8(d)):
default workload c3 = BASELINE.json configs[2]: 500k Gaussians, 4 views 256x256, RGB + 32 feature channels.
One JSON line is printed by rank 0.  Keys are described in DESIGN.md ("Measurement").

  value      whole-job Gaussians/s (P * views / s), inputs resident in HBM, through the C ABI (raw calls)
  e2e        same metric through the public autograd API (ours: gaussian_renderer.render_views) with the step's inputs
             copied pinned-host -> device every step (one packed copy) and the loss read back D2H every step
  roofline   dominant kernel (backward blend; on c4 the HBM-bound pre-op kernels): algorithmic bytes / CUDA-event time
             vs the measured HBM peak
  cpu_baseline  the CPU oracle (oracle/gs_oracle.c, OpenMP) timed on a bounded sample of the same workload

--impl reference times the UNMODIFIED reference rasterizer compiled for sm_100 (oracle/_ref, built by
oracle/build_ref.py) with the identical harness; the reference has no CPU implementation of this path, so the
CPU leg of both arms is the oracle port.  Under torchrun (N > 1) views are sharded across ranks (weak scaling:
`views` per GPU) and the packed per-Gaussian gradient buffer is summed with one NCCL all-reduce per step.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "c1": dict(P=50_000, views=1, W=128, H=128, F=0, depth=False, desc="50k Gaussians, 1 view 128x128, RGB-only"),
    "c2": dict(P=200_000, views=1, W=256, H=256, F=0, depth=True, desc="200k Gaussians, 1 view 256x256, RGB+depth"),
    "c3": dict(P=500_000, views=4, W=256, H=256, F=32, depth=False, desc="500k Gaussians, 4 views 256x256, RGB+32 feat"),
    "c4": dict(P=500_000, views=4, W=256, H=256, F=32, depth=False, dyna=True,
               desc="500k Gaussians + deformation offsets (dyna path): 4 views current frame + 4 views next frame, 256x256, RGB+32 feat"),
    "c5": dict(P=1_000_000, views=1, W=256, H=256, F=32, depth=False, desc="1M Gaussians, 1 view/GPU 256x256, RGB+32 feat"),
    "mg": dict(P=16_384, views=1, W=128, H=128, F=3, depth=False, desc="ManiGaussian's real call: 16384 Gaussians, 128x128, F=3"),
}
SH_DEGREE = 1


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------ --dump-outputs
DUMP_MAX_BYTES = 64_000_000
DUMP_SAMPLE = 65_536  # per-Gaussian rows written for larger clouds


def dump_outputs(path, P, arrays, per_gaussian):
    """Writes every array as <path>/<name>.npy, float64 kept and everything else as float32, so that the outputs of two
    builds of the project can be compared one for one.  `per_gaussian` arrays have the Gaussian index on axis 0; for clouds
    of more than DUMP_SAMPLE Gaussians only a fixed, seeded sample of those rows is written, their indices as
    gaussian_index.npy.  Fails rather than write more than DUMP_MAX_BYTES in all."""
    def host(x):
        x = x.detach().cpu().numpy() if hasattr(x, "detach") else np.asarray(x)
        return x if x.dtype == np.float64 else x.astype(np.float32)
    out = {k: host(v) for k, v in arrays.items()}
    idx = slice(None)
    if P > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(P, DUMP_SAMPLE, replace=False))
        out["gaussian_index"] = idx.astype(np.float64)
    for k, v in per_gaussian.items():
        v = host(v)
        assert v.shape[0] == P, (k, v.shape)
        out[k] = np.ascontiguousarray(v[idx])
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the limit of {DUMP_MAX_BYTES}")
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v)
    log(f"[bench] wrote {len(out)} arrays, {total} bytes, to {path}")


def view_outputs(impl, outs):
    """outs: (R, colour, feature, radii[, depth]) of every view.  Returns them as the caller receives them, stacked over
    views: colour [V,3,H,W], feature [V,F,H,W], depth [V,H,W], and radii as [P,V] (per Gaussian)."""
    import torch
    st = lambda xs, dim=0: torch.stack(list(xs), dim)
    arrays = {"color": st(o[1] for o in outs)}
    if impl.name == "reference":  # the build's padded feature width, depth in channel F (RefImpl)
        feats = [o[2][:impl.F] for o in outs]
        depths = [o[2][impl.F] for o in outs]
    else:
        feats = [o[2] for o in outs]
        depths = [o[4] for o in outs] if impl.depth else []
    if impl.F:
        arrays["feature"] = st(feats)
    if impl.depth:
        arrays["depth"] = st(depths)
    return arrays, {"radii": st((o[3] for o in outs), 1)}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region.  Uses in-process NVML (initialised before
    warm-up: spawning nvidia-smi makes NVML initialise concurrently with the timed region, which stalls CUDA driver
    calls for tens of milliseconds); falls back to an `nvidia-smi -lms` child that is given time to start."""
    BITS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("sw_power_cap", 0x4))

    def __init__(self, index, period=0.1):
        self.index, self.period, self.rows, self.stop_flag, self.thread, self.h = index, period, [], False, None, None
        self.max_mhz = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = self.index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except Exception:
                    pass
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml

            def loop():
                while not self.stop_flag:
                    try:
                        mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                        try:
                            rs = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                        except Exception:
                            rs = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                        self.rows.append((time.perf_counter(), float(mhz), int(rs)))
                    except Exception:
                        pass
                    time.sleep(self.period)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
        except Exception:
            self.h = None

    def stop(self, t0=None, t1=None):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=1.0)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["NVML unavailable"], "samples": 0}
        rows = [r for r in self.rows if (t0 is None or r[0] >= t0) and (t1 is None or r[0] <= t1)] or self.rows[-1:]
        reasons = sorted({n for (_, _, rs) in rows for (n, b) in self.BITS if rs & b})
        return {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(rows), "source": "NVML, in-process, %.0f ms period" % (self.period * 1e3)}


# ------------------------------------------------------------------------------------------------ workload
def host_inputs(wl, rank, world):
    from manigaussian_b200 import scenes
    P, V, W, H, F = wl["P"], wl["views"], wl["W"], wl["H"], wl["F"]
    g = scenes.make_gaussians(P, F=F, sh_degree=SH_DEGREE, seed=1234)
    cams = [scenes.make_camera(W, H, rank * V + v, world * V) for v in range(V)]
    cts = [scenes.make_cotangents(W, H, F, seed=100 + rank * V + v, depth=wl["depth"]) for v in range(V)]
    return g, cams, cts


class Impl:
    """fwd(view tensors) -> handle ; bwd(handle, cotangents) -> 9-tuple of gradients (reference order)."""
    name = "ours"

    def __init__(self, F, depth):
        from manigaussian_b200 import rasterizer as R
        self.R, self.F, self.depth = R, F, depth

    def fwd(self, G, cam):
        out = self.R.rasterize_gaussians_raw(cam["bg"], G["means3D"], G["empty"], G["feature"], G["opacities"], G["scales"],
                                             G["rotations"], 1.0, G["empty"], cam["viewmatrix"], cam["projmatrix"], cam["tanfovx"],
                                             cam["tanfovy"], cam["H"], cam["W"], G["shs"], SH_DEGREE, cam["campos"], False, False,
                                             self.F > 0, return_depth=self.depth)
        return out

    def bwd(self, G, cam, out, ct):
        return self.R.rasterize_gaussians_backward_raw(
            cam["bg"], G["means3D"], out[3], G["empty"], G["feature"], G["scales"], G["rotations"], 1.0, G["empty"],
            cam["viewmatrix"], cam["projmatrix"], cam["tanfovx"], cam["tanfovy"], ct["dL_dcolor"], ct["dL_dfeature"], G["shs"],
            SH_DEGREE, cam["campos"], out[4], out[0], out[5], out[6], False, self.F > 0,
            dL_dout_depth=ct["dL_ddepth"] if self.depth else None)


class RefImpl(Impl):
    """The unmodified reference kernels (oracle/_ref).  The build's feature width is fixed (3 or 32): features are
    padded to it; depth (absent in the reference) rides in a spare feature channel as SURVEY.md 8(d) prescribes."""
    name = "reference"

    def __init__(self, F, depth):
        import torch
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import util
        self.torch = torch
        self.F, self.depth = F, depth
        need = F + (1 if depth else 0)
        self.Fb = 32 if need > 3 else 3
        self.mod = util.load_reference(self.Fb)
        if self.mod is None:
            raise RuntimeError("oracle/_ref is not built")

    def _feat(self, G, cam):
        key = ("featb", id(cam))
        if key not in G:
            t = self.torch.zeros((G["means3D"].shape[0], self.Fb), device="cuda")
            if self.F:
                t[:, :self.F] = G["feature"]
            if self.depth:
                vm = cam["viewmatrix"].reshape(-1)
                t[:, self.F] = G["means3D"] @ self.torch.stack([vm[2], vm[6], vm[10]]) + vm[14]
            G[key] = t
        return G[key]

    def fwd(self, G, cam):
        inc = (self.F > 0) or self.depth
        return self.mod.rasterize_gaussians(cam["bg"], G["means3D"], G["empty"], self._feat(G, cam), G["opacities"], G["scales"],
                                            G["rotations"], 1.0, G["empty"], cam["viewmatrix"], cam["projmatrix"], cam["tanfovx"],
                                            cam["tanfovy"], cam["H"], cam["W"], G["shs"], SH_DEGREE, cam["campos"], False, False, inc)

    def bwd(self, G, cam, out, ct):
        inc = (self.F > 0) or self.depth
        key = ("ctb", id(ct))
        if key not in G:
            t = self.torch.zeros((self.Fb, cam["H"], cam["W"]), device="cuda")
            if self.F:
                t[:self.F] = ct["dL_dfeature"]
            if self.depth:
                t[self.F] = ct["dL_ddepth"]
            G[key] = t
        return self.mod.rasterize_gaussians_backward(
            cam["bg"], G["means3D"], out[3], G["empty"], self._feat(G, cam), G["scales"], G["rotations"], 1.0, G["empty"],
            cam["viewmatrix"], cam["projmatrix"], cam["tanfovx"], cam["tanfovy"], ct["dL_dcolor"], G[key], G["shs"], SH_DEGREE,
            cam["campos"], out[4], out[0], out[5], out[6], False, inc)


def to_device(g, cams, cts, torch, pinned=False):
    def t(x):
        if x is None:
            return None
        x = torch.from_numpy(np.ascontiguousarray(x))
        return x.pin_memory() if pinned else x.cuda()
    G = {k: t(g[k]) for k in ("means3D", "scales", "rotations", "opacities", "shs", "feature")}
    G["empty"] = torch.Tensor([])
    C = []
    for c in cams:
        d = {k: t(c[k]) for k in ("viewmatrix", "projmatrix", "campos")}
        d.update(W=c["W"], H=c["H"], tanfovx=c["tanfovx"], tanfovy=c["tanfovy"], bg=t(np.zeros(3, np.float32)))
        C.append(d)
    T = [{k: t(v) for k, v in ct.items()} for ct in cts]
    return G, C, T


GRAD_ORDER = ("dL_dmeans2D", "dL_dcolors", "dL_dfeature", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh", "dL_dscales",
              "dL_drotations")
PACKED = ("dL_dmeans3D", "dL_dmeans2D", "dL_dscales", "dL_drotations", "dL_dopacity", "dL_dsh", "dL_dfeature")


def make_packed(P, F, M, torch, registered=False):
    """One flat fp32 buffer holding every per-Gaussian gradient the optimiser needs; the all-reduce message."""
    from manigaussian_b200.parallel import PackedGradients
    pk = PackedGradients(P, F, M, "cuda", registered=registered)
    _PACKS[pk.flat.data_ptr()] = pk
    return pk.flat, pk.views


_PACKS = {}


def run_step_views(G, C, T, flat, acc, dist, F, depth):
    """ours, multi-view entry points: ONE C call enqueues every view's forward on its own stream, one more every view's
    backward, neither synchronises with the host (manigaussian_b200.rasterizer.rasterize_views_raw); the backward sums the
    per-Gaussian gradients of all views in registers and writes them ONCE into the packed buffer -- the all-reduce message."""
    from manigaussian_b200 import rasterizer as R
    from manigaussian_b200 import GaussianRasterizationSettings as S
    if "settings" not in G:
        G["settings"] = [S(c["H"], c["W"], c["tanfovx"], c["tanfovy"], c["bg"], 1.0, c["viewmatrix"], c["projmatrix"], SH_DEGREE,
                           c["campos"], False, False, F > 0) for c in C]
    views = G["settings"]
    outs, sts = R.rasterize_views_raw(views, G["means3D"], G["empty"], G["feature"], G["opacities"], G["scales"], G["rotations"], 1.0,
                                      G["empty"], G["shs"], SH_DEGREE, F > 0, return_depth=depth)
    pk = _PACKS[flat.data_ptr()] if dist is not None else None
    R.rasterize_views_backward_raw(views, outs, sts, [t["dL_dcolor"] for t in T],
                                   [t["dL_dfeature"] for t in T] if F else None, G["means3D"], G["empty"], G["feature"],
                                   G["scales"], G["rotations"], 1.0, G["empty"], G["shs"], SH_DEGREE, F > 0,
                                   grads_depth=[t["dL_ddepth"] for t in T] if depth else None, accumulate_into=acc,
                                   after_blend=pk.all_reduce_begin if pk is not None else None)
    if pk is not None:
        pk.all_reduce_finish()  # the rest of the ONE packed message; the feature field left while the last kernel ran
    G["last_outs"] = outs  # instance counts are read after the timed region (no host synchronisation inside it)
    return 0


def run_step(impl, G, C, T, flat, acc, dist=None, streams=None):
    """One step: fwd+bwd of every local view, gradients summed into the packed buffer, one all-reduce.
    With `streams` (ours only: the C ABI takes the caller's stream) independent views are enqueued on different CUDA
    streams so their kernels overlap; the reference launches on the legacy default stream and cannot."""
    import torch
    if streams and impl.name == "ours":
        return run_step_views(G, C, T, flat, acc, dist, impl.F, impl.depth)
    flat.zero_()
    Rs = 0
    if not streams:
        images = []
        for cam, ct in zip(C, T):
            out = impl.fwd(G, cam)
            grads = impl.bwd(G, cam, out, ct)
            images.append(out[:4] + out[7:])
            Rs += int(out[0])
            gd = dict(zip(GRAD_ORDER, grads))
            for k, v in acc.items():
                v.add_(gd[k].reshape(v.shape))
    else:
        main = torch.cuda.current_stream()
        for s in streams:
            s.wait_stream(main)
        results = []
        for i, (cam, ct) in enumerate(zip(C, T)):
            with torch.cuda.stream(streams[i % len(streams)]):
                out = impl.fwd(G, cam)
                results.append((out, impl.bwd(G, cam, out, ct)))
        for s in streams:
            main.wait_stream(s)
        for out, grads in results:
            Rs += int(out[0])
            gd = dict(zip(GRAD_ORDER, grads))
            for k, v in acc.items():
                gd[k].record_stream(main)
                v.add_(gd[k].reshape(v.shape))
        images = [out[:4] + out[7:] for out, _ in results]
    G["last_images"] = images  # (R, colour, feature, radii[, depth]) of every view, for --dump-outputs
    if dist is not None:
        dist.all_reduce(flat)
    return Rs


# ------------------------------------------------------------------------------------------------ e2e (public API)
def make_render(impl_name, wl, torch):
    """render(st, **kw) -> (color, feature, radii[, depth]) through the autograd API of the chosen implementation."""
    P, F = wl["P"], wl["F"]
    if impl_name == "ours":
        from manigaussian_b200 import GaussianRasterizationSettings, GaussianRasterizer

        def render(st, **kw):
            return GaussianRasterizer(st, return_depth=wl["depth"])(**kw)
    else:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import util
        from manigaussian_b200 import GaussianRasterizationSettings
        need = F + (1 if wl["depth"] else 0)
        Fb = 32 if need > 3 else 3
        mod = util.load_reference(Fb)

        pkg = util.load_reference_package(Fb)  # the reference's OWN diff_gaussian_rasterization/__init__.py around its compiled _C
        if pkg is None:
            raise RuntimeError("oracle/_ref/python (the reference's Python operator) is missing: run oracle/build_ref.py")

        def render(st, means3D, means2D, opacities, shs, language_feature_precomp, scales, rotations):
            k = 0
            if F == Fb and not wl["depth"]:
                feat = language_feature_precomp  # the build's width: handed over as is
            else:
                feat = torch.zeros((P, Fb), device="cuda")
                if F:
                    feat = torch.cat([language_feature_precomp, feat[:, F:]], 1)
                    k = F
            if wl["depth"]:
                vm = st.viewmatrix.reshape(-1)
                z = means3D @ torch.stack([vm[2], vm[6], vm[10]]) + vm[14]
                feat = torch.cat([feat[:, :k], z[:, None], feat[:, k + 1:]], 1)
            rst = pkg.GaussianRasterizationSettings(*st)  # same 13 fields, in the reference's own NamedTuple
            color, lf, radii = pkg.GaussianRasterizer(raster_settings=rst)(
                means3D=means3D, means2D=means2D, shs=shs, colors_precomp=None, language_feature_precomp=feat, opacities=opacities,
                scales=scales, rotations=rotations, cov3D_precomp=None)
            if wl["depth"]:
                return color, lf[:F], radii, lf[F]
            return color, lf[:F], radii

    return render, GaussianRasterizationSettings


def make_e2e(impl_name, wl, torch, dist=None, heads=False):
    """heads=True: the step's loss is ManiGaussian's two rendering heads on every view (L2 on the colour image + cosine
    embedding loss on the feature image, agents/manigaussian_bc/loss.py:12-23 as neural_rendering.py:300-318 applies them),
    the uploaded image tensors serving as the ground truth; ours computes them in the blend epilogue (render_views(targets=)),
    the reference arm with the PyTorch ops of its own loss.py."""
    P, F = wl["P"], wl["F"]
    render, GaussianRasterizationSettings = make_render(impl_name, wl, torch)
    copy_stream = torch.cuda.Stream()
    V = wl["views"]
    view_streams = None  # ours: render_views owns its per-view streams; the reference launches on the legacy default stream

    pack_state = {}

    def build_pack(Gh, Ch, Th):
        """All tensors of one step (Gaussian parameters, camera matrices, cotangents) laid out in ONE pinned fp32 buffer,
        every field on a 128-byte boundary: the step's H2D transfer is a single copy, the device tensors are views."""
        fields = [("G", None, k, v) for k, v in Gh.items() if hasattr(v, "numel") and v.numel()]
        fields += [("C", i, k, v) for i, ch in enumerate(Ch) for k, v in ch.items() if hasattr(v, "numel")]
        fields += [("T", i, k, th[k]) for k in ("dL_dcolor", "dL_dfeature", "dL_ddepth") for i, th in enumerate(Th)
                   if th.get(k) is not None]
        offs, off = [], 0
        for _, _, _, v in fields:
            offs.append(off)
            off += (v.numel() + 31) // 32 * 32
        packed = torch.empty(off, dtype=torch.float32).pin_memory()
        for (_, _, _, v), o in zip(fields, offs):
            packed[o:o + v.numel()].copy_(v.reshape(-1))
        pack_state.update(fields=fields, offs=offs, packed=packed)

    def upload(Gh, Ch, Th):
        """H2D copy of ONE step's inputs (pinned host -> device) on a copy stream, so that step i+1's inputs travel while
        step i computes (what a prefetching data loader does).  Returns the device tensors and a completion event."""
        if not pack_state:
            build_pack(Gh, Ch, Th)
        with torch.cuda.stream(copy_stream):
            buf = pack_state["packed"].cuda(non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        G = {k: v for k, v in Gh.items() if not (hasattr(v, "numel") and v.numel())}
        C = [{k: v for k, v in ch.items() if not hasattr(v, "numel")} for ch in Ch]
        T = [{k: None for k in th} for th in Th]
        for (kind, i, k, v), o in zip(pack_state["fields"], pack_state["offs"]):
            t = buf[o:o + v.numel()].view(v.shape)
            if kind == "G":
                G[k] = t
            elif kind == "C":
                C[i][k] = t
            else:
                T[i][k] = t
        return G, C, T, ev, buf

    ring = [torch.zeros(1).pin_memory() for _ in range(2)]
    pending = []

    def read_back(loss):
        """D2H read of the step's loss, every step, into pinned memory.  The copy is asynchronous and the VALUE is consumed one
        step later (lagged logging, what a training loop that does not want to stall its launch queue does); the flush at
        the end of the timed loop waits for and reads the last one, so all K results are read inside the timed region."""
        buf = ring[len(state_log) % 2]
        buf.copy_(loss.detach().reshape(1), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        pending.append((buf, ev))
        out = None
        while len(pending) > 1:
            b, e = pending.pop(0)
            e.synchronize()
            out = float(b[0])
            state_log.append(out)
        return out

    def flush():
        while pending:
            b, e = pending.pop(0)
            e.synchronize()
            state_log.append(float(b[0]))
        return state_log[-1] if state_log else None

    state_log = []

    def compute(dev):
        """render + loss + backward of every view through the autograd module, then D2H of the loss."""
        G, C, T, ev, buf = dev
        main = torch.cuda.current_stream()
        main.wait_event(ev)
        buf.record_stream(main)  # allocated on the copy stream, consumed here (every input is a view of it)
        G = {k: (v.requires_grad_(True) if v is not None and v.numel() else v) for k, v in G.items()}
        if impl_name == "ours":
            # the public multi-view call: ONE autograd node for all views, gradients summed on the device
            from manigaussian_b200.gaussian_renderer import render_views
            views = [GaussianRasterizationSettings(cam["H"], cam["W"], cam["tanfovx"], cam["tanfovy"], cam["bg"], 1.0, cam["viewmatrix"],
                                                   cam["projmatrix"], SH_DEGREE, cam["campos"], False, False, F > 0) for cam in C]
            if heads:
                tg = {"rgb": torch.stack([ct["dL_dcolor"] for ct in T])}
                if F:
                    tg["embed"] = torch.stack([ct["dL_dfeature"] for ct in T])
                o = render_views(views, G["means3D"], G["rotations"], G["scales"], G["opacities"], features_color=G["shs"],
                                 features_language=G["feature"] if F else None, normalize_feature=False, targets=tg,
                                 sync_gradients=True if dist is not None else None)
                loss = o["loss_rgb"].sum() + (o["loss_embed"].sum() if F else 0.0)
                loss.backward()
                return read_back(loss)
            o = render_views(views, G["means3D"], G["rotations"], G["scales"], G["opacities"], features_color=G["shs"],
                             features_language=G["feature"] if F else None, return_depth=wl["depth"], normalize_feature=False,
                             sync_gradients=True if dist is not None else None)  # N > 1: the one all-reduce, inside the backward
            loss = (o["render"] * torch.stack([ct["dL_dcolor"] for ct in T])).sum()
            if F:
                loss = loss + (o["render_embed"] * torch.stack([ct["dL_dfeature"] for ct in T])).sum()
            if wl["depth"]:
                loss = loss + (o["depth"] * torch.stack([ct["dL_ddepth"] for ct in T])).sum()
            loss.backward()
            return read_back(loss)
        losses = []
        for cam, ct in zip(C, T):
            st = GaussianRasterizationSettings(cam["H"], cam["W"], cam["tanfovx"], cam["tanfovy"], cam["bg"], 1.0,
                                               cam["viewmatrix"], cam["projmatrix"], SH_DEGREE, cam["campos"], False, False, True)
            out = render(st, means3D=G["means3D"], means2D=torch.zeros_like(G["means3D"], requires_grad=True),
                         opacities=G["opacities"], shs=G["shs"], language_feature_precomp=G["feature"] if F else None,
                         scales=G["scales"], rotations=G["rotations"])
            if heads:
                # the reference's own heads (loss.py:12-13, 18-23); its cosine head works on [..., F] rows
                lv = ((out[0] - ct["dL_dcolor"]) ** 2).mean()
                if F:
                    pe, ge = out[1].permute(1, 2, 0), ct["dL_dfeature"].permute(1, 2, 0)
                    lv = lv + (1.0 - torch.nn.functional.cosine_similarity(pe, ge, dim=-1).mean())
                losses.append(lv)
                continue
            lv = (out[0] * ct["dL_dcolor"]).sum()
            if F:
                lv = lv + (out[1] * ct["dL_dfeature"]).sum()
            if wl["depth"]:
                lv = lv + (out[3] * ct["dL_ddepth"]).sum()
            losses.append(lv)
        loss = losses[0]
        for lv in losses[1:]:
            loss = loss + lv
        loss.backward()
        if dist is not None:  # N > 1: the reference has no packed buffer; its per-Gaussian gradients are summed field by field
            for v in G.values():
                if getattr(v, "grad", None) is not None:
                    dist.all_reduce(v.grad)
        return read_back(loss)

    def step(Gh, Ch, Th, state):
        """state carries the prefetched inputs of this step; the next step's upload is started before computing."""
        dev = state.get("dev") or upload(Gh, Ch, Th)
        state["dev"] = upload(Gh, Ch, Th)
        return compute(dev)

    def graph_step_factory(Gh, Ch, Th):
        """CUDA-graph variant (ours only): the whole step -- render_views forward, loss, backward -- is captured ONCE with
        torch.cuda.graph (possible because nothing in it synchronises with the host or allocates outside torch's allocator;
        the reference's forward blocks on a device->host copy of its instance count and cannot be captured) and replayed per
        step.  Per step: one H2D copy of the packed inputs into the graph's static input buffer, one graph launch, one
        asynchronous D2H copy of the loss."""
        if not pack_state:
            build_pack(Gh, Ch, Th)
        from manigaussian_b200.gaussian_renderer import render_views
        static = torch.empty_like(pack_state["packed"], device="cuda")
        static.copy_(pack_state["packed"], non_blocking=True)
        G = {k: v for k, v in Gh.items() if not (hasattr(v, "numel") and v.numel())}
        C = [{k: v for k, v in ch.items() if not hasattr(v, "numel")} for ch in Ch]
        T = [{k: None for k in th} for th in Th]
        for (kind, i, k, v), o in zip(pack_state["fields"], pack_state["offs"]):
            t = static[o:o + v.numel()].view(v.shape)
            if kind == "G":
                G[k] = t.requires_grad_(True)
            elif kind == "C":
                C[i][k] = t
            else:
                T[i][k] = t
        views = [GaussianRasterizationSettings(cam["H"], cam["W"], cam["tanfovx"], cam["tanfovy"], cam["bg"], 1.0, cam["viewmatrix"],
                                               cam["projmatrix"], SH_DEGREE, cam["campos"], False, False, F > 0) for cam in C]
        cc = torch.stack([ct["dL_dcolor"] for ct in T])
        cf = torch.stack([ct["dL_dfeature"] for ct in T]) if F else None
        cd = torch.stack([ct["dL_ddepth"] for ct in T]) if wl["depth"] else None

        def fwd_bwd():
            if heads:
                o = render_views(views, G["means3D"], G["rotations"], G["scales"], G["opacities"], features_color=G["shs"],
                                 features_language=G["feature"] if F else None, normalize_feature=False,
                                 targets={"rgb": cc, "embed": cf} if F else {"rgb": cc})
                loss = o["loss_rgb"].sum() + (o["loss_embed"].sum() if F else 0.0)
                loss.backward()
                return loss
            o = render_views(views, G["means3D"], G["rotations"], G["scales"], G["opacities"], features_color=G["shs"],
                             features_language=G["feature"] if F else None, return_depth=wl["depth"], normalize_feature=False)
            loss = (o["render"] * cc).sum()
            if F:
                loss = loss + (o["render_embed"] * cf).sum()
            if wl["depth"]:
                loss = loss + (o["depth"] * cd).sum()
            loss.backward()
            return loss

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):  # eager warm-up: learns the binning capacities, fills the allocator
                for v in G.values():
                    if getattr(v, "grad", None) is not None:
                        v.grad = None
                fwd_bwd()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for v in G.values():
            if getattr(v, "grad", None) is not None:
                v.grad = None
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_loss = fwd_bwd()

        def gstep(Gh_, Ch_, Th_, state):
            static.copy_(pack_state["packed"], non_blocking=True)  # this step's inputs, pinned host -> the graph's input buffer
            graph.replay()
            return read_back(static_loss)
        gstep.flush = flush
        gstep.grads = lambda: {k: v.grad for k, v in G.items() if getattr(v, "grad", None) is not None}
        return gstep

    step.flush = flush
    step.graph_step_factory = graph_step_factory
    return step


# ------------------------------------------------------------------------------------------------ dyna path (c4)
def dyna_host_inputs(g, seed=4321):
    """Raw network outputs whose activations reproduce the synthetic cloud (SURVEY.md 8(d), c4): xyz + xyz_maps, log-scales,
    opacity logits, un-normalised quaternions/features, and the deformation field's offsets for the next frame."""
    rng = np.random.default_rng(seed)
    P = g["means3D"].shape[0]
    f32 = lambda x: np.ascontiguousarray(x, np.float32)
    xyz_maps = rng.normal(0, 0.01, (P, 3))
    return dict(xyz=f32(g["means3D"] - xyz_maps), xyz_maps=f32(xyz_maps), rot_maps=f32(g["rotations"] * rng.uniform(0.5, 2.0, (P, 1))),
                scale_maps=f32(np.log(g["scales"])), opacity_maps=f32(np.log(g["opacities"] / (1 - g["opacities"]))), sh=f32(g["shs"]),
                feature_maps=f32(g["feature"] * rng.uniform(0.5, 2.0, (P, 1))), next_xyz=f32(rng.normal(0, 0.01, (P, 3))),
                next_rot=f32(rng.normal(0, 0.05, (P, 4))), next_scale=f32(rng.normal(0, 0.1, (P, 3)) * g["scales"]))


def make_dyna_step(impl_name, wl, torch):
    """step(raw, C, T2) -> loss tensor: activations -> V current-frame views + V next-frame views -> backward to every raw
    map and offset (models_embed.py:245-252, 297-304; neural_rendering.py:383-402 for both frames)."""
    F, V = wl["F"], wl["views"]
    if impl_name == "ours":
        from manigaussian_b200 import GaussianRasterizationSettings
        from manigaussian_b200.gaussian_params import activate_gaussians
        from manigaussian_b200.gaussian_renderer import render_views

        def step(raw, C, T2):
            L = {k: (v.detach().requires_grad_(True) if k != "xyz" else v) for k, v in raw.items()}
            views = [GaussianRasterizationSettings(c["H"], c["W"], c["tanfovx"], c["tanfovy"], c["bg"], 1.0, c["viewmatrix"],
                                                   c["projmatrix"], SH_DEGREE, c["campos"], False, False, True) for c in C]
            cur = activate_gaussians(L["xyz"], L["rot_maps"], L["scale_maps"], L["opacity_maps"], L["feature_maps"], d_means=L["xyz_maps"])
            nxt = activate_gaussians(cur[0].detach(), cur[1].detach(), cur[2].detach(), cur[3].detach(), None, d_means=L["next_xyz"],
                                     d_rotations=L["next_rot"], d_scales=L["next_scale"], scale_activation=None, opacity_activation=None)
            oc = render_views(views, cur[0], cur[1], cur[2], cur[3], features_color=L["sh"], features_language=cur[4], normalize_feature=False)
            on = render_views(views, nxt[0], nxt[1], nxt[2], nxt[3], features_color=L["sh"].detach(),
                              features_language=cur[4].detach(), normalize_feature=False)
            loss = (oc["render"] * T2["color"][0]).sum() + (oc["render_embed"] * T2["feature"][0]).sum() + \
                   (on["render"] * T2["color"][1]).sum() + (on["render_embed"] * T2["feature"][1]).sum()
            loss.backward()
            return loss, L
    else:
        render, GaussianRasterizationSettings = make_render(impl_name, wl, torch)

        def step(raw, C, T2):
            L = {k: (v.detach().requires_grad_(True) if k != "xyz" else v) for k, v in raw.items()}
            scales = torch.clamp_max(torch.exp(L["scale_maps"]), 0.05)
            means = L["xyz"] + L["xyz_maps"]
            rots = torch.nn.functional.normalize(L["rot_maps"], dim=-1)
            opac = torch.sigmoid(L["opacity_maps"])
            n_means = means.detach() + L["next_xyz"]
            n_rots = torch.nn.functional.normalize(rots.detach() + L["next_rot"], dim=-1)
            n_scales = scales.detach() + L["next_scale"]
            loss = 0
            for v, c in enumerate(C):
                st = GaussianRasterizationSettings(c["H"], c["W"], c["tanfovx"], c["tanfovy"], c["bg"], 1.0, c["viewmatrix"],
                                                   c["projmatrix"], SH_DEGREE, c["campos"], False, False, True)
                for fr, (m, r, s_, o, sh, f) in enumerate(((means, rots, scales, opac, L["sh"], L["feature_maps"]),
                                                            (n_means, n_rots, n_scales, opac.detach(), L["sh"].detach(),
                                                             L["feature_maps"].detach()))):
                    fn = f / (f.norm(dim=-1, keepdim=True) + 1e-12)   # the reference normalises inside every render()
                    out = render(st, means3D=m, means2D=torch.zeros_like(m, requires_grad=True), opacities=o, shs=sh,
                                 language_feature_precomp=fn, scales=s_, rotations=r)
                    loss = loss + (out[0] * T2["color"][fr][v]).sum() + (out[1] * T2["feature"][fr][v]).sum()
            loss.backward()
            return loss, L
    return step


def main_dyna(a, wl, base, cfg, torch, rank, world):
    """c4: device-timed value and host-buffer e2e of the dyna step, same JSON contract."""
    P, V, W, H, F = wl["P"], wl["views"], wl["W"], wl["H"], wl["F"]
    g, cams, _ = host_inputs(wl, rank, world)
    raw_h = dyna_host_inputs(g)
    rng = np.random.default_rng(77)
    T2_h = {"color": rng.standard_normal((2, V, 3, H, W)).astype(np.float32), "feature": rng.standard_normal((2, V, F, H, W)).astype(np.float32)}
    pin = lambda x: torch.from_numpy(x).pin_memory()
    raw_p, T2_p = {k: pin(v) for k, v in raw_h.items()}, {k: pin(v) for k, v in T2_h.items()}
    _, C, _ = to_device(g, cams, [], torch)
    raw = {k: v.cuda() for k, v in raw_p.items()}
    T2 = {k: v.cuda() for k, v in T2_p.items()}
    step = make_dyna_step(a.impl, wl, torch)
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", 0)), period=0.025)
    if not a.no_clocks:
        sampler.start()
        time.sleep(0.3)
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < a.settle:
        step(raw, C, T2)
        torch.cuda.synchronize()
    for _ in range(a.warmup):
        step(raw, C, T2)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start = time.perf_counter()
    e0.record()
    for _ in range(a.steps):
        loss, L = step(raw, C, T2)
    e1.record()
    torch.cuda.synchronize()
    t_stop = time.perf_counter()
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, P, {"loss": loss}, {"grad_" + k: v.grad for k, v in L.items() if v.requires_grad})
    clocks = sampler.stop(t_start, t_stop)
    ms_step = e0.elapsed_time(e1) / a.steps
    units = P * 2 * V
    out = dict(base, value=units / (ms_step * 1e-3), ms_per_step=ms_step, clocks=clocks)
    cfg.update(gaussian_views_per_step=2 * V, l2="no flush: per-step working set exceeds the 126 MB L2")
    meas = dict(loss=float(loss.item()),
                grads_checked={k: bool(torch.isfinite(v.grad).all().item()) for k, v in L.items() if v.requires_grad})
    out["config"] = cfg
    out["measured"] = meas
    if not a.no_e2e:
        copy_stream = torch.cuda.Stream()

        def upload():
            with torch.cuda.stream(copy_stream):
                d = ({k: v.cuda(non_blocking=True) for k, v in raw_p.items()}, {k: v.cuda(non_blocking=True) for k, v in T2_p.items()})
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return d + (ev,)

        def e2e_step(state):
            dev = state.get("dev") or upload()
            state["dev"] = upload()
            r, t2, ev = dev
            torch.cuda.current_stream().wait_event(ev)
            for d in (r, t2):
                for v in d.values():
                    v.record_stream(torch.cuda.current_stream())
            return float(step(r, C, t2)[0].item())
        state = {}
        for _ in range(3):
            e2e_step(state)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            e2e_step(state)
        torch.cuda.synchronize()
        te = (time.perf_counter() - t0) / a.steps
        out["e2e"] = {"value": units / te, "unit": "Gaussians/s", "ms_per_step": te * 1e3, "d2h_bytes_per_step": 4,
                      "h2d_bytes_per_step": int(sum(v.numel() * 4 for v in raw_p.values()) + sum(v.numel() * 4 for v in T2_p.values()))}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    out["gpu_launches"] = (7 * 2 * V + 4) * a.steps if a.impl == "ours" else 0
    out["roofline"] = {"bound": "hbm", "kernel": "whole pipeline", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None,
                       "traffic": None, "note": "per-kernel roofline is reported by the c3 line (same rasterizer kernels)"}
    if a.impl == "ours" and not a.no_stage_timing:
        # the pre-op kernels are the HBM-bound part of this workload: time them alone (CUDA events inside the library)
        from manigaussian_b200 import _binding
        _binding.profile_read()
        _binding.profile_enable(True)
        for _ in range(3):
            step(raw, C, T2)
        torch.cuda.synchronize()
        st = _binding.profile_read()
        _binding.profile_enable(False)
        per = {k: v[0] / max(v[1], 1) for k, v in st.items()}
        meas["stage_ms_per_launch"] = {k: round(v, 4) for k, v in per.items()}
        # algorithmic bytes of the two launches per direction (current frame: all fields + F features; next frame: no features)
        small = 4 * (3 + 4 + 3 + 1)
        fwd_b = P * ((small + 12 + 4 * F) + (small + 4 * F)) + P * ((small + 12 + 16 + 12) + small)
        bwd_b = P * ((small + 12 + 4 * F) + (small + 4 * F) + (small + 12 + 4 * F)) + P * ((small + 40) + small + (small + 40))
        if per.get("activate_fwd", 0) > 0 and per.get("activate_bwd", 0) > 0:
            ach_f = fwd_b / 2 / (per["activate_fwd"] * 1e-3) / 1e9
            ach_b = bwd_b / 2 / (per["activate_bwd"] * 1e-3) / 1e9
            out["roofline"] = {"bound": "hbm", "kernel": "activate_bwd", "achieved": ach_b, "peak": peak, "unit": "GB/s",
                               "frac": ach_b / peak, "traffic": None, "ms_per_launch": per["activate_bwd"],
                               "alg_bytes_per_launch": bwd_b / 2,
                               "also": {"activate_fwd": {"achieved": ach_f, "frac": ach_f / peak, "ms_per_launch": per["activate_fwd"]}},
                               "note": "mean of the current-frame and next-frame launches; the blend kernels' roofline is on the c3 line"}
    if a.gpus == 1 and not a.no_cpu_baseline:
        cb, _ = cpu_baseline(wl)
        cb["sample"] += " [rasterizer of one frame; activations not included]"
        out["cpu_baseline"] = cb
    print(json.dumps(out))
    return 0


def nbytes(d):
    return sum(v.numel() * v.element_size() for v in d.values() if hasattr(v, "numel"))


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_baseline(wl, target_s=12.0):
    """Oracle port (oracle/gs_oracle.c, OpenMP, all host threads) on a bounded sample of the workload.  A probe on the
    first 100k Gaussians of view 0 sizes the sample: the full cloud, as many of the workload's views as fit in about
    `target_s` seconds of CPU work (at least one)."""
    from manigaussian_b200 import scenes
    from oracle import gs_oracle as O
    P, W, H, F, V = wl["P"], wl["W"], wl["H"], wl["F"], wl["views"]
    gfull = scenes.make_gaussians(P, F=F, sh_degree=SH_DEGREE, seed=1234)
    bg = np.zeros(3, np.float32)
    cores = O.max_threads()

    def run(n, view):
        g = {k: (v[:n] if isinstance(v, np.ndarray) else v) for k, v in gfull.items()}
        cam = scenes.make_camera(W, H, view, V)
        ct = scenes.make_cotangents(W, H, F, seed=100 + view)
        kw = dict(scales=g["scales"], rotations=g["rotations"], shs=g["shs"], sh_degree=SH_DEGREE, feature=g["feature"])
        t0 = time.perf_counter()
        fw = O.forward(g["means3D"], g["opacities"], cam["viewmatrix"], cam["projmatrix"], cam["campos"], W, H, cam["tanfovx"],
                       cam["tanfovy"], bg, **kw)
        O.backward(fw, ct["dL_dcolor"], ct["dL_dfeature"], g["means3D"], cam["viewmatrix"], cam["projmatrix"], cam["campos"],
                   cam["tanfovx"], cam["tanfovy"], bg, **kw)
        return time.perf_counter() - t0

    probe_n = min(P, 100_000)
    probe = min(run(probe_n, 0), run(probe_n, 0))
    est_view = probe * P / probe_n * 1.3  # deeper per-pixel lists at full density
    nviews = int(max(1, min(V, target_s // max(est_view, 1e-3))))
    total, reps = 0.0, 0
    while reps < 4 and total < 0.8 * target_s:
        total += sum(run(P, v) for v in range(nviews))
        reps += 1
    nviews *= reps
    return {"value": P * nviews / total, "unit": "Gaussians/s", "cores": cores, "kind": "port",
            "sample": f"all {P} Gaussians, {nviews} view renders (views of the workload, repeated {reps}x), {W}x{H}, F={F}, fwd+bwd, "
                      f"{total:.1f} s of CPU work "
                      f"(probe: {probe_n} Gaussians in {probe:.2f} s)"}, total


# ------------------------------------------------------------------------------------------------ c5: strong scaling
def strong_scaling_c5(torch, dist, rank, world, steps, warmup):
    """BASELINE.json configs[4] / north_star's multi-GPU split: 1M Gaussians (replicated), 8 views 256x256 with 32 feature
    channels sharded round-robin over the ranks (view v on rank v % world: one view per GPU at 8 GPUs), ONE all-reduce of the
    packed per-Gaussian gradient buffer per step.  Strong scaling: the 8 views are fixed, `value` = P * 8 / step time.
    Also checks the exchange: the all-reduced gradients must equal the sum over all 8 views rendered on rank 0 alone."""
    from manigaussian_b200 import scenes
    from manigaussian_b200.parallel import shard_views
    wl = dict(WORKLOADS["c5"])
    P, W, H, F, VT = wl["P"], wl["W"], wl["H"], wl["F"], 8
    M = (SH_DEGREE + 1) ** 2
    g = scenes.make_gaussians(P, F=F, sh_degree=SH_DEGREE, seed=1238)
    mine = shard_views(VT, rank, world)

    def dev_views(ids):
        cams = [scenes.make_camera(W, H, v, VT) for v in ids]
        cts = [scenes.make_cotangents(W, H, F, seed=200 + v) for v in ids]
        return to_device(g, cams, cts, torch)

    G, C, T = dev_views(mine)
    flat, acc = make_packed(P, F, M, torch, registered=world > 1)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(warmup, 3)):
        run_step_views(G, C, T, flat, acc, dist, F, False)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        run_step_views(G, C, T, flat, acc, dist, F, False)
    e1.record()
    barrier()
    tmax = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if dist is not None:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_step = float(tmax.item()) / steps
    Rs = [o.num_rendered() for o in G["last_outs"]]
    out = {"workload": "c5: 1M Gaussians, 8 views 256x256, RGB + 32 features, views sharded v % N, one all-reduce of packed grads",
           "scaling": "strong", "views_total": VT, "views_per_gpu": [len(shard_views(VT, r, world)) for r in range(world)],
           "value": P * VT / (ms_step * 1e-3), "unit": "Gaussians/s", "ms_per_step": ms_step, "steps": steps,
           "allreduce_bytes": int(flat.numel() * 4) if world > 1 else 0,
           "num_rendered_rank0": Rs}
    # gradient check of the exchange (rank 0 renders all views alone)
    if world > 1:
        run_step_views(G, C, T, flat, acc, dist, F, False)  # one more step: `flat` now holds the all-reduced sum
        torch.cuda.synchronize()
        if rank == 0:
            Ga, Ca, Ta = dev_views(list(range(VT)))
            flat1, acc1 = make_packed(P, F, M, torch)
            run_step_views(Ga, Ca, Ta, flat1, acc1, None, F, False)
            torch.cuda.synchronize()
            num = float((flat.double() - flat1.double()).norm())
            den = float(flat1.double().norm())
            out["grad_check_rel_l2"] = num / den if den > 0 else num
            out["grad_check"] = "all-reduced gradients of the sharded views vs all 8 views on rank 0 (bar 1e-5, SURVEY.md 8(e))"
        barrier()
    return out


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cpu"])
    ap.add_argument("--workload", default="c3", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-graph", action="store_true", help="also time the e2e step replayed from a CUDA graph (always done for small clouds)")
    ap.add_argument("--heads", action="store_true", help="e2e: the loss is ManiGaussian's L2-colour + cosine-embedding heads per view "
                    "(ours: fused into the blend kernels; reference: its PyTorch ops) instead of a fixed cotangent")
    ap.add_argument("--no-c5", action="store_true", help="skip the strong-scaling block (BASELINE configs[4]: 1M Gaussians, 8 views over the ranks)")
    ap.add_argument("--settle", type=float, default=1.5, help="seconds of untimed steps before the W warm-up steps "
                    "(lets clocks/power state and the caching allocator reach steady state)")
    ap.add_argument("--no-clocks", action="store_true", help="do not poll nvidia-smi during the run")
    ap.add_argument("--no-stage-timing", action="store_true", help="do not bracket stages with CUDA events")
    ap.add_argument("--streams", type=int, default=4, help="CUDA streams over which independent views are enqueued (ours only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed "
                    "(images, radii, per-Gaussian gradients; a seeded sample of rows for large clouds) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    wl = dict(WORKLOADS[a.workload])
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    base = {"metric": "Gaussians/s fwd+bwd", "unit": "Gaussians/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "impl": a.impl}
    cfg = {"workload": f"{a.workload}: {wl['desc']}", "P": wl["P"], "views_per_gpu": wl["views"], "image": [wl["W"], wl["H"]],
           "feature_channels": wl["F"], "depth": wl["depth"], "sh_degree": SH_DEGREE,
           "parallelism": f"view-parallel x{world}, 1 NCCL all-reduce of packed per-Gaussian grads per step" if world > 1 else "1 GPU"}

    if world > 1 and rank == 0 and "NCCL_DEBUG_FILE" not in os.environ:
        # record which algorithms/transports NCCL sets up (NVLS = in-switch reduction over NVSwitch) next to the numbers;
        # must be in the environment before the NCCL library initialises its logging
        os.environ["MGS_NCCL_LOG"] = f"/tmp/mgs_nccl_{os.getpid()}.log"
        os.environ.update(NCCL_DEBUG="INFO", NCCL_DEBUG_SUBSYS="INIT,ENV,TUNING,NVLS", NCCL_DEBUG_FILE=os.environ["MGS_NCCL_LOG"])
    # ---- CPU-only arm / reference arm without a reference build -------------------------------------------------
    import torch
    use_cpu = a.impl == "cpu"
    if a.impl == "reference":
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import util
        need = wl["F"] + (1 if wl["depth"] else 0)
        if not torch.cuda.is_available() or util.load_reference(32 if need > 3 else 3) is None:
            use_cpu = True
    if use_cpu:
        if a.dump_outputs:
            raise SystemExit("--dump-outputs needs a GPU arm: the CPU arm times a sample of views sized by its own speed")
        if rank != 0:
            return 0
        cb, best = cpu_baseline(wl)
        out = dict(base, value=cb["value"], ms_per_step=best * 1e3, config=cfg, cpu_baseline=cb,
                   e2e={"value": cb["value"], "unit": "Gaussians/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                   gpu_launches=0, note="CPU oracle port (the reference ships no CPU path and oracle/_ref is unavailable here)")
        print(json.dumps(out))
        return 0

    # ---- GPU arms ------------------------------------------------------------------------------------------------
    torch.cuda.set_device(local_rank)
    dist = None
    nccl_log = None
    if world > 1:
        import torch.distributed as dist_mod
        import datetime
        nccl_log = os.environ.get("MGS_NCCL_LOG")
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=120))
        dist = dist_mod
    if wl.get("dyna"):
        if world > 1:
            raise SystemExit("workload c4 is a single-GPU configuration (BASELINE.json configs[3])")
        return main_dyna(a, wl, base, cfg, torch, rank, world)
    P, V, W, H, F = wl["P"], wl["views"], wl["W"], wl["H"], wl["F"]
    M = (SH_DEGREE + 1) ** 2
    g, cams, cts = host_inputs(wl, rank, world)
    G, C, T = to_device(g, cams, cts, torch)
    impl = Impl(F, wl["depth"]) if a.impl == "ours" else RefImpl(F, wl["depth"])
    flat, acc = make_packed(P, F, M, torch, registered=(world > 1 and a.impl == "ours"))
    packed_bytes = int(flat.numel() * 4)
    pk0 = _PACKS.get(flat.data_ptr())

    streams = None
    if a.impl == "ours" and (a.streams > 1 or V == 1):
        # truthy = "use the multi-view entry points" (rasterize_views_raw owns the per-view streams; a single view runs on the
        # caller's stream): no host read-back of the instance count in the timed loop, also for one view
        streams = [torch.cuda.Stream() for _ in range(min(a.streams, V))] if V > 1 else [torch.cuda.current_stream()]
    cfg["view_streams"] = len(streams) if streams else 1
    meas = {}  # everything MEASURED goes here, `config` only names the workload
    if world > 1 and pk0 is not None:
        meas["packed_buffer_nccl_registered"] = bool(pk0.registered)
        if getattr(pk0, "registration_error", None):
            meas["packed_buffer_registration_error"] = pk0.registration_error[:200]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local_rank, period=0.025)
    if not a.no_clocks:
        sampler.start()
        time.sleep(0.3)
    if a.impl == "ours":
        from manigaussian_b200 import _binding
        _binding.profile_enable(False)
    t_settle, n_settle = time.perf_counter(), 0
    while time.perf_counter() - t_settle < a.settle:
        Rtot = run_step(impl, G, C, T, flat, acc, None, streams)  # no collective: ranks settle for a time, not a count
        torch.cuda.synchronize()
        n_settle += 1
    meas["settle_steps"] = n_settle
    for _ in range(a.warmup):
        Rtot = run_step(impl, G, C, T, flat, acc, dist, streams)
    if a.impl == "ours":
        _binding.profile_read()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start = time.perf_counter()
    e0.record()
    step_marks = []
    for _ in range(a.steps):
        Rtot = run_step(impl, G, C, T, flat, acc, dist, streams)
        step_marks.append(time.perf_counter())
    e1.record()
    barrier()
    t_stop = time.perf_counter()
    if a.dump_outputs and rank == 0:
        last = [o[:4] + o[7:] for o in G["last_outs"]] if streams and a.impl == "ours" else G["last_images"]
        arrays, per_gaussian = view_outputs(impl, last)
        per_gaussian.update(acc)  # the per-Gaussian gradients summed over the views (all-reduced over the ranks)
        dump_outputs(a.dump_outputs, P, arrays, per_gaussian)
    hs = sorted((b_ - a_) * 1e3 for a_, b_ in zip([t_start] + step_marks[:-1], step_marks))
    meas["host_step_ms"] = {"min": round(hs[0], 3), "median": round(hs[len(hs) // 2], 3), "max": round(hs[-1], 3)}
    if G.get("last_outs") is not None and streams and a.impl == "ours":
        Rtot = sum(o.num_rendered() for o in G["last_outs"])  # read after the timed region: no host sync inside it
        meas["binning_capacity_per_view"] = [int(o[0]) for o in G["last_outs"]]
        meas["binning_overflow"] = any(o.overflowed() for o in G["last_outs"])
    clocks = sampler.stop(t_start, t_stop)
    ms = e0.elapsed_time(e1)
    meas["wall_ms_per_step"] = (t_stop - t_start) * 1e3 / a.steps
    stages = None
    if a.impl == "ours" and not a.no_stage_timing:
        # per-stage CUDA-event durations for the roofline leg: a separate short pass with views enqueued one after the
        # other on ONE stream, so that each duration is that kernel alone (in the timed region above views overlap)
        _binding.profile_read()
        _binding.profile_enable(True)
        for _ in range(3):
            run_step(impl, G, C, T, flat, acc, None, None)
        torch.cuda.synchronize()
        stages = _binding.profile_read()
        if streams:
            # the timed region's backward runs ONE per-Gaussian kernel for all views after the join: time that launch too
            run_step(impl, G, C, T, flat, acc, None, streams)
            torch.cuda.synchronize()
            mv = _binding.profile_read()
            if mv.get("project_bwd", (0, 0))[1] > 0:
                meas["project_bwd_views_ms"] = round(mv["project_bwd"][0] / mv["project_bwd"][1], 4)
            # the same stages as they run in the timed region (views on their own streams, kernels of different views
            # sharing the GPU): the elapsed time of a launch then includes what it waited for its share of the SMs
            meas["stage_ms_per_launch_overlapped"] = {k: round(v[0] / max(v[1], 1), 4) for k, v in mv.items() if v[1] > 0}
        _binding.profile_enable(False)
    tmax = torch.tensor([ms], device="cuda")
    if dist is not None:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms = float(tmax.item())
    ms_step = ms / a.steps
    value = P * V * world / (ms_step * 1e-3)

    # ---- end-to-end leg through the public API, host buffers -----------------------------------------------------
    e2e = None
    if not a.no_e2e:
        Gh, Ch, Th = to_device(g, cams, cts, torch, pinned=True)
        step = make_e2e(a.impl, wl, torch, dist, heads=a.heads)
        e2e_state = {}
        for _ in range(max(3, a.warmup)):
            step(Gh, Ch, Th, e2e_state)
        step.flush()
        barrier()
        per_step = []
        t0 = time.perf_counter()
        for _ in range(a.steps):
            ts = time.perf_counter()
            step(Gh, Ch, Th, e2e_state)
            per_step.append(time.perf_counter() - ts)
        step.flush()
        barrier()
        te = torch.tensor([(time.perf_counter() - t0) / a.steps], device="cuda")
        per_step.sort()
        meas["e2e_host_ms_per_call"] = {"min": round(per_step[0] * 1e3, 3), "median": round(per_step[len(per_step) // 2] * 1e3, 3),
                                        "max": round(per_step[-1] * 1e3, 3)}
        if dist is not None:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": P * V * world / float(te.item()), "unit": "Gaussians/s",
               "h2d_bytes_per_step": int(nbytes(Gh) + sum(nbytes(c) for c in Ch) + sum(nbytes(t) for t in Th)),
               "d2h_bytes_per_step": 4, "ms_per_step": float(te.item()) * 1e3,
               "note": "wall clock around K steps; every step copies all its inputs pinned-host->device (prefetched one step ahead on a "
                       "copy stream), runs the public autograd API (ours: manigaussian_b200.gaussian_renderer.render_views, one node "
                       "for all views; reference: its autograd Function per view), and copies the loss to pinned host memory (async, value consumed one "
                       "step later, all K read before the clock stops)",
               "loss": "L2 colour + cosine embedding heads per view (ours: fused in the blend kernels; reference: PyTorch ops)" if a.heads
                       else "sum(image * fixed cotangent)"}

    if e2e is not None and a.impl == "ours" and world == 1 and (a.e2e_graph or P <= 100_000):
        try:
            gstep = step.graph_step_factory(Gh, Ch, Th)
            gs = {}
            for _ in range(max(3, a.warmup)):
                gstep(Gh, Ch, Th, gs)
            gstep.flush()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.steps):
                gstep(Gh, Ch, Th, gs)
            gstep.flush()
            torch.cuda.synchronize()
            tg = (time.perf_counter() - t0) / a.steps
            e2e["cuda_graph"] = {"value": P * V / tg, "unit": "Gaussians/s", "ms_per_step": tg * 1e3,
                                 "note": "same step, captured once with torch.cuda.graph and replayed: per step one H2D copy of the packed "
                                         "inputs into the graph's input buffer, one graph launch, one async D2H of the loss"}
        except Exception as ex:  # pragma: no cover
            e2e["cuda_graph"] = {"error": repr(ex)[:300]}

    c5 = None
    if a.impl == "ours" and a.workload == "c3" and not a.no_c5:
        # drop this workload's device tensors first: the c5 cloud is twice the size
        del G, C, T, flat, acc
        torch.cuda.empty_cache()
        c5 = strong_scaling_c5(torch, dist, rank, world, a.steps, a.warmup)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    from manigaussian_b200 import scenes
    R_view = Rtot / V
    N = W * H
    balg_view = scenes.alg_bytes_per_view(P, R_view, N, M, F, depth=wl["depth"])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    out = dict(base, value=value, ms_per_step=ms_step, config=cfg, measured=meas, clocks=clocks)
    cfg["l2"] = "no flush: per-step working set (inputs + state + gradients) exceeds the 126 MB L2"
    meas.update(num_rendered_per_view=R_view, R_over_P=R_view / P, alg_bytes_per_view=balg_view,
                pipeline_hbm_gbs=balg_view * V / (ms_step * 1e-3) / 1e9, pipeline_frac_of_peak=balg_view * V / (ms_step * 1e-3) / 1e9 / peak,
                working_set_mb=(P * (232 + 4 * (27 + F + 3 * M)) + 100 * R_view + 8 * N * (3 + F)) / 1e6)
    dom = None
    if stages is not None:
        per = {k: (v[0] / max(v[1], 1)) for k, v in stages.items()}
        meas["stage_ms_per_launch"] = {k: round(v, 4) for k, v in per.items()}
        # hand-written kernels launched inside the timed region, per view and step: project_fwd, emit_tiles, fill_tail,
        # ranges_pack, tile_order, blend_fwd, blend_bwd; plus ONE project_bwd_views per step (multi-view path) or one per view
        out["gpu_launches"] = (7 * V + 1) * a.steps if streams else 8 * V * a.steps
        meas["library_launches_cub"] = "depth sort + scan + tile sort (CUB) per view, not counted in gpu_launches"
        dom = max(per, key=per.get)
        if per[dom] <= 0:
            dom = None
    if stages is not None and dom is not None:
        Fp = F + (1 if wl["depth"] else 0)
        live = P  # upper bound: every Gaussian's record/channel row touched once
        alg = {
            "blend_bwd": 4 * R_view + live * (32 + 4 * (3 + Fp)) + N * (4 * (3 + Fp) + 8) + P * 4 * (12 + F),
            "blend_fwd": 4 * R_view + live * (32 + 4 * (3 + Fp)) + N * (4 * (3 + Fp) + 8),
            "project_fwd": P * (44 + 12 * M + 4 + 32 + 4),
            "project_bwd": P * (44 + 12 * M + 48 + 56 + 12 * M),
            "depth_sort": 2 * 8 * P, "tile_sort": 2 * 8 * R_view, "emit_tiles": P * 20 + 8 * R_view,
            "ranges_pack": R_view * (8 + 32) + 32 * R_view, "scan": 8 * P,
        }.get(dom, 0)
        ach = alg / (per[dom] * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json"))).get(a.workload, {}).get(dom)
        except Exception:
            pass
        out["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                           "traffic": traffic, "alg_bytes_per_launch": alg, "ms_per_launch": per[dom], "peak_source": peak_src,
                           "note": "blend kernels are FP32-issue bound, not HBM bound (DESIGN.md)"}
    else:
        if stages is None:
            out["gpu_launches"] = 0
        out["roofline"] = {"bound": "hbm", "kernel": "whole pipeline", "achieved": meas["pipeline_hbm_gbs"],
                           "peak": peak, "unit": "GB/s", "frac": meas["pipeline_frac_of_peak"], "traffic": None, "peak_source": peak_src}
    if e2e is not None:
        out["e2e"] = e2e
    if c5 is not None:
        out["c5"] = c5
    if world > 1:
        meas["nccl_env"] = {k: v for k, v in os.environ.items() if k.startswith("NCCL_")}
    if nccl_log and os.path.exists(nccl_log):
        try:
            lines = [ln.strip() for ln in open(nccl_log, errors="replace") if any(k in ln for k in ("NVLS", "NCCL version", "Using network", "Channel", "nRanks", "P2P", "Ring", "Tree", "TUNING"))]
            keep = [ln for ln in lines if "Channel " not in ln and "via P2P" not in ln][:12]
            out["nccl"] = {"log_lines": [ln[-200:] for ln in keep], "nvls_lines": sum("NVLS" in ln for ln in lines),
                           "allreduce_bytes_per_step": packed_bytes}
        except Exception as ex:  # pragma: no cover
            out["nccl"] = {"error": str(ex)}
    if a.gpus == 1 and not a.no_cpu_baseline:
        try:
            out["cpu_baseline"] = cpu_baseline(wl)[0]
        except Exception as ex:  # pragma: no cover
            out["cpu_baseline"] = {"error": str(ex)}
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
