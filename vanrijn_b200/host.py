"""Script-level plumbing over the host library: build a scene from a scenes.SceneSpec through the
C++ host mirror (load_obj, BoundingVolumeHierarchy::build, flatten), upload it, and call the
C ABI.  Nothing here computes a ray, a hit or a colour; it only moves arrays across ctypes."""
import ctypes as C

import numpy as np

from . import capi
from .capi import dp


def _d(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(dp)


class HostScene:
    """A vanrijn::Scene built by the C++ host side, plus its flattened / uploaded forms."""

    def __init__(self, spec, device_builder=False, per_triangle_objects=False):
        """device_builder: False/0 = BoundingVolumeHierarchy::build on the host; True/1 = on the GPU (vrj_bvh_build);
        "upload"/2 = only the triangles are kept and the tree is built on the GPU inside vrj_scene_create.
        The tree is the same in all three cases.  per_triangle_objects: build through one Triangle object per triangle,
        like the reference's Vec<Arc<dyn Primitive>> (same result; the default goes through arrays)."""
        H = capi.host()
        self.device_builder = (2 if device_builder == "upload" else int(device_builder)) | (4 if per_triangle_objects else 0)
        self.H = H
        self.h = C.c_void_p(H.vrjh_scene_new(*[float(x) for x in spec.camera]))
        self.spec = spec
        self._keep = []
        for sp in spec.spectra:
            if sp[0] == "rgb":
                H.vrjh_add_spectrum_rgb(self.h, *[float(x) for x in sp[1]])
            elif sp[0] == "grey":
                H.vrjh_add_spectrum_grey(self.h, float(sp[1]))
            elif sp[0] == "diamond":
                H.vrjh_add_spectrum_diamond(self.h)
            else:
                arr, p = _d(sp[3])
                H.vrjh_add_spectrum(self.h, float(sp[1]), float(sp[2]), len(arr), p)
        for m in spec.materials:
            H.vrjh_add_material(self.h, m.kind, m.spectrum, m.p0, m.p1, m.p2)
        for obj in spec.objects:
            if obj[0] == "list":
                H.vrjh_begin_list(self.h)
                for prim in obj[1]:
                    if prim[0] == "sphere":
                        H.vrjh_list_add_sphere(self.h, *[float(x) for x in prim[1]], float(prim[2]), prim[3])
                    elif prim[0] == "plane":
                        H.vrjh_list_add_plane(self.h, *[float(x) for x in prim[1]], float(prim[2]), prim[3])
                    else:
                        v, pv = _d(prim[1])
                        n, pn = _d(prim[2])
                        H.vrjh_list_add_triangle(self.h, pv, pn, prim[3])
            elif obj[0] == "mesh":
                v, pv = _d(obj[1])
                n, pn = _d(obj[2])
                r = H.vrjh_add_bvh(self.h, v.size // 9, pv, pn, obj[3], int(self.device_builder))
                if r < 0:
                    raise capi.VrjError(H.vrjh_last_error().decode())
            elif obj[0] == "obj":
                r = H.vrjh_add_bvh_obj(self.h, obj[1].encode(), obj[2], int(self.device_builder))
                if r < 0:
                    raise capi.VrjError(H.vrjh_last_error().decode())
        self._dev = {}

    def save_cache(self, path):
        """save_scene_cache: the flattened scene (primitives, triangles, tree if built on the host) to one file."""
        if self.H.vrjh_scene_save_cache(self.h, str(path).encode()) != 0:
            raise capi.VrjError(self.H.vrjh_last_error().decode())

    @classmethod
    def from_cache(cls, path, spec=None):
        """load_scene_cache: a scene that can be rendered (and flattened) but holds no primitive objects."""
        self = cls.__new__(cls)
        self.H = capi.host()
        h = self.H.vrjh_scene_load_cache(str(path).encode())
        if not h:
            raise capi.VrjError(self.H.vrjh_last_error().decode())
        self.h, self.spec, self._keep, self._dev, self.device_builder = C.c_void_p(h), spec, [], {}, 0
        return self

    def __del__(self):
        try:
            for comm, ms in getattr(self, "_comm", {}).values():
                capi.cuda().vrj_comm_scene_destroy(ms)
                capi.cuda().vrj_comm_destroy(comm)
            self.H.vrjh_scene_free(self.h)
        except Exception:
            pass

    # ---- flattened description (host memory, owned by the C++ scene) ----
    def desc(self):
        d = self.H.vrjh_flatten(self.h)
        if not d:
            raise capi.VrjError(self.H.vrjh_last_error().decode())
        return d.contents

    def spectrum_data(self, spectrum_id):
        """(SpectrumData, keepalive) for a spectrum of the spec, e.g. a light's."""
        lo, hi = C.c_double(), C.c_double()
        # the first call only returns the count: a spectrum may hold any number of samples
        n = self.H.vrjh_get_spectrum(self.h, spectrum_id, C.byref(lo), C.byref(hi), None, 0)
        if n < 0:
            raise capi.VrjError(self.H.vrjh_last_error().decode())
        buf = np.zeros(max(n, 1))
        self.H.vrjh_get_spectrum(self.h, spectrum_id, C.byref(lo), C.byref(hi), buf.ctypes.data_as(dp), n)
        buf = buf[:n]
        return capi.SpectrumData(lo.value, hi.value, n, 0, buf.ctypes.data_as(dp)), buf

    # ---- device ----
    def device_scene(self, device=0):
        if device not in self._dev:
            s = self.H.vrjh_device_scene(self.h, device)
            if not s:
                raise capi.VrjError(self.H.vrjh_last_error().decode())
            self._dev[device] = C.c_void_p(s)
        return self._dev[device]

    def device_bytes(self, device=0):
        return int(capi.cuda().vrj_scene_device_bytes(self.device_scene(device)))

    def trace(self, origins, dirs, bvh_filter=capi.FILTER_F32, device=0):
        o, po = _d(origins)
        d, pd = _d(dirs)
        n = o.size // 3
        obj = np.empty(n, np.int32)
        prim = np.empty(n, np.int32)
        t = np.empty(n, np.float64)
        st = capi.Stats()
        capi.check(capi.cuda().vrj_trace_rays(self.device_scene(device), n, po, pd, bvh_filter,
                                              obj.ctypes.data_as(C.POINTER(C.c_int32)),
                                              prim.ctypes.data_as(C.POINTER(C.c_int32)), t.ctypes.data_as(dp), C.byref(st)))
        return obj, prim, t, st

    def make_params(self, spp=1, max_depth=128, sample_offset=0, seed=1, integrator=capi.INTEGRATOR_SIMPLE_RANDOM,
                    bvh_filter=capi.FILTER_F32, bias=1e-7, lights=(), ambient=-1, sample_stride=1, count_traversal=False,
                    precision=capi.PRECISION_F64):
        keep = []
        larr = (capi.Light * max(1, len(lights)))()
        for i, (direction, spectrum_id) in enumerate(lights):
            larr[i].direction[:] = [float(x) for x in direction]
            sd, buf = self.spectrum_data(spectrum_id)
            larr[i].spectrum = sd
            keep.append(buf)
        amb = None
        if ambient >= 0:
            amb, buf = self.spectrum_data(ambient)
            keep.append(buf)
        p = capi.RenderParams(spp=spp, max_depth=max_depth, sample_offset=sample_offset, seed=seed, integrator=integrator,
                              bvh_filter=bvh_filter, bias=bias, lights=larr,
                              ambient_light=C.pointer(amb) if amb is not None else None, n_lights=len(lights),
                              sample_stride=sample_stride, count_traversal=1 if count_traversal else 0, precision=precision)
        keep.extend([larr, amb])
        return p, keep

    def render(self, tile, height, width, want=("colour", "colour_sum", "colour_bias", "weight", "weight_bias"),
               want_photons=False, device=0, buffers=None, **kw):
        """vrj_render_tile with host output buffers (`buffers`: optional dict of caller-owned, e.g. pinned,
        float64 arrays to fill instead of fresh ones).  Returns a dict of numpy arrays + 'stats'."""
        sc, ec, sr, er = tile
        npix = (ec - sc) * (er - sr)
        p, keep = self.make_params(**kw)
        out = {}
        ao = capi.AccumOut(memory=capi.MEM_HOST, accumulate=0)
        for name, per in (("colour", 3), ("colour_sum", 3), ("colour_bias", 3), ("weight", 1), ("weight_bias", 1)):
            if name in want:
                out[name] = buffers[name] if buffers is not None else np.zeros(npix * per)
                assert out[name].size == npix * per and out[name].dtype == np.float64
                setattr(ao, name, out[name].ctypes.data)
        if want_photons:
            out["photons"] = np.zeros(p.spp * npix * 2)
            ao.photons = out["photons"].ctypes.data
        if "srgb8" in want:
            out["srgb8"] = np.zeros(npix * 3, np.uint8)
            ao.srgb8 = out["srgb8"].ctypes.data
        st = capi.Stats()
        ao.stats = C.pointer(st)
        t = capi.Tile(sc, ec, sr, er)
        capi.check(capi.cuda().vrj_render_tile(self.device_scene(device), C.byref(t), height, width, C.byref(p), C.byref(ao)))
        if want_photons:
            out["photons"] = out["photons"].reshape(p.spp, npix, 2)
        out["stats"] = st
        return out

    def render_adaptive(self, tile, height, width, min_samples, max_samples, pass_samples, rel_error, abs_floor=0.0,
                        want=("colour", "colour_sum", "colour_bias", "weight", "weight_bias", "y_sq_sum"), device=0, **kw):
        """vrj_render_adaptive with host output buffers: every pixel takes min_samples, then pass_samples more per pass until
        the standard error of its mean Y is at most rel_error * max(mean, abs_floor) or it holds max_samples.  `kw` are the
        render parameters of make_params (spp excepted; pass spp=... to check the call refuses it).  Returns a dict of numpy
        arrays (those in `want`, "srgb8" included if asked for) + 'stats' (VrjStats) + 'adaptive' (VrjAdaptiveStats)."""
        sc, ec, sr, er = tile
        npix = (ec - sc) * (er - sr)
        kw.setdefault("spp", 0)
        p, keep = self.make_params(**kw)
        ap = capi.AdaptiveParams(min_samples=min_samples, max_samples=max_samples, pass_samples=pass_samples,
                                 rel_error=rel_error, abs_floor=abs_floor)
        out = {}
        ao = capi.AccumOut(memory=capi.MEM_HOST, accumulate=0)
        for name, per in (("colour", 3), ("colour_sum", 3), ("colour_bias", 3), ("weight", 1), ("weight_bias", 1)):
            if name in want:
                out[name] = np.zeros(npix * per)
                setattr(ao, name, out[name].ctypes.data)
        if "srgb8" in want:
            out["srgb8"] = np.zeros(npix * 3, np.uint8)
            ao.srgb8 = out["srgb8"].ctypes.data
        ysq = None
        if "y_sq_sum" in want:
            out["y_sq_sum"] = np.zeros(npix)
            ysq = out["y_sq_sum"].ctypes.data
        st, ast = capi.Stats(), capi.AdaptiveStats()
        ao.stats = C.pointer(st)
        t = capi.Tile(sc, ec, sr, er)
        capi.check(capi.cuda().vrj_render_adaptive(self.device_scene(device), C.byref(t), height, width, C.byref(p), C.byref(ap),
                                                   C.byref(ao), ysq, C.byref(ast)))
        out["stats"], out["adaptive"] = st, ast
        return out

    def render_progressive(self, tile, height, width, min_samples, max_samples, pass_samples, rel_error, abs_floor=0.0,
                           max_passes=0, state=None, want=("colour",), device=0, **kw):
        """vrj_render_progressive with host buffers: continues `state` (the dict a previous call returned; None: start from
        zero) for at most `max_passes` passes (0: until no pixel is active) of the adaptive schedule.  `want` adds the optional
        outputs ("colour", "srgb8"); `kw` are the render parameters of make_params (spp excepted).  Returns a dict with the
        new state (colour_sum, colour_bias, weight, weight_bias, y_sq_sum: fresh arrays, `state` is not modified), the wanted
        outputs, 'stats' (VrjStats) and 'progressive' (VrjProgressiveStats)."""
        sc, ec, sr, er = tile
        npix = (ec - sc) * (er - sr)
        kw.setdefault("spp", 0)
        p, keep = self.make_params(**kw)
        pp = capi.ProgressiveParams(min_samples=min_samples, max_samples=max_samples, pass_samples=pass_samples,
                                    max_passes=max_passes, rel_error=rel_error, abs_floor=abs_floor)
        out = {}
        ao = capi.AccumOut(memory=capi.MEM_HOST, accumulate=0 if state is None else 1)
        for name, per in (("colour_sum", 3), ("colour_bias", 3), ("weight", 1), ("weight_bias", 1), ("y_sq_sum", 1)):
            out[name] = np.zeros(npix * per) if state is None else np.array(state[name], np.float64, copy=True)
            assert out[name].size == npix * per
            if name != "y_sq_sum":
                setattr(ao, name, out[name].ctypes.data)
        if "colour" in want:
            out["colour"] = np.zeros(npix * 3)
            ao.colour = out["colour"].ctypes.data
        if "srgb8" in want:
            out["srgb8"] = np.zeros(npix * 3, np.uint8)
            ao.srgb8 = out["srgb8"].ctypes.data
        st, pst = capi.Stats(), capi.ProgressiveStats()
        ao.stats = C.pointer(st)
        t = capi.Tile(sc, ec, sr, er)
        capi.check(capi.cuda().vrj_render_progressive(self.device_scene(device), C.byref(t), height, width, C.byref(p), C.byref(pp),
                                                      C.byref(ao), out["y_sq_sum"].ctypes.data, C.byref(pst)))
        out["stats"], out["progressive"] = st, pst
        return out

    def render_counts(self, tile, height, width, counts, state=None, want=("colour",), device=0, **kw):
        """vrj_render_counts with host buffers: pixel p of `tile` takes counts[p] (uint32, one per tile pixel, row-major) new
        samples in full wavefronts, continuing `state` (a dict with colour_sum, colour_bias, weight, weight_bias and y_sq_sum,
        as render_progressive / render_counts return it; None: start from zero).  `want` adds the optional outputs ("colour",
        "srgb8"); `kw` are the render parameters of make_params (spp excepted).  Returns a dict with the new state (fresh
        arrays; `state` is not modified), the wanted outputs, 'stats' (VrjStats) and 'counts' (VrjCountsStats)."""
        sc, ec, sr, er = tile
        npix = (ec - sc) * (er - sr)
        kw.setdefault("spp", 0)
        p, keep = self.make_params(**kw)
        cmap = np.ascontiguousarray(counts, dtype=np.uint32).reshape(-1)
        assert cmap.size == npix, (cmap.size, npix)
        out = {}
        ao = capi.AccumOut(memory=capi.MEM_HOST, accumulate=0 if state is None else 1)
        for name, per in (("colour_sum", 3), ("colour_bias", 3), ("weight", 1), ("weight_bias", 1), ("y_sq_sum", 1)):
            out[name] = np.zeros(npix * per) if state is None else np.array(state[name], np.float64, copy=True)
            assert out[name].size == npix * per
            if name != "y_sq_sum":
                setattr(ao, name, out[name].ctypes.data)
        if "colour" in want:
            out["colour"] = np.zeros(npix * 3)
            ao.colour = out["colour"].ctypes.data
        if "srgb8" in want:
            out["srgb8"] = np.zeros(npix * 3, np.uint8)
            ao.srgb8 = out["srgb8"].ctypes.data
        st, cst = capi.Stats(), capi.CountsStats()
        ao.stats = C.pointer(st)
        t = capi.Tile(sc, ec, sr, er)
        capi.check(capi.cuda().vrj_render_counts(self.device_scene(device), C.byref(t), height, width, C.byref(p), cmap.ctypes.data,
                                                 C.byref(ao), out["y_sq_sum"].ctypes.data, C.byref(cst)))
        out["stats"], out["counts"] = st, cst
        return out

    def render_planned(self, tile, height, width, min_samples, max_samples, pass_samples, rel_error, abs_floor=0.0, rounds=0,
                       state=None, want=("colour",), device=0, **kw):
        """The planned loop: plan_counts -> render_counts, for at most `rounds` rounds (0: until a plan asks for no sample),
        from `state` (None: zero, so the first round is the uniform pilot at min_samples).  Returns the last render_counts
        dict (the state itself when no round ran) with 'rounds', 'samples' and 'batches' of this loop and 'plan' (the
        VrjPlanStats of the last plan)."""
        sc, ec, sr, er = tile
        npix = (ec - sc) * (er - sr)
        if state is None:
            state = {"colour_sum": np.zeros(npix * 3), "colour_bias": np.zeros(npix * 3), "weight": np.zeros(npix),
                     "weight_bias": np.zeros(npix), "y_sq_sum": np.zeros(npix)}
        res, n, samples, batches = dict(state), 0, 0, 0
        while rounds == 0 or n < rounds:
            counts, plan = plan_counts(res["weight"], res["colour_sum"], res["y_sq_sum"], min_samples, max_samples, pass_samples,
                                       rel_error, abs_floor, device=device)
            res["plan"] = plan
            if plan.samples == 0:
                break
            res = self.render_counts(tile, height, width, counts, state=res, want=want, device=device, **kw)
            res["plan"] = plan
            n, samples, batches = n + 1, samples + res["counts"].samples, batches + res["counts"].batches
        res["rounds"], res["samples"], res["batches"] = n, samples, batches
        return res

    def render_aux(self, tile, height, width, spp=1, want=("normal", "depth", "object_id", "material"), device=0, **kw):
        """vrj_render_aux with host output buffers: the first-hit features of the camera rays that a render with the same
        spp, seed, sample_offset and sample_stride traces (`kw`: the other keywords of make_params).  Returns a dict of numpy
        arrays (those in `want`: normal, 3 per pixel; depth; object_id and material, int32) + 'stats'."""
        sc, ec, sr, er = tile
        npix = (ec - sc) * (er - sr)
        p, keep = self.make_params(spp=spp, **kw)
        ao = capi.AuxOut(memory=capi.MEM_HOST)
        out = {}
        for name, per, dtype in (("normal", 3, np.float64), ("depth", 1, np.float64), ("object_id", 1, np.int32), ("material", 1, np.int32)):
            if name in want:
                out[name] = np.zeros(npix * per, dtype)
                setattr(ao, name, out[name].ctypes.data)
        st = capi.Stats()
        ao.stats = C.pointer(st)
        t = capi.Tile(sc, ec, sr, er)
        capi.check(capi.cuda().vrj_render_aux(self.device_scene(device), C.byref(t), height, width, C.byref(p), C.byref(ao)))
        out["stats"] = st
        return out

    def render_device(self, tile, height, width, sum_ptr, weight_ptr, device=0, accumulate=False, colour_ptr=None, **kw):
        """vrj_render_tile writing colour_sum / weight straight into caller-owned DEVICE memory
        (e.g. torch tensors that torch.distributed then reduces).  Returns the stats."""
        p, keep = self.make_params(**kw)
        ao = capi.AccumOut(memory=capi.MEM_DEVICE, accumulate=1 if accumulate else 0)
        ao.colour_sum = sum_ptr
        ao.weight = weight_ptr
        if colour_ptr:
            ao.colour = colour_ptr
        st = capi.Stats()
        ao.stats = C.pointer(st)
        t = capi.Tile(*tile)
        capi.check(capi.cuda().vrj_render_tile(self.device_scene(device), C.byref(t), height, width, C.byref(p), C.byref(ao)))
        return st

    def render_sharded(self, devices, tile, height, width, want=("colour", "colour_sum", "weight"), **kw):
        """vrj_comm_* path: one process, the scene replicated on `devices`, samples sharded by index, one NCCL
        reduce into devices[0].  Host outputs.  The communicator and replicas are cached on this object."""
        L = capi.cuda()
        key = tuple(devices)
        if not hasattr(self, "_comm"):
            self._comm = {}
        if key not in self._comm:
            comm, ms = C.c_void_p(), C.c_void_p()
            arr = (C.c_int32 * len(devices))(*devices)
            capi.check(L.vrj_comm_create(len(devices), arr, C.byref(comm)))
            d = self.desc()
            capi.check(L.vrj_comm_scene_create(comm, C.byref(d), C.byref(ms)))
            self._comm[key] = (comm, ms)
        comm, ms = self._comm[key]
        sc, ec, sr, er = tile
        npix = (ec - sc) * (er - sr)
        p, keep = self.make_params(**kw)
        out = {}
        ao = capi.AccumOut(memory=capi.MEM_HOST, accumulate=0)
        for name, per in (("colour", 3), ("colour_sum", 3), ("colour_bias", 3), ("weight", 1), ("weight_bias", 1)):
            if name in want:
                out[name] = np.zeros(npix * per)
                setattr(ao, name, out[name].ctypes.data)
        st = capi.Stats()
        ao.stats = C.pointer(st)
        t = capi.Tile(sc, ec, sr, er)
        capi.check(L.vrj_render_sharded(ms, C.byref(t), height, width, C.byref(p), C.byref(ao)))
        out["stats"] = st
        return out

    def partial_render_scene(self, tile, height, width, seed=1, sample_offset=None):
        """The reference call: partial_render_scene(&scene, tile, height, width) -> AccumulationBuffer.
        sample_offset=None is the reference's behaviour -- every call renders a fresh sample (the index comes from the
        host library's process-wide counter, next_sample_index()); pass an index for a reproducible render."""
        if sample_offset is None:
            sample_offset = 0xFFFFFFFFFFFFFFFF
        sc, ec, sr, er = tile
        npix = (ec - sc) * (er - sr)
        out = {k: np.zeros(npix * 3) for k in ("colour", "colour_sum", "colour_bias")}
        out["weight"] = np.zeros(npix)
        out["weight_bias"] = np.zeros(npix)
        t4 = (C.c_uint64 * 4)(sc, ec, sr, er)
        r = self.H.vrjh_partial_render_scene(self.h, t4, height, width, seed, sample_offset, *[out[k].ctypes.data_as(dp) for k in
                                             ("colour", "colour_sum", "colour_bias", "weight", "weight_bias")])
        if r != 0:
            raise capi.VrjError(self.H.vrjh_last_error().decode())
        return out


def render_like_main(hs, width, height, calls, workers, tile_size=2048, spp=0, max_depth=128, seed=1, sample_offset=0,
                     kahan_state=True, device=0, colour=None, weight=None):
    """main.rs:192-217 through the C++ mirror (render_like_main): `workers` threads call partial_render_scene on the cycled
    tiles, the calling thread merge_tile()s.  spp=0: the reference's own call (1 spp, limit 128, fresh samples).
    Returns (colour, weight, stats dict)."""
    n = width * height
    colour = np.zeros(n * 3) if colour is None else colour
    weight = np.zeros(n) if weight is None else weight
    st = np.zeros(9)
    r = hs.H.vrjh_render_like_main(hs.h, width, height, tile_size, calls, workers, spp, max_depth, seed, sample_offset,
                                   1 if kahan_state else 0, device, colour.ctypes.data_as(dp), weight.ctypes.data_as(dp),
                                   st.ctypes.data_as(dp))
    if r != 0:
        raise capi.VrjError(hs.H.vrjh_last_error().decode())
    keys = ("wall_s", "call_s", "merge_s", "device_ms", "rays", "calls", "bytes_to_host", "merge_passes", "wavefront_calls")
    return colour, weight, dict(zip(keys, [float(x) for x in st[:9]]))


def tone_map(colour, source=capi.TONEMAP_XYZ, device=0):
    """ClampingToneMapper on host arrays through the device (vrj_tone_map): (n,3) float64 -> (n,3) uint8."""
    c = np.ascontiguousarray(colour, dtype=np.float64).reshape(-1, 3)
    out = np.zeros((c.shape[0], 3), np.uint8)
    capi.check(capi.cuda().vrj_tone_map(device, capi.MEM_HOST, source, c.ctypes.data_as(dp), c.shape[0], out.ctypes.data))
    return out


def plan_counts(weight, colour_sum, y_sq_sum, min_samples, max_samples, pass_samples, rel_error, abs_floor=0.0, device=0):
    """vrj_plan_counts on a host state: the count map (uint32, one per pixel) that the rule of the header gives each
    pixel, and the VrjPlanStats."""
    ins = [np.ascontiguousarray(weight, np.float64), np.ascontiguousarray(colour_sum, np.float64),
           np.ascontiguousarray(y_sq_sum, np.float64)]
    npix = ins[0].size
    assert ins[1].size == 3 * npix and ins[2].size == npix
    counts = np.zeros(npix, np.uint32)
    rule = capi.AdaptiveParams(min_samples=min_samples, max_samples=max_samples, pass_samples=pass_samples,
                               rel_error=rel_error, abs_floor=abs_floor)
    ps = capi.PlanStats()
    capi.check(capi.cuda().vrj_plan_counts(device, capi.MEM_HOST, npix, *[a.ctypes.data for a in ins], C.byref(rule),
                                           counts.ctypes.data, C.byref(ps)))
    return counts, ps


# vrj_denoise's defaults (VRJ_DENOISE_DEFAULT_* in include/vanrijn_cuda.h), chosen with tools/denoise_quality.py
DENOISE_ITERATIONS, DENOISE_SIGMA_LUMINANCE, DENOISE_SIGMA_NORMAL, DENOISE_SIGMA_DEPTH = 4, 32.0, 128.0, 0.5


def denoise(colour_sum, weight, y_sq_sum, aux, tile_width, tile_height, iterations=DENOISE_ITERATIONS,
            sigma_luminance=DENOISE_SIGMA_LUMINANCE, sigma_normal=DENOISE_SIGMA_NORMAL, sigma_depth=DENOISE_SIGMA_DEPTH,
            want_srgb8=False, device=0):
    """vrj_denoise on host arrays: one tile's colour_sum / weight / y_sq_sum (HostScene.render_adaptive) and the normal /
    depth / material of `aux` (HostScene.render_aux).  Returns a dict: colour (npix * 3 float64), srgb8 (npix * 3 uint8, if
    asked for) and device_ms."""
    npix = tile_width * tile_height
    ins = [np.ascontiguousarray(colour_sum, np.float64), np.ascontiguousarray(weight, np.float64),
           np.ascontiguousarray(y_sq_sum, np.float64), np.ascontiguousarray(aux["normal"], np.float64),
           np.ascontiguousarray(aux["depth"], np.float64), np.ascontiguousarray(aux["material"], np.int32)]
    for a, per in zip(ins, (3, 1, 1, 3, 1, 1)):
        assert a.size == npix * per, (a.size, npix, per)
    out = {"colour": np.zeros(npix * 3)}
    if want_srgb8:
        out["srgb8"] = np.zeros(npix * 3, np.uint8)
    ms = C.c_double(0.0)
    params = capi.DenoiseParams(iterations=iterations, sigma_luminance=sigma_luminance, sigma_normal=sigma_normal,
                                sigma_depth=sigma_depth)
    capi.check(capi.cuda().vrj_denoise(device, capi.MEM_HOST, tile_width, tile_height, *[a.ctypes.data for a in ins], C.byref(params),
                                       out["colour"].ctypes.data, out["srgb8"].ctypes.data if want_srgb8 else None, C.byref(ms)))
    out["device_ms"] = ms.value
    return out


def bvh_build(vertices, device=0):
    """vrj_bvh_build on (n, 9) float64 vertices -> dict(order, node_min, node_max, node_child, depth, stats)."""
    v = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 9)
    n = v.shape[0]
    n_nodes = 2 * n - 1 if n else 1
    order = np.zeros(max(n, 1), np.uint32)
    node_min, node_max = np.zeros((n_nodes, 4)), np.zeros((n_nodes, 4))
    child = np.zeros((n_nodes, 2), np.int32)
    depth, stats = C.c_uint32(0), capi.BvhBuildStats()
    capi.check(capi.cuda().vrj_bvh_build(device, n, v.ctypes.data_as(dp), order.ctypes.data_as(C.POINTER(C.c_uint32)),
                                         node_min.ctypes.data_as(dp), node_max.ctypes.data_as(dp),
                                         child.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(depth), C.byref(stats)))
    return dict(order=order[:n], node_min=node_min, node_max=node_max, node_child=child, depth=depth.value, stats=stats)


def build_scene(spec, device_builder=False, per_triangle_objects=False):
    return HostScene(spec, device_builder=device_builder, per_triangle_objects=per_triangle_objects)
