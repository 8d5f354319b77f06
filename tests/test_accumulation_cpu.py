"""The numpy replay of AccumulationBuffer::update_pixel (accumulation_buffer.rs:44-60) that the GPU accumulation tests
(test_gpu_accumulation.py) compare every resolve kernel with, checked here bit for bit against the oracle's own update.

The replay uses elementwise binary64 operations only (numpy never fuses a multiply-add), in the kernels' order:

    wy = 1.0 - wb; wt = w + wy; wb = (wt - w) - wy; w = wt
    y = c * 1.0 - b; t = s + y; b = (t - s) - y; s = t
    q = q + c.y * c.y;   colour = s * (1.0 / w)

where c is a sample's XYZ (ColourXyz::from_photon) and q the y_sq_sum the pass-based calls keep."""
import ctypes as C

import numpy as np

import oraclelib as O

STATE = (("colour_sum", 3), ("colour_bias", 3), ("weight", 1), ("weight_bias", 1), ("y_sq_sum", 1))
OUTPUTS = (("colour", 3),) + STATE


def replay(state0, per_sample, active=None):
    """Apply `per_sample` (k, npix, 3: sample j's XYZ for every pixel, in sample order) to `state0` (a dict of the STATE
    arrays; a missing or None array is zeros, as a NULL array of a continued call is).  active: optional (k, npix) bool;
    sample j changes only the pixels where active[j] is set.  Returns fresh arrays of OUTPUTS, flat like the library's."""
    per_sample = np.asarray(per_sample, np.float64)
    npix = per_sample.shape[1]

    def get(name, per):
        v = state0.get(name)
        return np.zeros((npix, per) if per > 1 else npix) if v is None else np.array(v, np.float64).reshape((npix, per) if per > 1 else npix)

    s, b, w, wb, q = (get(n, per) for n, per in STATE)
    with np.errstate(all="ignore"):
        for j, c in enumerate(per_sample):
            wy = 1.0 - wb
            wt = w + wy
            nwb = (wt - w) - wy
            y = c * 1.0 - b
            t = s + y
            nb = (t - s) - y
            nq = q + c[:, 1] * c[:, 1]
            if active is None:
                w, wb, s, b, q = wt, nwb, t, nb, nq
            else:
                m = np.asarray(active[j], bool)
                w, wb, q = np.where(m, wt, w), np.where(m, nwb, wb), np.where(m, nq, q)
                s, b = np.where(m[:, None], t, s), np.where(m[:, None], nb, b)
        colour = s * (1.0 / w)[:, None]
    return {"colour": colour.reshape(-1), "colour_sum": s.reshape(-1), "colour_bias": b.reshape(-1), "weight": w.copy(),
            "weight_bias": wb.copy(), "y_sq_sum": q.copy()}


def cmf_xyz(wavelengths):
    """the oracle's colour matching functions (colour_xyz.rs) at each wavelength: (n, 3)"""
    L = O.lib()
    out = np.zeros((len(wavelengths), 3))
    for i, lam in enumerate(wavelengths):
        L.orc_cmf_xyz(float(lam), out[i].ctypes.data_as(O.dp))
    return out


def random_states(rng, n):
    """states a real accumulator can hold and ones it cannot: sums of any sign and scale, biases of up to an ulp of the
    sum (either sign, some exactly zero), weights integral and not, weight biases of up to an ulp of the weight"""
    scale = 10.0 ** rng.uniform(-6, 4, (n, 1))
    s = rng.uniform(-0.2, 1.0, (n, 3)) * scale
    b = rng.uniform(-1.0, 1.0, (n, 3)) * np.spacing(np.abs(s))
    b[rng.random((n, 3)) < 0.2] = 0.0
    w = np.where(rng.random(n) < 0.5, rng.integers(0, 1 << 20, n).astype(np.float64), rng.uniform(0.0, 1e6, n))
    wb = rng.uniform(-1.0, 1.0, n) * np.spacing(np.maximum(w, 1.0))
    wb[rng.random(n) < 0.2] = 0.0
    return {"colour_sum": s, "colour_bias": b, "weight": w, "weight_bias": wb}


def test_replay_equals_the_oracle_update_bit_for_bit():
    """2000 random states, 1-19 updates each, intensities +0, -0 and up to 1e3: the replay's five arrays equal, bit for bit,
    what orc_accum_update (PixelAccum::update with weight 1) leaves."""
    L = O.lib()
    rng = np.random.default_rng(20261021)
    n, kmax = 2000, 19
    st0 = random_states(rng, n)
    k = rng.integers(1, kmax + 1, n)
    lam = rng.uniform(380.0, 780.0, (kmax, n))
    intensity = rng.uniform(0.0, 1.0, (kmax, n)) * 10.0 ** rng.uniform(-8, 3, (kmax, n))
    intensity[rng.random((kmax, n)) < 0.3] = 0.0
    intensity[rng.random((kmax, n)) < 0.05] = -0.0
    xyz = cmf_xyz(lam.reshape(-1)).reshape(kmax, n, 3)
    c = xyz * intensity[..., None]
    active = np.arange(kmax)[:, None] < k[None, :]
    got = replay(st0, c, active)

    want = {name: np.zeros((n, per)) for name, per in OUTPUTS[:-1]}
    st = np.zeros(11)
    for i in range(n):
        st[:] = 0.0
        st[3:6], st[6:9], st[9], st[10] = st0["colour_sum"][i], st0["colour_bias"][i], st0["weight"][i], st0["weight_bias"][i]
        for j in range(k[i]):
            L.orc_accum_update(st.ctypes.data_as(O.dp), float(lam[j, i]), float(intensity[j, i]), 1.0)
        want["colour"][i], want["colour_sum"][i], want["colour_bias"][i] = st[0:3], st[3:6], st[6:9]
        want["weight"][i], want["weight_bias"][i] = st[9], st[10]
    assert (c == 0.0).any() and (st0["colour_bias"] != 0.0).any() and (st0["weight"] % 1.0 != 0.0).any()
    for name, per in OUTPUTS[:-1]:
        a, b = got[name].reshape(n, per), want[name].reshape(n, per)
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), (name, np.flatnonzero((a.view(np.uint64) != b.view(np.uint64)).any(1))[:5])
    # the compensation terms really did something: a plain sum differs from the Kahan sum somewhere
    plain = st0["colour_sum"] + np.where(active[..., None], c, 0.0).sum(0)
    assert (plain != got["colour_sum"].reshape(n, 3)).any()


def test_replay_keeps_y_sq_sum_and_treats_missing_arrays_as_zeros():
    rng = np.random.default_rng(3)
    c = rng.uniform(0.0, 2.0, (5, 4, 3))
    full = replay({n: np.zeros(4 * per) for n, per in STATE}, c)
    assert np.array_equal(replay({}, c)["colour_sum"], full["colour_sum"])
    q = np.zeros(4)
    for j in range(5):
        q = q + c[j, :, 1] * c[j, :, 1]
    assert np.array_equal(full["y_sq_sum"], q) and np.array_equal(full["weight"], np.full(4, 5.0))
    # one sample into a zero state is the sample itself, with zero compensation: the identity the GPU tests extract samples by
    one = replay({}, c[:1])
    assert np.array_equal(one["colour_sum"], c[0].reshape(-1)) and not one["colour_bias"].any() and not one["weight_bias"].any()
    # an inactive sample leaves the pixel's bits as they were
    part = replay({}, c, active=np.arange(5)[:, None] < np.array([0, 1, 3, 5])[None, :])
    assert np.isnan(part["colour"][:3]).all() and np.array_equal(part["weight"], [0.0, 1.0, 3.0, 5.0])
    assert np.array_equal(part["colour_sum"][9:], full["colour_sum"][9:])
