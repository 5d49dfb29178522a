"""First-hit feature buffers and denoising on device buffers and across the GPUs of one box (rtnw_render_aov_device,
rtnw_denoise_device, rtnw_render_aov_multi): against the host entry points bit for bit, each rank's rotated share against
its restatement from single-sample calls of the C oracle (tests/aov_oracle.c), the multi-GPU frame against the one-GPU
buffers and its own ranks, and argument errors.  On a one-GPU box the same device is listed several times (several
contexts, the same code path); with two GPUs also [0, 1]."""
import ctypes as C

import numpy as np
import pytest

from denoise_ref import synthetic_frame
from test_aov import KEYS, assert_matches_oracle, bits, oracle_aov, scenes  # noqa: F401 (fixtures)

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SHAPES = dict(albedo=(3, np.float32), normal=(3, np.float32), depth=(0, np.float32), hits=(0, np.int32), prim_id=(0, np.int32))
TORCH = {np.float32: torch.float32, np.int32: torch.int32}


def device_lists(rtnw):
    return [[0, 0], [0, 0, 0]] + ([[0, 1]] if rtnw.device_count() >= 2 else [])


def device_aov(ny, nx, fill=0):
    """five device tensors of a frame's AOV buffers, filled with `fill` (NaN bits for the floats when fill is None)"""
    out = {}
    for k, (c, dt) in SHAPES.items():
        t = torch.empty((ny, nx, c) if c else (ny, nx), dtype=TORCH[dt], device="cuda:0")
        t.fill_(-7 if fill is None and dt is np.int32 else float("nan") if fill is None else fill)
        out[k] = t
    return out


def ptrs(bufs):
    return {k: v.data_ptr() for k, v in bufs.items()}


def host(bufs):
    return {k: v.cpu().numpy() for k, v in bufs.items()}


def rank_share(rtnw, hs, ds, cam, nx, ny, ns, g, G, seed):
    """rank g of G's AOV share (RTNW_F_ROTATE_SAMPLES) through rtnw_render_aov_device, as host arrays, and its Stats"""
    bufs = device_aov(ny, nx, fill=None)
    p = hs.params(nx=nx, ny=ny, ns=ns, seed=seed, sample_begin=g, sample_stride=G, flags_extra=rtnw.F_ROTATE_SAMPLES)
    st = ds.render_aov_device(cam, p, ptrs(bufs))
    torch.cuda.synchronize()
    return host(bufs), st


def samples_per_pixel(nx, ny, ns, g, G):
    s0 = (g - np.arange(nx * ny).reshape(ny, nx)) % G
    return s0, np.where(s0 < ns, (ns - s0 + G - 1) // G, 0)


def restated_share(per_sample, nx, ny, ns, g, G):
    """rank g's buffers from the single-sample oracle buffers: pixel p sums its samples (g - p) mod G + k*G < ns in that
    order, in float32; prim_id is its first sample's, -1 without one"""
    s0, count = samples_per_pixel(nx, ny, ns, g, G)
    yy, xx = np.indices((ny, nx))
    planes = {k: np.stack([q[k] for q in per_sample]) for k in KEYS}
    out = {k: np.zeros_like(per_sample[0][k]) for k in ("albedo", "normal", "depth", "hits")}
    for k in range(-(-ns // G)):
        on = k < count
        s = np.minimum(s0 + k * G, ns - 1)
        for key in out:
            v = planes[key][s, yy, xx]
            out[key] = np.where(on[..., None] if v.ndim == 3 else on, out[key] + v, out[key]).astype(out[key].dtype)
    out["prim_id"] = np.where(count > 0, planes["prim_id"][np.minimum(s0, ns - 1), yy, xx], -1).astype(np.int32)
    return out


# ------------------------------------------------------------------------------------------------ rtnw_render_aov_device
@pytest.mark.parametrize("name", ["cornell_box", "cornell_smoke", "final_northstar"])
def test_device_aov_equals_host_aov(rtnw, scenes, name):
    nx, ny = 96, 64
    hs, ds = scenes(name)
    cam, params = hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=4, seed=13)
    want = ds.render_aov(cam, params)
    # on a side stream, behind a long sleep: if the call did not wait for the fill, the fill would land on its output
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        bufs = {k: torch.empty(v.shape, dtype=TORCH[v.dtype.type], device="cuda:0") for k, v in want.items()}
        torch.cuda._sleep(50_000_000)
        for k, v in bufs.items():
            v.fill_(-3)
    st = ds.render_aov_device(cam, params, ptrs(bufs), stream=side.cuda_stream)
    got = host(bufs)
    for k in KEYS:
        assert got[k].tobytes() == want[k].tobytes(), k
    assert st.paths == st.rays == nx * ny * 4 and st.kernel_launches == 1 and st.total_ms == st.kernel_ms > 0
    # the legacy default stream (0)
    bufs = device_aov(ny, nx, fill=None)
    ds.render_aov_device(cam, params, ptrs(bufs))
    got = host(bufs)
    for k in KEYS:
        assert got[k].tobytes() == want[k].tobytes(), k


@pytest.mark.parametrize("G", [2, 3])
@pytest.mark.parametrize("name", ["cornell_box", "cornell_smoke", "final_northstar"])
def test_rotated_shares_match_the_restatement(rtnw, scenes, oracle_aov, name, G):
    nx, ny, seed = 40, 30, 17
    hs, ds = scenes(name)
    cam = hs.camera(nx, ny)
    per_sample = [oracle_aov(hs.desc_ptr, cam, hs.params(nx=nx, ny=ny, ns=1, seed=seed, sample_begin=s)) for s in range(5)]
    for ns in (1, 2, 4, 5):
        total_hits = np.zeros((ny, nx), np.int64)
        for g in range(G):
            got, st = rank_share(rtnw, hs, ds, cam, nx, ny, ns, g, G, seed)
            assert_matches_oracle(rtnw, hs, got, restated_share(per_sample[:ns], nx, ny, ns, g, G))
            _, count = samples_per_pixel(nx, ny, ns, g, G)
            assert st.paths == st.rays == count.sum() and (count == 0).any() == (ns < G)
            total_hits += got["hits"]
        assert np.array_equal(total_hits, sum(q["hits"] for q in per_sample[:ns]))


# ------------------------------------------------------------------------------------------------ rtnw_render_aov_multi
@pytest.mark.parametrize("name, ns", [("final_northstar", 7), ("cornell_smoke", 2)])
def test_multi_gpu_frame(rtnw, ctx, scenes, name, ns):
    nx, ny, seed = 96, 64, 21
    hs, ds = scenes(name)
    cam, params = hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=seed)
    one = ds.render_aov(cam, params)
    dp = rtnw.DenoiseParams(5, 4.0, 1.0, 7)
    for devs in device_lists(rtnw):
        G = len(devs)
        mc = rtnw.MultiContext(devs)
        ms = mc.upload(hs.desc_ptr)
        colour, _ = ms.render(cam, params)
        sums, aov, den, st = ms.render_aov(cam, params, dp)
        assert sums.tobytes() == colour.tobytes()
        assert np.array_equal(aov["hits"], one["hits"]) and np.array_equal(aov["prim_id"], one["prim_id"])
        shares = [rank_share(rtnw, hs, ds, cam, nx, ny, ns, g, G, seed)[0] for g in range(G)]
        for k in ("albedo", "normal", "depth"):
            want = shares[0][k]
            for r in shares[1:]:
                want = want + r[k]
            assert bits(aov[k]).tobytes() == bits(want).tobytes(), k
            assert np.allclose(aov[k], one[k], rtol=1e-5, atol=1e-5), k
        assert den.tobytes() == ctx.denoise(sums, aov, ns).tobytes()
        assert st.paths == nx * ny * ns and st.rays >= st.paths
        assert st.kernel_launches >= 2 * G + 2 + dp.iterations + 2 and st.total_ms >= st.kernel_ms > 0
        sums2, aov2, none, _ = ms.render_aov(cam, params)
        assert none is None and sums2.tobytes() == sums.tobytes()
        for k in KEYS:
            assert aov2[k].tobytes() == aov[k].tobytes(), k
        ms.close()
        mc.close()


def test_one_device_multi_frame_is_the_one_gpu_frame(rtnw, ctx, scenes):
    nx, ny, ns = 64, 48, 3
    hs, ds = scenes("final_northstar")
    cam, params = hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=5)
    mc = rtnw.MultiContext([0])
    ms = mc.upload(hs.desc_ptr)
    sums, aov, den, st = ms.render_aov(cam, params, rtnw.DenoiseParams(3, 4.0, 1.0, 7))
    assert sums.tobytes() == ds.render(cam, params)[0].tobytes()
    one = ds.render_aov(cam, params)
    for k in KEYS:
        assert aov[k].tobytes() == one[k].tobytes(), k
    assert den.tobytes() == ctx.denoise(sums, aov, ns, iterations=3).tobytes()
    ms.close()
    mc.close()


# ------------------------------------------------------------------------------------------------ rtnw_denoise_device
SETTINGS = [(1, 4.0, 1.0, 7), (5, 4.0, 1.0, 7), (8, 1.5, 0.25, 2)]


def denoise_both(rtnw, ctx, sums, aov, ns, setting):
    it, sl, sz, k = setting
    kw = dict(iterations=it, sigma_luminance=sl, sigma_depth=sz, normal_power_log2=k)
    want = ctx.denoise(sums, aov, ns, **kw)
    dev = {k: torch.from_numpy(np.ascontiguousarray(aov[k])).cuda() for k in ("albedo", "normal", "depth", "hits")}
    colour = torch.from_numpy(np.ascontiguousarray(sums)).cuda()
    out = torch.full(colour.shape, float("nan"), device="cuda:0")
    st = ctx.denoise_device(colour.data_ptr(), ptrs(dev), sums.shape[1], sums.shape[0], ns, out.data_ptr(), stats=None, **kw)
    assert st.kernel_launches == it + 2 and st.total_ms == st.kernel_ms > 0 and st.paths == 0
    return out.cpu().numpy(), want


@pytest.mark.parametrize("setting", SETTINGS)
@pytest.mark.parametrize("name, nx, ny", [("cornell_box", 64, 64), ("final_northstar", 96, 64), ("earth", 96, 64)])
def test_denoise_device_equals_denoise_on_real_frames(rtnw, ctx, scenes, name, nx, ny, setting):
    hs, ds = scenes(name)
    cam, params = hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=4, seed=11)
    sums, _ = ds.render(cam, params)
    got, want = denoise_both(rtnw, ctx, sums, ds.render_aov(cam, params), 4, setting)
    assert bits(got).tobytes() == bits(want).tobytes()


@pytest.mark.parametrize("setting", SETTINGS)
@pytest.mark.parametrize("nx, ny, hit_fraction", [(1, 1, 1.0), (1, 37, 0.6), (37, 1, 0.6), (129, 67, 0.7), (129, 67, 0.0),
                                                  (129, 67, 1.0), (300, 200, 0.7)])
def test_denoise_device_equals_denoise_on_synthetic_frames(rtnw, ctx, nx, ny, hit_fraction, setting):
    sums, aov = synthetic_frame(nx, ny, 4, seed=nx * 7 + ny, hit_fraction=hit_fraction)
    got, want = denoise_both(rtnw, ctx, sums, aov, 4, setting)
    assert bits(got).tobytes() == bits(want).tobytes()


# ------------------------------------------------------------------------------------------------ argument errors
def test_rejected_arguments_leave_the_handles_usable(rtnw, ctx, scenes):
    L = rtnw.device_lib()
    nx, ny, ns = 32, 32, 3
    hs, ds = scenes("cornell_box")
    cam, good = hs.camera(nx, ny), hs.params(nx=nx, ny=ny, ns=ns, seed=4)
    want = ds.render_aov(cam, good)
    bufs = device_aov(ny, nx)
    p = ptrs(bufs)

    def aov_device(params=good, **null):
        a = rtnw.Aov(*(None if null.get(k) else p[k] for k in KEYS))
        return L.rtnw_render_aov_device(ctx._h, ds._h, C.byref(cam), C.byref(params), C.byref(a), None, None)

    for k in KEYS:
        assert aov_device(**{k: True}) == rtnw.RTNW_ERR_INVALID, k
    assert L.rtnw_render_aov_device(ctx._h, ds._h, C.byref(cam), C.byref(good), None, None, None) == rtnw.RTNW_ERR_INVALID
    for bad in (hs.params(nx=nx, ny=ny, ns=ns, pixel_count=4), hs.params(nx=nx, ny=ny, ns=ns, flags_extra=rtnw.F_ACCUMULATE),
                hs.params(nx=nx, ny=ny, ns=0), hs.params(nx=nx, ny=ny, ns=ns, sample_stride=0, flags_extra=rtnw.F_ROTATE_SAMPLES)):
        assert aov_device(bad) == rtnw.RTNW_ERR_INVALID
    assert aov_device() == rtnw.RTNW_OK
    got = host(bufs)
    for k in KEYS:
        assert got[k].tobytes() == want[k].tobytes(), k

    # rtnw_denoise_device: null buffers, overlapping output, bad parameters
    sums, _ = ds.render(cam, good)
    colour = torch.from_numpy(sums).cuda()
    out = torch.empty_like(colour)
    dp = rtnw.DenoiseParams(5, 4.0, 1.0, 7)

    def denoise(color=colour.data_ptr(), feats=None, n=(nx, ny, ns), d=dp, rgb=out.data_ptr()):
        f = [p[k] for k in ("albedo", "normal", "depth", "hits")] if feats is None else feats
        return L.rtnw_denoise_device(ctx._h, color, C.byref(rtnw.Aov(*f, None)), *n, None if d is None else C.byref(d), rgb, None, None)

    assert denoise() == rtnw.RTNW_OK
    base = [p[k] for k in ("albedo", "normal", "depth", "hits")]
    bad = [dict(color=None), dict(rgb=None), dict(d=None), dict(n=(0, ny, ns)), dict(n=(nx, ny, 0)),
           dict(d=rtnw.DenoiseParams(0, 4.0, 1.0, 7)), dict(d=rtnw.DenoiseParams(5, float("nan"), 1.0, 7)),
           dict(rgb=colour.data_ptr()), dict(rgb=colour.data_ptr() + 4), dict(rgb=p["albedo"]), dict(rgb=p["hits"] - 8)]
    bad += [dict(feats=[None if q == k else v for q, v in enumerate(base)]) for k in range(4)]
    for kw in bad:
        assert denoise(**kw) == rtnw.RTNW_ERR_INVALID, kw
    assert L.rtnw_denoise_device(ctx._h, colour.data_ptr(), None, nx, ny, ns, C.byref(dp), out.data_ptr(), None, None) == rtnw.RTNW_ERR_INVALID
    out.fill_(0)
    assert denoise() == rtnw.RTNW_OK
    assert out.cpu().numpy().tobytes() == ctx.denoise(sums, want, ns).tobytes()

    # rtnw_render_aov_multi
    mc = rtnw.MultiContext([0, 0])
    ms = mc.upload(hs.desc_ptr)
    ref_sums, ref_aov, ref_den, _ = ms.render_aov(cam, good, dp)
    h_sums = np.empty((ny, nx, 3), np.float32)
    h_den = np.empty((ny, nx, 3), np.float32)
    h_aov, h_bufs = rtnw._aov_arrays(good)

    def multi(params=good, sums_=h_sums.ctypes.data, aov=C.byref(h_bufs), d=C.byref(dp), den=h_den.ctypes.data, m=mc._h, s=ms._h):
        return L.rtnw_render_aov_multi(m, s, C.byref(cam), C.byref(params), sums_, aov, d, den, None)

    incomplete = rtnw.Aov(h_bufs.albedo, h_bufs.normal, h_bufs.depth, h_bufs.hits, None)
    bad = [dict(m=None), dict(s=None), dict(sums_=None, aov=None, d=None, den=None), dict(d=None), dict(den=None),
           dict(aov=C.byref(incomplete)), dict(d=C.byref(rtnw.DenoiseParams(9, 4.0, 1.0, 7))),
           dict(params=hs.params(nx=nx, ny=ny, ns=ns, sample_begin=1, sample_stride=2)),
           dict(params=hs.params(nx=nx, ny=ny, ns=ns, flags_extra=rtnw.F_ROTATE_SAMPLES)),
           dict(params=hs.params(nx=nx, ny=ny, ns=ns, flags_extra=rtnw.F_ACCUMULATE)),
           dict(params=hs.params(nx=nx, ny=ny, ns=ns, pixel_count=5)), dict(params=hs.params(nx=nx, ny=ny, ns=0))]
    for kw in bad:
        assert multi(**kw) == rtnw.RTNW_ERR_INVALID, kw
    assert multi() == rtnw.RTNW_OK
    assert h_sums.tobytes() == ref_sums.tobytes() and h_den.tobytes() == ref_den.tobytes()
    for k in KEYS:
        assert h_aov[k].tobytes() == ref_aov[k].tobytes(), k
    # each output on its own
    h_sums[:] = np.nan
    assert multi(aov=None, d=None, den=None) == rtnw.RTNW_OK and h_sums.tobytes() == ref_sums.tobytes()
    h_den[:] = np.nan
    assert multi(sums_=None, aov=None) == rtnw.RTNW_OK and h_den.tobytes() == ref_den.tobytes()
    ms.close()
    mc.close()
