"""The C restatement of rtnw_denoise (tests/denoise_oracle.c) compiled with the oracle's flags into a temporary directory, and
synthetic denoiser inputs.  TEST INFRASTRUCTURE for tests/test_denoise_cpu.py and tests/test_denoise.py."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent


class DenoiseOracle:
    def __init__(self, rtnw, tmpdir):
        so = Path(tmpdir) / "libdenoise_oracle.so"
        subprocess.run([os.environ.get("CC", "gcc"), "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra",
                        f"-I{ROOT / 'include'}", "-shared", "-o", str(so), str(ROOT / "tests" / "denoise_oracle.c"), "-lm"],
                       check=True)
        self.rtnw = rtnw
        self.lib = C.CDLL(str(so))
        self.lib.rtnw_oracle_exp_neg.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        self.lib.rtnw_oracle_exp_neg.restype = None
        self.lib.rtnw_oracle_denoise.argtypes = [C.c_void_p, C.POINTER(rtnw.Aov), C.c_int32, C.c_int32, C.c_int32,
                                                 C.POINTER(rtnw.DenoiseParams), C.c_void_p]

    def exp_neg(self, x):
        x = np.ascontiguousarray(x, dtype=np.float32)
        out = np.empty_like(x)
        self.lib.rtnw_oracle_exp_neg(x.ctypes.data, x.size, out.ctypes.data)
        return out

    def denoise(self, sums, aov, ns, iterations=5, sigma_luminance=4.0, sigma_depth=1.0, normal_power_log2=7):
        """same signature and result as Context.denoise"""
        ny, nx, _ = sums.shape
        sums = np.ascontiguousarray(sums, dtype=np.float32)
        b = {k: np.ascontiguousarray(aov[k], dtype=np.int32 if k == "hits" else np.float32) for k in ("albedo", "normal", "depth", "hits")}
        feats = self.rtnw.Aov(b["albedo"].ctypes.data, b["normal"].ctypes.data, b["depth"].ctypes.data, b["hits"].ctypes.data, None)
        out = np.empty((ny, nx, 3), np.float32)
        dp = self.rtnw.DenoiseParams(iterations, sigma_luminance, sigma_depth, normal_power_log2)
        assert self.lib.rtnw_oracle_denoise(sums.ctypes.data, C.byref(feats), nx, ny, ns, C.byref(dp), out.ctypes.data) == 0
        return out


def synthetic_frame(nx, ny, ns, seed, hit_fraction=0.7, zero_albedo_fraction=0.05):
    """Random sums of ns samples: per pixel hits in 0..ns (misses, partial and full hits), noisy colour, albedo with some
    exact zeros, random normals (some summing to zero length) and depths."""
    rng = np.random.default_rng(seed)
    hits = np.where(rng.random((ny, nx)) < hit_fraction, rng.integers(1, ns + 1, (ny, nx)), 0).astype(np.int32)
    albedo = (rng.random((ny, nx, 3)) * ns).astype(np.float32)
    albedo[rng.random((ny, nx)) < zero_albedo_fraction] = 0
    color = (albedo * rng.gamma(2.0, 0.5, (ny, nx, 3))).astype(np.float32)
    n = rng.normal(size=(ny, nx, 3))
    n /= np.linalg.norm(n, axis=2, keepdims=True)
    n = n * hits[..., None]
    n[rng.random((ny, nx)) < 0.02] = 0  # normals that cancel out
    depth = (rng.uniform(1, 50, (ny, nx)) * hits).astype(np.float32)
    return color, dict(albedo=albedo, normal=n.astype(np.float32), depth=depth, hits=hits)
