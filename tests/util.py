import hashlib
import json
import os

import numpy as np
import torch


def rel_err(a, b):
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def assert_close(a, b, tol, name):
    assert tuple(a.shape) == tuple(b.shape), "%s: shape %s vs %s" % (name, tuple(a.shape), tuple(b.shape))
    a64 = torch.as_tensor(a).detach().double().cpu()
    assert torch.isfinite(a64).all(), "%s: non-finite values" % name
    e = rel_err(a, b)
    assert e <= tol, "%s: max-abs error / max-abs reference = %.3e > %.1e" % (name, e, tol)
    return e


def rms_err(a, b):
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt().clamp_min(1e-30)).item()


def gen(seed, *shape, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


# ---- stored outputs of the reference's own CUDA kernels (tests/golden/ref_*.npz, make_golden_ref_kernels.py) ----
def _canonical(t):
    """Values as a contiguous numpy array: integers as int64, floats as float64 (exact for fp32), so that a digest does
    not depend on the integer width or device a kernel returns."""
    a = torch.as_tensor(t).detach().cpu()
    return np.ascontiguousarray(a.to(torch.float64 if a.is_floating_point() else torch.int64).numpy())


def digest(t):
    return hashlib.sha256(_canonical(t).tobytes()).hexdigest()


def record(store, key, t, sample):
    """Keep what a test needs to compare against the reference output `t`: its shape, SHA-256 (for bit-exact checks),
    max-abs and rms (the denominators of rel_err / rms_err over the whole tensor) and its values at `sample` fixed,
    seeded positions -- drawn among its non-zero entries when there are enough of them, every position when small."""
    flat = _canonical(t).ravel()
    if flat.size <= sample:
        pos = np.arange(flat.size)
    else:
        nz = np.flatnonzero(flat)
        pos = np.sort(np.random.RandomState(0).choice(nz if nz.size >= sample else flat.size, sample, replace=False))
    store[key] = {"shape": list(t.shape), "sha256": digest(t), "absmax": float(np.abs(flat).max()) if flat.size else 0.0,
                  "rms": float(np.sqrt(np.mean(np.square(flat)))) if flat.size else 0.0, "pos": pos, "val": flat[pos]}


def save_golden(path, store):
    """One .npz per test module: a JSON index (key -> shape, digest, max-abs, rms, slice) and the sampled positions
    and values of every output, concatenated."""
    meta, n = {}, 0
    for key, r in store.items():
        meta[key] = {k: r[k] for k in ("shape", "sha256", "absmax", "rms")}
        meta[key].update(offset=n, count=len(r["pos"]))
        n += len(r["pos"])
    np.savez_compressed(path, meta=np.array(json.dumps(meta, sort_keys=True)),
                        pos=np.concatenate([r["pos"] for r in store.values()]).astype(np.int32),
                        val=np.concatenate([r["val"].astype(np.float64) for r in store.values()]))


class RefGolden:
    """Reference-kernel outputs stored in tests/golden/<name>.npz (save_golden), compared against by key."""

    def __init__(self, name):
        self.path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz")
        self._meta = None

    def keys(self):
        if self._meta is None:
            z = np.load(self.path)
            self._meta, self._pos, self._val = json.loads(str(z["meta"])), z["pos"], z["val"]
        return self._meta.keys()

    def _entry(self, key, t, name):
        self.keys()
        m = self._meta[key]
        assert tuple(t.shape) == tuple(m["shape"]), "%s: shape %s vs reference %s" % (name, tuple(t.shape), tuple(m["shape"]))
        sl = slice(m["offset"], m["offset"] + m["count"])
        return m, self._pos[sl], self._val[sl]

    def exact(self, key, t, name):
        """bit-exact: same values as the reference output everywhere (SHA-256 of the whole tensor)"""
        m, pos, val = self._entry(key, t, name)
        if digest(t) != m["sha256"]:
            got = _canonical(t).ravel()[pos]
            raise AssertionError("%s differs from the reference kernel (%d of %d sampled values differ)" % (
                name, int((got != val).sum()), got.size))

    def _sampled(self, key, t, name):
        m, pos, val = self._entry(key, t, name)
        return m, torch.from_numpy(_canonical(t).ravel()[pos]), torch.from_numpy(val)

    def close(self, key, t, tol, name):
        """max-abs error at the stored positions / max-abs of the whole reference output <= tol"""
        assert np.isfinite(_canonical(t)).all(), "%s: non-finite values" % name
        m, got, want = self._sampled(key, t, name)
        e = (got - want).abs().max().item() / max(m["absmax"], 1e-30) if want.numel() else 0.0
        assert e <= tol, "%s: max-abs error / max-abs reference = %.3e > %.1e (%d sampled positions)" % (name, e, tol, want.numel())
        return e

    def rms(self, key, t):
        """rms error at the stored positions / rms of the whole reference output"""
        m, got, want = self._sampled(key, t, key)
        return ((got - want).pow(2).mean().sqrt() / max(m["rms"], 1e-30)).item()
