"""Shared test helpers (CPU-only imports at module level)."""
import copy
import hashlib
import os
from pathlib import Path

import numpy as np
import torch

REL_TOL = 1e-3  # BASELINE.json north_star: grouped features / MLP outputs within 1e-3 relative
RECORDED = Path(__file__).resolve().parent / "golden" / "recorded_b200.npz"
_recorded_cache = {}


def rel_err(got, want):
    """max |got - want| relative to the largest magnitude of the reference tensor."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    scale = max(np.abs(want).max(), 1e-30)
    return float(np.abs(got - want).max() / scale)


def assert_close(got, want, tol=REL_TOL, what=""):
    assert np.asarray(got).shape == np.asarray(want).shape, f"{what}: shape {np.asarray(got).shape} vs {np.asarray(want).shape}"
    e = rel_err(got, want)
    assert e <= tol, f"{what}: relative error {e:.3e} > {tol:.1e}"


def small_sa_cfg(npoints=(512, 128, 64, 32)):
    """IA-SSD KITTI SA_CONFIG (same radii / nsample / widths) with fewer points, for second-scale tests."""
    from spsnet_b200.backbone import KITTI_IASSD_SA_CONFIG, Cfg

    c = copy.deepcopy(KITTI_IASSD_SA_CONFIG)
    c["NPOINT_LIST"] = [[npoints[0]], [npoints[1]], [npoints[2]], [npoints[3]], [-1], [npoints[3]]]
    return Cfg({"SA_CONFIG": c})


def make_backbone(cfg, input_channels=4, num_class=3, seed=0, cls=None):
    from spsnet_b200 import backbone as bb

    torch.manual_seed(seed)
    net = (cls or bb.IASSD_Backbone)(cfg, num_class=num_class, input_channels=input_channels)
    bb.randomize_bn_stats(net, seed=seed)
    return net.eval()


def _np(x):
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().numpy()
    return np.ascontiguousarray(x)


def _sample(a, k):
    """A fixed sample of k elements of a flattened array (legacy RandomState: its stream is frozen across NumPy versions)."""
    flat = a.reshape(-1)
    if flat.size <= k:
        return flat
    return flat[np.sort(np.random.RandomState(flat.size % (1 << 32)).choice(flat.size, k, replace=False))]


class Recorded:
    """Outputs of this implementation recorded on a B200 into tests/golden/recorded_b200.npz, compared with what the code
    computes now.  The upstream reference build (oracle/_ref) is not part of the repository: the tests that run it side by side
    where it is installed also compare against these recordings, so a checkout without it still pins the same computations.
    Arrays that must match bit for bit are kept as a SHA-256 of their bytes; float arrays as a fixed sample plus the largest
    magnitude of the whole array (the range-relative error of `rel_err`, evaluated on the sample).

    Recording: `SPSK_RECORD=DIR python -m pytest -m gpu tests -k <tests>` on a B200 writes DIR/recorded_b200.npz (the
    comparisons then pass trivially); copy it over tests/golden/recorded_b200.npz."""

    def __init__(self, key):
        self.key = key
        self.record_dir = os.environ.get("SPSK_RECORD")
        self.new = {}
        if not self.record_dir and "data" not in _recorded_cache:
            _recorded_cache["data"] = dict(np.load(RECORDED)) if RECORDED.exists() else {}

    def _put(self, name, field, value):
        self.new.setdefault(f"{self.key}|{name}|{field}", np.asarray(value))   # the first call records

    def _get(self, name, field):
        k = f"{self.key}|{name}|{field}"
        if self.record_dir:
            return self.new[k]
        data = _recorded_cache["data"]
        assert k in data, f"{RECORDED.name} holds no `{k}` (record it, see tests/helpers.py::Recorded)"
        return data[k]

    def save(self):
        if not (self.record_dir and self.new):
            return
        out = Path(self.record_dir) / RECORDED.name
        out.parent.mkdir(parents=True, exist_ok=True)
        data = dict(np.load(out)) if out.exists() else {}
        data.update(self.new)
        np.savez_compressed(out, **data)

    def same(self, name, got):
        """Whether `got` equals the recorded array bit for bit (shape, dtype and bytes)."""
        a = _np(got)
        sig = f"{a.dtype.str}{list(a.shape)}:" + hashlib.sha256(a.tobytes()).hexdigest()
        if self.record_dir:
            self._put(name, "sha", sig)
        return sig == str(self._get(name, "sha"))

    def exact(self, name, got):
        assert self.same(name, got), f"{name}: differs from the recorded output"

    def err(self, name, got, k=512):
        """Range-relative error of `got` against the recorded array, on the recorded sample (k elements when recorded)."""
        a = _np(got).astype(np.float32)
        if self.record_dir:   # one float32 array: largest magnitude, rank, shape, sample
            absmax = np.abs(a).max() if a.size else 0.0
            self._put(name, "f", np.concatenate([[absmax, a.ndim], a.shape, _sample(a, k)]).astype(np.float32))
        f = self._get(name, "f")
        ndim = int(f[1])
        shape, want = tuple(int(x) for x in f[2:2 + ndim]), f[2 + ndim:].astype(np.float64)
        assert a.shape == shape, f"{name}: shape {a.shape} vs recorded {shape}"
        if not a.size:
            return 0.0
        return float(np.abs(_sample(a, len(want)).astype(np.float64) - want).max() / max(float(f[0]), 1e-30))

    def close(self, name, got, tol=REL_TOL, k=512):
        e = self.err(name, got, k)
        assert e <= tol, f"{name}: relative error {e:.3e} > {tol:.1e} against the recorded output"
        return e


def check_backbone_vs_recorded(rec, out, tol=REL_TOL):
    """A backbone forward against a recorded forward of the same weights and batch: every layer's sampled points bit-exact
    (D-FPS and score-based layers alike), every layer's features and class logits, the centres, their offsets and the centre
    features within `tol`.  A score-based layer picks by the last bits of the confidence logits, so a change of summation
    order that flips a near-tie fails here loudly (the teacher-forced check of oracle/parity.py, against the live reference,
    is the comparison that tolerates it)."""
    for i in range(1, len(out["encoder_xyz"])):
        rec.exact(f"encoder_xyz{i}", out["encoder_xyz"][i])
        f = out["encoder_features"][i]
        if f is not None and f.numel():
            rec.close(f"encoder_features{i}", f, tol)
    for i in range(len(out["sa_ins_preds"])):
        p = out["sa_ins_preds"][i]
        if isinstance(p, torch.Tensor) and p.numel():
            rec.close(f"logits{i}", p[..., 1:], tol)   # column 0 is the batch index
    for k in ("centers_features", "centers", "ctr_offsets"):
        rec.close(k, out[k], tol)
