"""Stored results of the original DPM-Solver implementation (LuChengTHU/dpm-solver: dpm_solver_pytorch.py and the
solver copies of its examples), so that the parity tests need nothing outside the repository.

    REF = refstore.Store(__file__)
    want = REF("case/key", lambda: <run the original on the test's inputs>)

The values live in tests/golden/reference/<test module>.json. A tensor is stored as a digest (128 bits of SHA-256)
of its bytes, NaNs and signed zeros canonicalised so that the digest compares like `torch.equal` with NaNs equal
positionally, with its dtype, shape and finiteness; a list (intermediate states, a trace of network calls) as one
digest of its items. The comparisons they feed are bit for bit, so the digest carries the same assertion. Each
item of a returned tuple is stored on its own. Where a test compares within a tolerance it needs values: `keep(t)`
stores a small tensor whole, `sample(t)` a fixed, seeded sample of SAMPLE elements and max |t| of the whole. An
exception the original raised is stored by its type and raised again on lookup.

Regenerating them needs the original (oracle/_ref, built by oracle/build_ref.py):

    DPM_RECORD_REFERENCE=<dir> python -m pytest tests -k <tests>

runs the original, and writes the updated files to <dir> (copy them to tests/golden/reference/)."""
import base64
import builtins
import hashlib
import json
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
RECORD = os.environ.get("DPM_RECORD_REFERENCE")


class Digest:
    """A stored tensor (or list) of the original, by its canonical bytes."""

    def __init__(self, d):
        self.digest, self.finite = d["d"], d["f"]
        self.dtype, self.shape = d.get("t"), tuple(d["s"]) if "s" in d else None

    def __repr__(self):
        return f"Digest({self.dtype}, {self.shape}, {self.digest})"


class keep:
    """Marks a tensor to be stored whole."""

    def __init__(self, t):
        self.t = t


SAMPLE = 256


def sample_index(numel):
    return torch.randperm(numel, generator=torch.Generator().manual_seed(0))[:SAMPLE]


class sample:
    """Marks a tensor to be stored as the elements at sample_index() and its max |x|."""

    def __init__(self, t):
        self.t = t


class Sample:
    """A stored sample of a tensor of the original."""

    def __init__(self, d):
        self.numel, self.absmax, self.finite, self.values = d["numel"], d["absmax"], d["f"], _decode(d["values"])

    def rel_err(self, have):
        """max |have - original| over the sampled elements / max |original| over all of them."""
        assert have.numel() == self.numel, (tuple(have.shape), self.numel)
        got = have.detach().cpu().reshape(-1)[sample_index(self.numel)].double()
        return float((got - self.values.double()).abs().max()) / max(self.absmax, 1e-30)


def _canonical_bytes(t):
    t = t.detach().cpu().contiguous()
    if t.is_floating_point():
        t = torch.where(torch.isnan(t), torch.full_like(t, float("nan")), t)
        t = torch.where(t == 0, torch.zeros_like(t), t)
    return t.reshape(-1).view(torch.uint8).numpy().tobytes()


def _hash(b):
    return hashlib.sha256(b).hexdigest()[:32]


def _tree_hash(v):
    """Digest of a tensor, a scalar or a (nested) list of them."""
    if torch.is_tensor(v):
        return _hash(f"{_dtype_name(v.dtype)}{list(v.shape)}".encode() + _canonical_bytes(v))
    if isinstance(v, (list, tuple)):
        return _hash(("L%d:" % len(v) + "".join(_tree_hash(u) for u in v)).encode())
    if isinstance(v, torch.dtype):
        v = str(v)
    return _hash(json.dumps(v).encode())


def _finite(v):
    if torch.is_tensor(v):
        return bool(torch.isfinite(v).all()) if v.is_floating_point() else True
    if isinstance(v, (list, tuple)):
        return all(_finite(u) for u in v)
    return True


def _encode_item(v):
    if isinstance(v, keep):
        t = v.t.detach().cpu().contiguous()
        return {"tensor": _dtype_name(t.dtype), "shape": list(t.shape),
                "b64": base64.b64encode(t.reshape(-1).view(torch.uint8).numpy().tobytes()).decode()}
    if isinstance(v, sample):
        t = v.t.detach().cpu().reshape(-1)
        return {"numel": t.numel(), "absmax": float(t.double().abs().max()), "f": _finite(t),
                "values": _encode_item(keep(t[sample_index(t.numel())].float()))}
    if torch.is_tensor(v):
        return {"d": _hash(_canonical_bytes(v)), "t": _dtype_name(v.dtype), "s": list(v.shape), "f": _finite(v)}
    if isinstance(v, (list, tuple)):
        return {"d": _tree_hash(v), "f": _finite(v)}
    if isinstance(v, dict):
        return {"dict": {k: _encode_item(u) for k, u in v.items()}}
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    raise TypeError(f"cannot store a {type(v).__name__}")


def _encode(v):
    if isinstance(v, (list, tuple)):
        return [_encode_item(u) for u in v]
    return _encode_item(v)


def _decode(v):
    if isinstance(v, list):
        return [_decode(u) for u in v]
    if isinstance(v, dict):
        if "d" in v:
            return Digest(v)
        if "numel" in v:
            return Sample(v)
        if "tensor" in v:
            dt = getattr(torch, v["tensor"])
            raw = np.frombuffer(base64.b64decode(v["b64"]), dtype=np.uint8).copy()
            return torch.from_numpy(raw).view(dt).reshape(v["shape"])
        if "dict" in v:
            return {k: _decode(u) for k, u in v["dict"].items()}
    return v


def _dtype_name(dt):
    return str(dt).replace("torch.", "")


def assert_same(have, want, msg=""):
    """`have` (a tensor, or a list such as intermediate states or a call trace, of the product) is bit-identical to
    `want` (a stored Digest or a tensor): same dtype, shape and values, NaNs equal positionally, +0 == -0."""
    if isinstance(want, Digest) and want.dtype is None:
        assert _tree_hash(have) == want.digest, f"{msg}: differs from the original"
    elif isinstance(want, Digest):
        assert _dtype_name(have.dtype) == want.dtype, (msg, _dtype_name(have.dtype), want)
        assert tuple(have.shape) == want.shape, (msg, tuple(have.shape), want)
        assert _hash(_canonical_bytes(have)) == want.digest, f"{msg}: values differ from the original ({want})"
    else:
        assert have.dtype == want.dtype and tuple(have.shape) == tuple(want.shape), (msg, have.dtype, want.dtype)
        np.testing.assert_array_equal(have.detach().cpu().float().numpy(), want.detach().cpu().float().numpy(), err_msg=str(msg))


def all_finite(v):
    if isinstance(v, (Digest, Sample)):
        return v.finite
    return bool(torch.isfinite(v).all())


def original(name="dpm_solver_pytorch", fresh=False):
    """The original module; only loaded while recording."""
    from oracle import ref_loader
    assert RECORD, "the original implementation is only run while recording (DPM_RECORD_REFERENCE)"
    return ref_loader.load(name, fresh=fresh)


class StoredError(Exception):
    pass


class Store:
    def __init__(self, test_file):
        self.name = os.path.splitext(os.path.basename(test_file))[0] + ".json"
        self._data = None

    def _path(self, root):
        return os.path.join(root, self.name)

    def data(self):
        if self._data is None:
            src = self._path(RECORD) if RECORD and os.path.exists(self._path(RECORD)) else self._path(GOLDEN)
            self._data = json.load(open(src)) if os.path.exists(src) else {}
        return self._data

    def __call__(self, key, compute):
        data = self.data()
        if RECORD:
            try:
                enc = _encode(compute())
            except Exception as e:
                enc = {"raises": type(e).__name__}
            data[key] = enc
            os.makedirs(RECORD, exist_ok=True)
            with open(self._path(RECORD), "w") as f:
                f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(data[k], separators=(',', ':'))}"
                                          for k in sorted(data)) + "\n}\n")
        if key not in data:
            raise KeyError(f"no stored result of the original for {key!r} in tests/golden/reference/{self.name}")
        enc = data[key]
        if isinstance(enc, dict) and "raises" in enc:
            exc = getattr(builtins, enc["raises"], None)
            if not (isinstance(exc, type) and issubclass(exc, Exception)):
                exc = StoredError
            raise exc(f"the original raised {enc['raises']}")
        return _decode(enc)
