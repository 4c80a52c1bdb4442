"""Results of the original EasyAnimate project that the CPU tests compare with, stored under tests/golden/reference_cpu.*.

Each test passes `want(key, compute)` the call into the original project (oracle/ref_*.py) that produced its expected values.
Where the original project is installed, `EA_MINT_REFERENCE=1 python -m pytest tests -k <test>` runs that call and stores the
result; everywhere else `want` returns the stored result, so the comparison runs on every machine.

A tensor of integers, or of up to FULL floating-point elements, is stored whole; a larger one as SAMPLE elements at fixed
positions spread over all of it (`sample_index`) plus the SHA-256 of all of it.  CPU results change in their last bits with
the instruction set and the thread count that torch, MKL and oneDNN pick, so bit-for-bit equality is asserted on the CPU
configuration the results were minted on and a tolerance elsewhere.
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NPZ, META = os.path.join(GOLD, "reference_cpu.npz"), os.path.join(GOLD, "reference_cpu.json")
FULL, SAMPLE = 16384, 1024
MINT = os.environ.get("EA_MINT_REFERENCE") == "1"


def sample_index(n: int) -> np.ndarray:
    """SAMPLE distinct positions scattered over n elements (7919 is prime and exceeds every n // SAMPLE used here)."""
    return np.unique((np.arange(SAMPLE, dtype=np.int64) * 7919 + 17) % n)


class Stored:
    """A tensor of the original project's run: shape, dtype, SHA-256 of its bytes (floating point widened to float32 or
    float64), and its values at `index` (all of them when `index` is None)."""

    def __init__(self, meta, values):
        self.shape, self.dtype, self.sha = tuple(meta["shape"]), meta["dtype"], meta["sha256"]
        n = int(np.prod(self.shape))
        self.values = torch.from_numpy(values)
        self.index = None if values.size == n else torch.from_numpy(sample_index(n))

    def pick(self, got):
        flat = _as_torch(got).reshape(-1).to(self.values.dtype)
        return flat if self.index is None else flat[self.index]


def cpu_config() -> str:
    model = ""
    try:
        with open("/proc/cpuinfo") as f:
            model = next((ln.split(":", 1)[1].strip() for ln in f if ln.startswith("model name")), "")
    except OSError:
        pass
    return f"torch {torch.__version__} | {torch.backends.cpu.get_cpu_capability()} | {torch.get_num_threads()} threads | {model}"


def _as_torch(x):
    return torch.from_numpy(np.asarray(x)) if not torch.is_tensor(x) else x.detach().cpu()


def _wide(x):
    x = _as_torch(x)
    if not x.is_floating_point():
        return x.long()
    return x.double() if x.dtype == torch.float64 else x.float()


def _sha(x) -> str:
    return hashlib.sha256(_wide(x).contiguous().numpy().tobytes()).hexdigest()


def _load():
    meta = json.load(open(META)) if os.path.exists(META) else {"minted_on": None, "entries": {}}
    arrays = dict(np.load(NPZ)) if os.path.exists(NPZ) else {}
    return meta, arrays


def _is_array(v):
    return torch.is_tensor(v) or isinstance(v, np.ndarray)


def _plain(v):
    if isinstance(v, dict):
        return all(_plain(x) for x in v.values())
    if isinstance(v, (list, tuple)):
        return all(_plain(x) for x in v)
    return not _is_array(v)


def _encode(key, value, arrays):
    if _is_array(value):
        x = _wide(value)
        flat = x.reshape(-1).numpy()
        if x.is_floating_point() and x.numel() > FULL:
            flat = flat[sample_index(x.numel())]
        arrays[key] = flat if x.is_floating_point() else flat.astype(np.int32)
        return {"tensor": key, "shape": list(x.shape), "dtype": str(_as_torch(value).dtype), "sha256": _sha(x)}
    if _plain(value):
        return {"json": value}
    if isinstance(value, dict):
        return {"dict": {k: _encode(f"{key}/{k}", v, arrays) for k, v in value.items()}}
    if isinstance(value, (list, tuple)):
        return {"list": [_encode(f"{key}/{i}", v, arrays) for i, v in enumerate(value)]}
    return {"json": value}


def _decode(node, arrays):
    if "tensor" in node:
        return Stored(node, arrays[node["tensor"]])
    if "dict" in node:
        return {k: _decode(v, arrays) for k, v in node["dict"].items()}
    if "list" in node:
        return [_decode(v, arrays) for v in node["list"]]
    return node["json"]


def want(key, compute):
    """The original project's result for `key`: tensors come back as `Stored`, tuples as lists, everything else as JSON."""
    meta, arrays = _load()
    if MINT:
        for k in [k for k in arrays if k == key or k.startswith(key + "/")]:
            del arrays[k]
        meta["entries"][key] = _encode(key, compute(), arrays)
        meta["minted_on"] = cpu_config()
        np.savez_compressed(NPZ, **arrays)
        with open(META, "w") as f:
            json.dump(meta, f, indent=1, sort_keys=True)
        meta, arrays = _load()  # what the tests elsewhere will read
    if key not in meta["entries"]:
        raise KeyError(f"{key}: no stored result of the original project (mint it with EA_MINT_REFERENCE=1 where it is installed)")
    return _decode(meta["entries"][key], arrays)


def minted_here() -> bool:
    return _load()[0]["minted_on"] == cpu_config()


def diff(got, ref: Stored):
    """(max |got - ref|, ||got - ref|| / ||ref||) over the stored elements."""
    a, b = ref.pick(got), ref.values
    return (a - b).abs().max().item(), ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def assert_equal(got, ref: Stored, rel: float):
    """Bit for bit on the CPU configuration the result was minted on, and integers everywhere; floating point elsewhere within
    `rel` (norm of the difference over the norm of the result) on the stored elements."""
    assert tuple(_as_torch(got).shape) == ref.shape and str(_as_torch(got).dtype) == ref.dtype, (tuple(got.shape), ref.shape)
    if minted_here() or not ref.values.is_floating_point():
        assert _sha(got) == ref.sha, diff(got, ref)
    else:
        assert diff(got, ref)[1] <= rel, diff(got, ref)


def assert_close(got, ref: Stored, atol: float, rtol: float = 0.0, elsewhere_rel: float | None = None):
    """torch.testing.assert_close on the stored elements; with `elsewhere_rel`, that is the criterion on a CPU configuration
    other than the one the result was minted on (see assert_equal)."""
    assert tuple(_as_torch(got).shape) == ref.shape, (tuple(got.shape), ref.shape)
    if elsewhere_rel is not None and not minted_here():
        assert diff(got, ref)[1] <= elsewhere_rel, diff(got, ref)
    else:
        torch.testing.assert_close(ref.pick(got), ref.values, atol=atol, rtol=rtol)
