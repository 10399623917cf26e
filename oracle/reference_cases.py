"""Seeded input cases for the differential tests against the reference's own functions.

`oracle.make_golden.gen_reference_cases` runs the reference on these inputs and stores its answers (long outputs as sha256
fingerprints) in tests/golden/reference_cases.json; tests/test_reference_live_cpu.py and tests/test_compare_cpu.py rebuild the same inputs
from the same seeds and compare this project's functions with the stored answers.  `digest()` fingerprints every case
list, so a generator that drifts from the one the answers were made with fails loudly instead of comparing unrelated data.

The generators draw from the ranges the properties are stated over (frame rates, spans, 0/1 tracks, nested values) and
mix in the boundary values of each range.

Test infrastructure only (see oracle/__init__.py).
"""

from __future__ import annotations

import hashlib

import attrs
import numpy as np

N_CASES = 150
N_TUBE_CASES = 60


def _canon(v):
    if isinstance(v, np.ndarray):
        return ("ndarray", v.dtype.str, v.shape, v.tobytes().hex())
    if isinstance(v, (list, tuple)):
        return (type(v).__name__, [_canon(x) for x in v])
    if isinstance(v, dict):
        return ("dict", [(repr(k), _canon(x)) for k, x in v.items()])
    if attrs.has(type(v)):
        return (type(v).__name__, _canon(attrs.asdict(v, recurse=False)))
    return (type(v).__name__, float.hex(v) if isinstance(v, float) else repr(v))


def digest(cases) -> str:
    return hashlib.sha256(repr(_canon(cases)).encode()).hexdigest()


def _float(rng, lo: float, hi: float) -> float:
    """Uniform in [lo, hi], with the ends, round values and tiny values over-represented."""
    u = rng.random()
    if u < 0.08:
        return float(lo)
    if u < 0.16:
        return float(hi)
    if u < 0.3:
        return float(min(hi, max(lo, round(rng.uniform(lo, hi)))))
    if u < 0.36:
        return float(min(hi, lo + 1e-6 * rng.random()))
    return float(rng.uniform(lo, hi))


def _text(rng, max_size: int) -> str:
    alphabet = "abcxyz019_-/:. " + "é中\U0001f600\x00"
    return "".join(alphabet[i] for i in rng.integers(0, len(alphabet), size=int(rng.integers(0, max_size + 1))))


def timestamp_cases() -> list[dict]:
    """Sorted float32 presentation times: constant or variable frame rate, optional dropped frames, optional start offset;
    with a sampling rate, endpoint and dedup flag each."""
    rng = np.random.default_rng(1)
    out = []
    for _ in range(N_CASES):
        n = int(rng.integers(2, 401))
        fps = float(rng.choice([10.0, 23.976, 24.0, 25.0, 29.97, 30.0, 50.0, 59.94, 60.0]))
        t = np.arange(n, dtype=np.float64) / fps + float(rng.choice([0.0, 0.0, 0.033, 1.5]))
        if rng.random() < 0.5:
            t = t + np.cumsum(rng.uniform(0.0, 0.02, size=n))  # variable frame rate
        if rng.random() < 0.5 and n > 10:
            keep = np.ones(n, bool)
            keep[rng.integers(1, n - 1, size=int(rng.integers(0, n // 5 + 1)))] = False  # dropped frames
            t = t[keep]
        out.append({"ts": np.sort(t.astype(np.float32)), "rate": float(rng.choice([0.5, 1.0, 2.0, 3.0, 4.0, 7.5, 8.0, 16.0, 30.0, 100.0])),
                    "endpoint": bool(rng.random() < 0.5), "dedup": bool(rng.random() < 0.5)})  # fmt: skip
    return out


def closest_targets(ts: np.ndarray) -> np.ndarray:
    return np.linspace(float(ts[0]) - 0.3, float(ts[-1]) + 0.3, 57).astype(np.float32)


def fixed_stride_cases() -> list[dict]:
    """Seeded cases, then windows whose length equals min_len exactly (full windows, and the last window cut at the end)."""
    rng = np.random.default_rng(2)
    cases = [{"end": _float(rng, 0.0, 400.0), "clip_len": _float(rng, 0.1, 60.0), "stride": _float(rng, 0.05, 90.0), "min_len": _float(rng, 0.0, 30.0),
              "session": _text(rng, 12)} for _ in range(N_CASES)]  # fmt: skip
    for end, clip_len, stride, min_len in ((30.0, 10.0, 10.0, 10.0), (25.0, 10.0, 10.0, 5.0), (12.5, 4.0, 4.0, 0.5), (7.0, 2.5, 2.0, 1.0)):
        cases.append({"end": end, "clip_len": clip_len, "stride": stride, "min_len": min_len, "session": "boundary"})
    return cases


def values_sha256(a) -> str:
    """Fingerprint of an array's shape and values (as float64: an int32 and an int64 array of equal values match, like np.array_equal)."""
    a = np.asarray(a)
    return hashlib.sha256(repr(a.shape).encode() + np.ascontiguousarray(a, dtype=np.float64).tobytes()).hexdigest()


def spans_sha256(spans) -> str:
    """Fingerprint of a span list, bit for bit (float.hex of both ends): small strides give thousands of spans per case."""
    return hashlib.sha256("\n".join(f"{float.hex(a)} {float.hex(b)}" for a, b in spans).encode()).hexdigest()


def uuids_sha256(uuids) -> str:
    """Fingerprint of a uuid list (the uuids are hashes themselves: stored verbatim they would not compress)."""
    return hashlib.sha256("\n".join(str(u) for u in uuids).encode()).hexdigest()


def chunk_cases() -> list[dict]:
    rng = np.random.default_rng(3)
    out = []
    for _ in range(N_CASES):
        durs = [_float(rng, 0.0, 40.0) for _ in range(int(rng.integers(0, 121)))]
        out.append({"spans": [(float(i), float(i) + d) for i, d in enumerate(durs)], "per_chunk": int(rng.integers(1, 41))})
    return out


def chunk_size(span) -> int:
    return int(span[1] - span[0])


def _leaf(rng):
    k = int(rng.integers(0, 7))
    if k == 0:
        return int(rng.integers(-5, 6))
    if k == 1:
        return _float(rng, -2.0, 2.0)
    if k == 2:
        return _text(rng, 3)
    if k == 3:
        return bool(rng.random() < 0.5)
    if k == 4:
        return None
    if k == 5:
        v = [float(np.float32(_float(rng, -3.0, 3.0))) if rng.random() < 0.8 else float("nan") for _ in range(int(rng.integers(0, 6)))]
        return np.array(v, dtype=str(rng.choice(["float32", "float64"])))
    return np.array(rng.integers(0, 256, size=int(rng.integers(0, 6))), dtype=np.uint8)


def _tree(rng, depth: int = 0):
    """Leaves, lists (up to 4), pairs and dicts (keys "a", "b", "c", 1) nested up to three levels."""
    k = int(rng.integers(0, 4)) if depth < 3 else 0
    if k == 0:
        return _leaf(rng)
    if k == 1:
        return [_tree(rng, depth + 1) for _ in range(int(rng.integers(0, 5)))]
    if k == 2:
        return (_tree(rng, depth + 1), _tree(rng, depth + 1))
    keys = ["a", "b", "c", 1]
    return {keys[i]: _tree(rng, depth + 1) for i in rng.permutation(4)[: int(rng.integers(0, 4))]}


def compare_cases() -> list[dict]:
    """Golden / candidate value trees; every third candidate is the golden tree with some leaves perturbed, so that both
    matching and differing subtrees occur."""
    rng = np.random.default_rng(4)
    out = []
    for i in range(N_CASES):
        golden = _tree(rng)
        candidate = _perturb(rng, golden) if i % 3 == 0 else _tree(rng)
        out.append({"golden": golden, "candidate": candidate, "atol": float(rng.choice([0.0, 1e-3, 0.5, 2.0]))})
    return out


def _perturb(rng, v):
    if isinstance(v, list):
        return [_perturb(rng, x) for x in v]
    if isinstance(v, tuple):
        return tuple(_perturb(rng, x) for x in v)
    if isinstance(v, dict):
        return {k: _perturb(rng, x) for k, x in v.items()}
    if isinstance(v, np.ndarray) and v.dtype.kind == "f" and v.size and rng.random() < 0.5:
        return (v + np.asarray(rng.choice([5e-4, 0.3, 1.5]), dtype=v.dtype)).astype(v.dtype)
    if isinstance(v, float) and rng.random() < 0.5:
        return v + float(rng.choice([5e-4, 0.3, 1.5]))
    return v


def shot_cases() -> list[dict]:
    rng = np.random.default_rng(5)
    out = []
    for _ in range(N_CASES):
        n = int(rng.integers(1, 601))
        out.append({"track": (rng.random(n) < 0.2).astype(np.uint8), "entire": bool(rng.random() < 0.5),
                    "min_len": None if rng.random() < 0.5 else int(rng.integers(1, 81)), "max_len": None if rng.random() < 0.5 else int(rng.integers(1, 201)),
                    "mode": str(rng.choice(["truncate", "stride"])), "crop": None if rng.random() < 0.5 else int(rng.integers(0, 21))})  # fmt: skip
    return out


def tube_cases() -> list[dict]:
    """Source sizes (1..260 px), target sizes (1..72 px) and frame counts (8..19) for the InternVideo2 tube formulation."""
    rng = np.random.default_rng(6)
    out = []
    for _ in range(N_TUBE_CASES):
        h, w = (int(rng.choice([1, 2, 260])) if rng.random() < 0.15 else int(rng.integers(1, 261)) for _ in range(2))
        th, tw = (int(rng.choice([1, 72])) if rng.random() < 0.15 else int(rng.integers(1, 73)) for _ in range(2))
        if rng.random() < 0.15:
            th, tw = h // 2 or 1, w // 2 or 1  # the exact-2x INTER_AREA reroute
        if rng.random() < 0.1:
            th, tw = min(h, 72), min(w, 72)
        out.append({"h": h, "w": w, "th": th, "tw": tw, "n": int(rng.integers(8, 20)), "seed": int(rng.integers(0, 2**31 - 1))})
    return out


def tube_frames(case: dict) -> list[np.ndarray]:
    rng = np.random.default_rng(case["seed"])
    return [rng.integers(0, 256, size=(case["h"], case["w"], 3), dtype=np.uint8) for _ in range(case["n"])]


def tube_sha256(tube: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(tube).tobytes()).hexdigest()


@attrs.define
class Leaf:
    score: float
    vec: np.ndarray
    tags: dict


def comparator_table() -> list[tuple]:
    """(name, golden, candidate, atol): one case per rule of the stage-output comparator."""
    a = np.arange(6, dtype=np.float32).reshape(2, 3)
    nan = np.array([1.0, np.nan, 3.0], dtype=np.float32)
    return [
        ("equal", {"a": a, "b": [1, "x", (2, 3)]}, {"a": a.copy(), "b": [1, "x", (2, 3)]}, 0.0),
        ("within", a, a + np.float32(9e-4), 1e-3),
        ("beyond", a, a + np.float32(2e-3), 1e-3),
        ("rtol_zero", np.array([1e6], np.float32), np.array([1e6 + 1], np.float32), 0.5),  # allclose's default rtol would pass this
        ("unsigned", np.array([0, 255], np.uint8), np.array([1, 0], np.uint8), 0.0),
        ("nan_match", nan, nan.copy(), 0.0),
        ("nan_one_side", nan, np.array([1.0, 2.0, 3.0], np.float32), 0.0),
        ("nan_plus_diff", nan, np.array([1.5, np.nan, 3.0], np.float32), 0.1),
        ("shape", a, a.T.copy(), 1.0),
        ("dtype_ok", a, a.astype(np.float64), 0.0),  # both ndarray: dtypes may differ
        ("type", [1, 2], (1, 2), 0.0),
        ("int_float", {"k": 1}, {"k": 1.0}, 0.0),
        ("keys", {"a": 1, "b": 2}, {"a": 1, "c": 2}, 0.0),
        ("length", [1, 2, 3], [1, 2], 0.0),
        ("strings", np.array(["a", "b"]), np.array(["a", "c"]), 0.0),
        ("bytes", b"abc", b"abd", 0.0),
        ("attrs", Leaf(1.0, a, {"x": [a]}), Leaf(1.5, a + 1, {"x": [a * 2]}), 0.25),
        ("nested_path", {"v": [{"w": a}]}, {"v": [{"w": a + 1}]}, 0.0),
        ("empty", [], [], 0.0),
    ]


def diff_key(d) -> tuple:
    """What the tests compare of one FieldDiff."""
    return (d.field, d.detail, d.max_diff_observed, d.shape_mismatch)
