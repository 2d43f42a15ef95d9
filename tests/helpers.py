"""Shared helpers of the parity tests."""
import hashlib
import os

import numpy as np

LAYERS = ["elevation", "variance", "is_valid", "traversability", "time", "upper_bound", "is_upper_bound"]
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def digest(a):
    """sha256 of an array's dtype, shape and bytes: a stored exact-equality check against the reference's output."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def load_golden(name):
    """tests/golden/<name>.npz as a dict of arrays (0-d entries as Python scalars / str)."""
    with np.load(os.path.join(GOLD, name + ".npz")) as z:
        return {k: (z[k].item() if z[k].ndim == 0 else z[k]) for k in z.files}


def compare_state(eng_map, eng_normal, om, trav_tol=2e-6, exact_layers=(0, 1, 2, 4, 5, 6), label=""):
    """CUDA engine state vs oracle state.  By construction (fixed-point accumulation, pinned
    contractions) every layer except traversability is expected BIT-identical; traversability goes
    through expf (CUDA vs glibc) and is compared to `trav_tol`."""
    for li in exact_layers:
        a, b = eng_map[li], om.elevation_map[li]
        if not np.array_equal(a, b):
            bad = np.argwhere(a != b)
            r, c = bad[0]
            raise AssertionError(f"{label} layer {LAYERS[li]}: {len(bad)} cells differ, first at ({r},{c}): "
                                 f"engine {a[r, c]!r} oracle {b[r, c]!r}; max abs diff {np.nanmax(np.abs(a - b))}")
    d = np.abs(eng_map[3] - om.elevation_map[3])
    assert d.max() <= trav_tol, f"{label} traversability max diff {d.max()}"
    assert np.array_equal(eng_normal, om.normal_map), f"{label} normals differ: max {np.abs(eng_normal - om.normal_map).max()}"
