"""Shared helpers for the parity tests."""
import json

import numpy as np


def load_meta(golden):
    return json.loads(bytes(golden["meta_json"]).decode())


def configure(ctx, case):
    """Apply a golden case's parameters to an mcb Context through the C ABI."""
    assert ctx.set_equation(case["eq"]) == 0
    assert ctx.set_grid_step(case["step"]) == case["M"]
    ctx.set_scaling(*case["scale"])
    ctx.set_surface_constant(case["iso"])
    for i in range(3):
        ctx.set_constraint(i, ">", 0.0, False)
    for i, (lhs, op, rhs) in enumerate(case.get("cons", [])):
        assert ctx.set_equation(lhs, slot=i + 1) == 0
        assert ctx.set_constraint(i, op, rhs, True) == 0


def same_bits(a, b):
    """fp32 arrays equal bit for bit, NaNs compared as a class."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    if a.shape != b.shape:
        return False
    eq = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    return bool(eq.all())


def rel_close(a, b, tol=1e-5):
    """north_star tolerance: |a-b| <= tol * max(1, |b|) (a purely relative test is ill-posed at 0)."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return bool(np.all(np.abs(a - b) <= tol * np.maximum(1.0, np.abs(b))))




def save_repeat_golden(path, arrays):
    """tests/golden/repeat_cases.npz.  Each case's soup is stored as the entries where it differs from its welded Poly_Data
    expanded (vertex_list[tri_list]: the weld keeps the first of points within 1e-6), and the archive is LZMA-compressed:
    the same bits in under a megabyte.  load_repeat_golden undoes both."""
    import io
    import zipfile
    out = {}
    for k, a in arrays.items():
        if k.endswith("/soup"):
            n = k[:-len("/soup")]
            rec = arrays[n + "/vertex_list"][arrays[n + "/tri_list"].astype(np.int64)].ravel()
            s = np.ascontiguousarray(a, np.float32).ravel()
            fix = np.flatnonzero((rec.view(np.uint32) != s.view(np.uint32)) & ~(np.isnan(rec) & np.isnan(s)))
            out[n + "/soup_fix_step"] = np.diff(fix, prepend=0).astype(np.uint32)  # gaps between the corrected entries
            out[n + "/soup_fix_value"] = s[fix]
        else:
            out[k] = a
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for k, a in out.items():
            b = io.BytesIO()
            np.save(b, a, allow_pickle=False)
            z.writestr(k + ".npy", b.getvalue())


def load_repeat_golden(path):
    """{name: array} of tests/golden/repeat_cases.npz, soups restored bit for bit (see save_repeat_golden)."""
    z = np.load(path, allow_pickle=False)
    out = {k: z[k] for k in z.files if "/soup_fix_" not in k}
    for k in z.files:
        if k.endswith("/soup_fix_step"):
            n = k[:-len("/soup_fix_step")]
            s = out[n + "/vertex_list"][out[n + "/tri_list"].astype(np.int64)].ravel()
            s[np.cumsum(z[k].astype(np.int64))] = z[n + "/soup_fix_value"]
            out[n + "/soup"] = s.reshape(-1, 3, 3)
    return out
