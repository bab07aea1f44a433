"""Generate tests/golden/reproject.npz by running the REFERENCE's ``_reproject_block``.

Needs the reference package where make_golden.py's ``reference_dir`` finds it; see make_golden.py for the stub recipe.
Inputs are seeded source-CRS coordinates of the target pixels of one tile plus a source window;
outputs are what ``xcube_resampling.reproject._reproject_block`` (reproject.py:268-335) returns,
for every interpolation method and a spread of dtypes.

    python tests/golden/make_golden_reproject.py
"""

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden import install_reference  # noqa: E402


def main():
    install_reference()
    from xcube_resampling import reproject as P

    rng = np.random.default_rng(42)
    out = {}
    cases = []
    # (name, window w/h, target tile w/h, x_res, y_res, x origin, y origin)
    specs = [
        ("geo", 40, 36, 24, 20, 0.0001, 0.0001, 8.1234567, 9.7654321),
        ("utm", 33, 47, 17, 29, 10.0, 10.0, 399960.0, 5900040.0),
        ("coarse", 12, 10, 31, 27, 0.25, 0.5, -12.3, 61.7),
    ]
    for name, ww, wh, tw, th, xres, yres, xo, yo in specs:
        x_coord = (xo + xres * np.arange(ww)).astype(np.float32).reshape(ww, 1, 1)
        y_coord = (yo - yres * np.arange(wh)).astype(np.float32).reshape(wh, 1, 1)
        # coordinates strictly inside the window so that every tap exists; some exactly on pixel centres
        fx = rng.uniform(0.0, ww - 1.001, size=(th, tw))
        fy = rng.uniform(0.0, wh - 1.001, size=(th, tw))
        fx[0, :5] = np.arange(5)
        fy[0, :5] = np.arange(5)
        fx[1, :4] = np.arange(4) + 0.5
        fy[1, :4] = np.arange(4) + 0.5
        xx = np.float64(x_coord[0, 0, 0]) + fx * xres
        yy = np.float64(y_coord[0, 0, 0]) - fy * yres
        out[f"{name}/xx"], out[f"{name}/yy"] = xx, yy
        out[f"{name}/x_coord"], out[f"{name}/y_coord"] = x_coord[:, 0, 0], y_coord[:, 0, 0]
        out[f"{name}/res"] = np.array([xres, yres])
        data = {
            "f32": rng.normal(size=(3, wh, ww)).astype(np.float32),
            "f64": rng.normal(size=(2, wh, ww)),
            "u8": rng.integers(0, 256, size=(2, wh, ww), dtype=np.uint8),
            "i16": rng.integers(-30000, 30000, size=(2, wh, ww)).astype(np.int16),
            "i32": rng.integers(-2**31, 2**31 - 1, size=(1, wh, ww)).astype(np.int32),
            "i64": rng.integers(-1000, 1000, size=(1, wh, ww)).astype(np.int64),
        }
        data["f32"][0, 3, 4] = np.nan
        for dn, arr in data.items():
            out[f"{name}/src_{dn}"] = arr
            for method in ("nearest", "bilinear", "triangular"):
                with np.errstate(all="ignore"):
                    res = P._reproject_block(xx, yy, arr, x_coord, y_coord, xres, yres, method)
                out[f"{name}/out_{dn}_{method}"] = res
        cases.append(name)
    out["cases"] = np.array(cases)
    path = os.path.join(HERE, "reproject.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: (v.shape, str(v.dtype)) for k, v in out.items() if "out_" in k and k.startswith("geo")})


if __name__ == "__main__":
    main()
