"""Coarsen goldens: the reference's own reducers (xcube_resampling/coarsen.py, imported from
where make_golden.py's ``reference_dir`` finds it, with its stub recipe) on seeded windows.  Run through make_golden.py."""

import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def make_coarsen():
    import xcube_resampling.coarsen as C
    from xcube_resampling.constants import AGG_METHODS  # the table affine.py resolves method names with

    rng = np.random.default_rng(21)
    out = {}
    cases = []
    for name, dtype, f_j, f_i in [("f32_f2", np.float32, 2, 2), ("f32_f4", np.float32, 4, 4), ("f32_f8", np.float32, 8, 8),
                                  ("f32_f3x5", np.float32, 3, 5), ("f64_f4", np.float64, 4, 4), ("u8_f4", np.uint8, 4, 4),
                                  ("u8_f8", np.uint8, 8, 8), ("i16_f2", np.int16, 2, 2)]:
        h, w = 6 * f_j, 7 * f_i
        if np.issubdtype(dtype, np.floating):
            a = rng.random((h, w)).astype(dtype)
            a[rng.random((h, w)) < 0.06] = np.nan
            a[:f_j, :f_i] = np.nan
        else:
            coarse = rng.integers(0, 12, (-(-h // 7), -(-w // 7)))
            a = np.repeat(np.repeat(coarse, 7, axis=0), 7, axis=1)[:h, :w].astype(dtype)
            a[rng.random((h, w)) < 0.15] = 5
        block = a.reshape(h // f_j, f_j, w // f_i, f_i)
        out[f"{name}/input"] = a
        out[f"{name}/factors"] = np.array([f_j, f_i])
        import warnings
        for agg, fn in AGG_METHODS.items():
            if agg == "mode" and np.issubdtype(dtype, np.floating):
                continue
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                out[f"{name}/{agg}"] = np.asarray(fn(block, (1, 3)))
        cases.append(name)
    out["cases"] = np.array(cases)
    np.savez_compressed(os.path.join(HERE, "coarsen.npz"), **out)
    print("coarsen.npz:", cases)


def make_all():
    make_coarsen()
