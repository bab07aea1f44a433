"""affine_transform_dataset / resample_dataset: regular grid -> regular grid, same CRS.

Same entry points, arguments and errors as the reference's
``xcube_resampling/affine.py:52-362``.  The per-variable work -- scipy's
``affine_transform`` (order 0/1, ``mode="constant"``) through dask-image, then
``dask.array.coarsen`` with the ``coarsen.py`` reducers when down-scaling -- is
one fused kernel of ``libxrs.so`` (``xrs_affine``, K4+K5).
"""

from __future__ import annotations

import math
from collections.abc import Iterable

import numpy as np
import torch

from . import _dev
from ._lib import check, load
from .constants import AGG_CODES, DTYPE_CODES
from .dataset import DataArray, Dataset, from_any, to_like
from .gridmapping import GridMapping
from .utils import (
    _can_apply_affine_transform,
    _get_agg_method,
    _get_fill_value,
    _get_interp_method_int,
    _get_recover_nan,
    _select_variables,
    normalize_grid_mapping,
)

_INT64_OUT_AGGS = ("mode", "count")
_ORDER_ERROR = (
    "interp_methods must be one of 0, 1, 'nearest', 'bilinear'. "
    "Higher order is not supported for 3D arrays in affine transforms, "
    "as it causes unintended blending across the non-spatial (e.g., time) "
    "dimension."
)


def _np_dtype(t: torch.Tensor) -> np.dtype:
    return np.dtype(str(t.dtype).replace("torch.", ""))


def has_nan_dev(src: torch.Tensor) -> bool:
    """``da.any(da.isnan(array))`` (affine.py:347-349) -- one pass, one 4-byte read-back."""
    lib = load()
    src3 = src.unsqueeze(0) if src.dim() == 2 else src
    if src3.stride(2) != 1:
        src3 = src3.contiguous()
    n, h, w = src3.shape
    flag = torch.zeros(1, dtype=torch.int32, device=src3.device)
    slice_stride = src3.stride(0) if n > 1 else h * src3.stride(1)
    check(lib.xrs_has_nan(_dev.ptr(src3), DTYPE_CODES[_np_dtype(src3)], n, h, w, src3.stride(1), slice_stride,
                          _dev.ptr(flag), _dev.stream_ptr(src3.device)), "xrs_has_nan")
    return bool(flag.item())


def affine_resample_dev(src: torch.Tensor, scale_ji, offset_ji, out_hw, order: int, cval, agg: str = "mean",
                        factors=(1, 1), slice_blend: bool | None = None, recover: bool = False) -> torch.Tensor:
    """``xrs_affine`` on device buffers.

    src: (h, w) or (n, h, w) device tensor; source index = intermediate index * scale + offset,
    the intermediate image being ``out_hw * factors``; windows of ``factors`` samples are reduced
    with ``agg``.  Returns (out_h, out_w) or (n, out_h, out_w).
    """
    lib = load()
    if order not in (0, 1):
        raise ValueError(_ORDER_ERROR)
    squeeze = src.dim() == 2
    src3 = src.unsqueeze(0) if squeeze else src
    if src3.stride(2) != 1:
        src3 = src3.contiguous()
    dt = _np_dtype(src3)
    n, h, w = src3.shape
    f_j, f_i = int(factors[0]), int(factors[1])
    is_float = dt.kind == "f"
    out_int64 = f_j * f_i > 1 and (agg in _INT64_OUT_AGGS or (not is_float and agg in ("sum", "prod")))
    out_dtype = np.dtype(np.int64) if out_int64 else dt
    if slice_blend is None:
        slice_blend = not squeeze
    slice_stride = src3.stride(0) if n > 1 else h * src3.stride(1)
    if recover:  # affine.py:344-360; the result is float64 (filtered image / float64 filtered mask)
        out = _dev.empty((n, int(out_hw[0]), int(out_hw[1])), np.float64, src3.device)
        check(lib.xrs_affine_recover(_dev.ptr(src3), _dev.ptr(out), DTYPE_CODES[dt], n, h, w, src3.stride(1),
                                     slice_stride, int(out_hw[0]), int(out_hw[1]), float(scale_ji[0]),
                                     float(offset_ji[0]), float(scale_ji[1]), float(offset_ji[1]), float(cval),
                                     AGG_CODES[agg], f_j, f_i, int(bool(slice_blend)), _dev.stream_ptr(src3.device)),
              "xrs_affine_recover")
        return out[0] if squeeze else out
    out = _dev.empty((n, int(out_hw[0]), int(out_hw[1])), out_dtype, src3.device)
    check(lib.xrs_affine(_dev.ptr(src3), _dev.ptr(out), DTYPE_CODES[dt], n, h, w, src3.stride(1), slice_stride,
                         int(out_hw[0]), int(out_hw[1]), float(scale_ji[0]), float(offset_ji[0]), float(scale_ji[1]),
                         float(offset_ji[1]), int(order), float(cval), AGG_CODES[agg], f_j, f_i, int(bool(slice_blend)),
                         _dev.stream_ptr(src3.device)), "xrs_affine")
    return out[0] if squeeze else out


def coarsen_dev(src: torch.Tensor, factors, agg: str) -> torch.Tensor:
    """``dask.array.coarsen(agg, array, {y: f_j, x: f_i})`` on device buffers (``xrs_coarsen``)."""
    lib = load()
    h, w = src.shape[-2:]
    f_j, f_i = int(factors[0]), int(factors[1])
    if h % f_j or w % f_i:
        raise ValueError("coarsening factors must divide the image size")
    squeeze = src.dim() == 2
    src3 = src.unsqueeze(0) if squeeze else src
    if src3.stride(2) != 1:
        src3 = src3.contiguous()
    dt = _np_dtype(src3)
    n = src3.shape[0]
    out_int64 = f_j * f_i > 1 and (agg in _INT64_OUT_AGGS or (dt.kind != "f" and agg in ("sum", "prod")))
    out = _dev.empty((n, h // f_j, w // f_i), np.dtype(np.int64) if out_int64 else dt, src3.device)
    slice_stride = src3.stride(0) if n > 1 else h * src3.stride(1)
    # xrs_coarsen, not xrs_affine: the values as stored, without scipy's float64 round trip
    check(lib.xrs_coarsen(_dev.ptr(src3), _dev.ptr(out), DTYPE_CODES[dt], n, h, w, src3.stride(1), slice_stride,
                          AGG_CODES[agg], f_j, f_i, _dev.stream_ptr(src3.device)), "xrs_coarsen")
    return out[0] if squeeze else out


def _resample_array_dev(src: torch.Tensor, affine_matrix, output_hw, interp_method: int, agg_method: str,
                        recover_nan: bool, fill_value) -> torch.Tensor:
    """affine.py:243-362 (_resample_array / _downscale / _upscale) for one variable."""
    ((i_scale, _, i_off), (m10, j_scale, j_off)) = affine_matrix
    if interp_method > 1:
        raise ValueError(_ORDER_ERROR)
    recover = bool(recover_nan) and interp_method > 0 and _np_dtype(src).kind == "f" and has_nan_dev(src)
    # affine.py:253 tests matrix[1][0] (always 0) instead of the y scale: only the x scale (or a
    # non-zero shear term) triggers aggregation -- kept as is for drop-in behaviour
    if (i_scale > 1 or m10 > 1) and interp_method != 0:
        j_div = math.ceil(abs(j_scale))
        i_div = math.ceil(abs(i_scale))
        return affine_resample_dev(src, (j_scale / j_div, i_scale / i_div), (j_off, i_off), output_hw, interp_method,
                                   fill_value, agg_method, (j_div, i_div), recover=recover)
    return affine_resample_dev(src, (j_scale, i_scale), (j_off, i_off), output_hw, interp_method, fill_value,
                               recover=recover)


def resample_coords_dev(src: torch.Tensor, var_name, var, affine_matrix, target_size, interp_methods=None,
                        agg_methods=None, recover_nans=False) -> torch.Tensor:
    """What :func:`resample_dataset` does to ONE variable, device buffer in, device buffer out: the
    per-variable option resolution of affine.py:176-205 followed by ``_resample_array``.  Used for the
    2-D coordinate images of rectify's pre-downscale (rectify.py:234-260), which stay on the device."""
    interp = _get_interp_method_int(interp_methods, var_name, var)
    agg = _get_agg_method(agg_methods, var_name, var)
    recover = _get_recover_nan(recover_nans, var_name, var)
    fill = _get_fill_value(None, var_name, var)
    return _resample_array_dev(src, affine_matrix, (target_size[1], target_size[0]), interp, agg, recover, fill)


def resample_dataset(dataset, affine_matrix, yx_dims, target_size, target_tile_size, interp_methods=None,
                     agg_methods=None, recover_nans=False, fill_values=None) -> Dataset:
    """Resample every variable (data variables AND coordinates) with trailing ``yx_dims``.

    Drop-in for ``xcube_resampling.affine.resample_dataset`` (affine.py:140-240).
    ``target_tile_size`` is accepted for signature compatibility; the result is eager.
    """
    ds = from_any(dataset)
    data_vars, coords = {}, {}
    yx_dims = tuple(yx_dims)
    for var_name, var in ds.variables.items():
        new_var = None
        if var.dims[-2:] == yx_dims:
            interp = _get_interp_method_int(interp_methods, var_name, var)
            agg = _get_agg_method(agg_methods, var_name, var)
            recover = _get_recover_nan(recover_nans, var_name, var)
            fill = _get_fill_value(fill_values, var_name, var)
            assert var.ndim in (2, 3), f"Variable {var_name} has {var.ndim} dimensions."
            lead = var.shape[:-2]
            src = _dev.to_device(var.values)
            out = _resample_array_dev(src, affine_matrix, (target_size[1], target_size[0]), interp, agg, recover, fill)
            out_np = _dev.to_host(out).reshape(lead + (target_size[1], target_size[0]))
            if out_np.dtype == np.int64 and var.dtype.kind == "u" and agg in ("sum", "prod"):
                # np.nansum / np.nanprod of unsigned data return uint64 (coarsen.py:50-90); the kernel's
                # two's-complement int64 accumulator holds the same bits
                out_np = out_np.view(np.uint64)
            new_var = DataArray(out_np, dims=var.dims, attrs=var.attrs, name=var_name)
        elif yx_dims[0] not in var.dims and yx_dims[1] not in var.dims:
            new_var = var
        if new_var is not None:
            if var_name in ds.coords:
                coords[var_name] = new_var
            else:
                data_vars[var_name] = new_var
    return Dataset(data_vars=data_vars, coords=coords, attrs=ds.attrs)


def affine_transform_dataset(
    source_ds,
    target_gm: GridMapping,
    source_gm: GridMapping | None = None,
    variables: str | Iterable[str] | None = None,
    interp_methods=None,
    agg_methods=None,
    recover_nans=False,
    fill_values=None,
):
    """Resample a regular-grid dataset onto another regular grid of the same CRS.

    Drop-in for ``xcube_resampling.affine.affine_transform_dataset`` (affine.py:52-137).
    """
    user_ds = source_ds
    ds = from_any(source_ds)
    if source_gm is None:
        source_gm = GridMapping.from_dataset(ds)
    ds = normalize_grid_mapping(ds, source_gm)
    assert _can_apply_affine_transform(source_gm, target_gm), (
        f"Affine transformation cannot be applied to source CRS "
        f"{source_gm.crs.name!r} and target CRS {target_gm.crs.name!r}"
    )
    ds = _select_variables(ds, variables)
    target_ds = resample_dataset(
        ds,
        target_gm.ij_transform_to(source_gm),
        (source_gm.xy_dim_names[1], source_gm.xy_dim_names[0]),
        target_gm.size,
        target_gm.tile_size,
        interp_methods,
        agg_methods,
        recover_nans,
        fill_values,
    )
    x_name, y_name = target_gm.xy_var_names
    target_ds = target_ds.assign_coords({x_name: target_gm.x_coords, y_name: target_gm.y_coords})
    return to_like(target_ds, user_ds)
