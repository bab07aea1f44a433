"""CF-convention grid-mapping discovery: which CRS and which coordinate variables describe a dataset.

Host-side counterpart of the reference's ``gridmapping/cfconv.py:66-212`` (what
``GridMapping.from_dataset`` runs before it derives the grid from the coordinates) and of
``add_spatial_ref`` (``cfconv.py:320-358``) for uncompressed Zarr-v2 directory stores.  The CRS
descriptor is this package's own (``crs.py``): grid-mapping attributes it cannot express
(rotated pole, ...) are skipped, exactly as ``pyproj.CRS.from_cf`` failing is in the reference.

Discovery order (same outcomes as the reference, expressed as data):

1. grid-mapping variables referenced by a ``grid_mapping`` attribute of any variable;
2. else the first variable whose own attributes describe a CRS;
3. else the dataset's attributes;
4. coordinate variables by CF ``standard_name``, then by the usual names, per CRS family
   (geographic, rotated pole, projected); bounds variables are never coordinates;
5. coordinates without a grid mapping get the caller's default CRS of their family
   (WGS 84 for lon / lat).
"""

from __future__ import annotations

import json
import os
import warnings
from collections.abc import Hashable

from .crs import CRS, CRS_WGS84
from .dataset import DataArray, Dataset, from_any

# (family, grid_mapping_name or None, CF standard names (x, y), common variable names (x), (y))
_FAMILIES = (
    ("latitude_longitude", ("longitude", "latitude"), ("lon", "longitude"), ("lat", "latitude")),
    ("rotated_latitude_longitude", ("grid_longitude", "grid_latitude"), ("rlon", "rlongitude"), ("rlat", "rlatitude")),
    (None, ("projection_x_coordinate", "projection_y_coordinate"), ("x", "xc", "transformed_x"),
     ("y", "yc", "transformed_y")),
)


class GridCoords:
    """The x and y coordinate variables of one CRS family."""

    def __init__(self):
        self.x: DataArray | None = None
        self.y: DataArray | None = None


class GridMappingProxy:
    """A CRS, its CF ``grid_mapping_name``, its coordinates and the spatial chunking, not yet a GridMapping."""

    def __init__(self, crs: CRS | None = None, name: str | None = None, coords: GridCoords | None = None,
                 tile_size: tuple[int, int] | None = None):
        self.crs, self.name, self.coords, self.tile_size = crs, name, coords, tile_size


def _proxy_from_attrs(attrs) -> GridMappingProxy | None:
    if not attrs:
        return None
    try:
        crs = CRS.from_cf(dict(attrs))
    except (ValueError, TypeError, KeyError):
        return None
    return GridMappingProxy(crs=crs, name=attrs.get("grid_mapping_name"))


def _is_bounds_name(ds: Dataset, name) -> bool:
    base, _, suffix = str(name).rpartition("_")
    return bool(base) and suffix in ("bnds", "bounds") and base in ds


def find_potential_coord_vars(ds: Dataset) -> list[Hashable]:
    """1-D / 2-D variables that may be coordinates: not bounds variables (CF ``bounds`` attribute or
    ``*_bnds`` / ``*_bounds`` names); those named by a global ``coordinates`` attribute come first."""
    variables = ds.variables
    bounds = {v.attrs.get("bounds") for v in variables.values() if v.attrs.get("bounds") in variables}
    bounds |= {n for n in variables if _is_bounds_name(ds, n)}

    def ok(name):
        return name in variables and variables[name].ndim in (1, 2) and name not in bounds

    first = [n for n in str(ds.attrs.get("coordinates") or "").split() if ok(n)]
    return first + [n for n in variables if n not in first and ok(n)]


def get_dataset_grid_mapping_proxies(dataset, *, missing_latitude_longitude_crs: CRS | None = None,
                                     missing_rotated_latitude_longitude_crs: CRS | None = None,
                                     missing_projected_crs: CRS | None = None,
                                     emit_warnings: bool = False) -> dict:
    """{grid-mapping variable name (or ``None``): :class:`GridMappingProxy`} for every CRS of the
    dataset that comes with usable x / y coordinates (same rules as ``cfconv.py:66-212``)."""
    ds = from_any(dataset)
    variables = ds.variables
    proxies: dict = {}
    for var in variables.values():  # 1. referenced grid-mapping variables
        ref = var.attrs.get("grid_mapping")
        if ref and ref not in proxies and ref in variables:
            proxies[ref] = _proxy_from_attrs(variables[ref].attrs)
    proxies = {k: v for k, v in proxies.items() if v is not None}
    if not proxies:  # 2. a variable that carries CRS attributes itself
        for name, var in variables.items():
            gmp = _proxy_from_attrs(var.attrs)
            if gmp is not None:
                proxies[name] = gmp
                break
    if not proxies:  # 3. the dataset's attributes
        gmp = _proxy_from_attrs(ds.attrs)
        if gmp is not None:
            proxies[None] = gmp

    # 4. coordinates per family: standard names win over common names, first match wins
    candidates = find_potential_coord_vars(ds)
    families = {fam[0]: GridCoords() for fam in _FAMILIES}
    for by_standard_name in (True, False):
        for name in candidates:
            var = variables[name]
            for family, std_names, x_names, y_names in _FAMILIES:
                coords = families[family]
                is_x = var.attrs.get("standard_name") == std_names[0] if by_standard_name else name in x_names
                is_y = var.attrs.get("standard_name") == std_names[1] if by_standard_name else name in y_names
                if coords.x is None and is_x:
                    coords.x = DataArray(var, name=name)
                if coords.y is None and is_y:
                    coords.y = DataArray(var, name=name)
    for gmp in proxies.values():
        gmp.coords = families[gmp.name if gmp.name in families else None]

    # 5. coordinates that no grid mapping claimed get the default CRS of their family
    defaults = {"latitude_longitude": missing_latitude_longitude_crs or CRS_WGS84,
                "rotated_latitude_longitude": missing_rotated_latitude_longitude_crs, None: missing_projected_crs}
    for family, coords in families.items():
        if coords.x is None and coords.y is None:
            continue
        gmp = next((g for g in proxies.values() if family is None or family == g.name), None)
        if gmp is None and defaults[family] is not None:
            gmp = proxies[None] = GridMappingProxy(crs=defaults[family], name=family)
        if gmp is not None:
            if gmp.coords is None:
                gmp.coords = coords
            # a CRS-84 GeoTIFF read by rioxarray names its 1-D lon / lat coordinates "x" and "y"
            if gmp.coords.x is None:
                gmp.coords.x = coords.x
            if gmp.coords.y is None:
                gmp.coords.y = coords.y

    complete = {}
    for key, gmp in proxies.items():
        c = gmp.coords
        usable = (c is not None and c.x is not None and c.y is not None and c.x.size >= 2 and c.y.size >= 2
                  and c.x.ndim == c.y.ndim and (c.x.ndim == 1 or (c.x.ndim == 2 and c.x.dims == c.y.dims)))
        if usable:
            complete[key] = gmp  # (eager numpy data has no chunking: tile_size stays None)
        elif emit_warnings:
            warnings.warn(f'CRS "{gmp.name}": missing x- and/or y-coordinates (grid mapping variable "{key}": '
                          f'grid_mapping_name="{gmp.name}")')
    return complete


def add_spatial_ref(store_path: str, crs: CRS, crs_var_name: str = "spatial_ref",
                    xy_dim_names: tuple[str, str] | None = None) -> None:
    """``cfconv.py:320-358`` for a Zarr v2 or v3 DIRECTORY store: add a scalar ``spatial_ref`` array that
    carries the CRS's CF attributes and point every array whose last two dimensions are (y, x) at it
    (``grid_mapping`` attribute); consolidated metadata, if present, is rewritten."""
    if not isinstance(store_path, str):
        raise TypeError(f"dataset_store must be a path, was {type(store_path)}")
    if not isinstance(crs_var_name, str):
        raise TypeError(f"crs_var_name must be an instance of {str}, was {type(crs_var_name)}")
    x_dim, y_dim = xy_dim_names or ("x", "y")
    if os.path.isfile(os.path.join(store_path, "zarr.json")):
        _add_spatial_ref_v3(store_path, crs, crs_var_name, x_dim, y_dim)
        return
    var_dir = os.path.join(store_path, crs_var_name)
    os.makedirs(var_dir, exist_ok=True)
    with open(os.path.join(var_dir, ".zarray"), "w") as fh:
        json.dump({"chunks": [], "compressor": None, "dtype": "|u1", "fill_value": 0, "filters": None, "order": "C",
                   "shape": [], "zarr_format": 2}, fh)
    with open(os.path.join(var_dir, "0"), "wb") as fh:
        fh.write(b"\x00")
    attrs = dict(crs.to_cf())
    attrs["_ARRAY_DIMENSIONS"] = []
    with open(os.path.join(var_dir, ".zattrs"), "w") as fh:
        json.dump(attrs, fh)
    for item in sorted(os.listdir(store_path)):
        zattrs = os.path.join(store_path, item, ".zattrs")
        if item == crs_var_name or not os.path.isfile(os.path.join(store_path, item, ".zarray")):
            continue
        meta = json.load(open(zattrs)) if os.path.isfile(zattrs) else {}
        dims = meta.get("_ARRAY_DIMENSIONS")
        if dims and len(dims) >= 2 and dims[-2] == y_dim and dims[-1] == x_dim:
            meta["grid_mapping"] = crs_var_name
            with open(zattrs, "w") as fh:
                json.dump(meta, fh)
    consolidated = os.path.join(store_path, ".zmetadata")
    if os.path.isfile(consolidated):
        entries = {}
        for root, _dirs, files in os.walk(store_path):
            for f in files:
                if f in (".zarray", ".zattrs", ".zgroup"):
                    key = os.path.relpath(os.path.join(root, f), store_path).replace(os.sep, "/")
                    entries[key] = json.load(open(os.path.join(root, f)))
        with open(consolidated, "w") as fh:
            json.dump({"metadata": entries, "zarr_consolidated_format": 1}, fh)


def _add_spatial_ref_v3(store_path: str, crs: CRS, crs_var_name: str, x_dim: str, y_dim: str) -> None:
    """:func:`add_spatial_ref` for a Zarr v3 group: a 0-D uint8 array (codecs ``[bytes]``, chunk key in the store's
    encoding), ``grid_mapping`` in the ``attributes`` of the (y, x) arrays, and the root's ``consolidated_metadata``
    entries rewritten when it has them."""
    from .io import _v3_key, v3_dimension_names

    root_path = os.path.join(store_path, "zarr.json")
    root = json.load(open(root_path))
    if root.get("zarr_format") != 3 or root.get("node_type") != "group":
        raise ValueError(f"{store_path}: not a Zarr v3 group")
    arrays = {}
    for item in sorted(os.listdir(store_path)):
        meta_path = os.path.join(store_path, item, "zarr.json")
        if item != crs_var_name and os.path.isfile(meta_path):
            meta = json.load(open(meta_path))
            if meta.get("node_type") == "array":
                arrays[item] = meta
    encoding = next((m["chunk_key_encoding"] for m in arrays.values() if m.get("chunk_key_encoding")),
                    {"name": "default", "configuration": {"separator": "/"}})
    var_dir = os.path.join(store_path, crs_var_name)
    os.makedirs(var_dir, exist_ok=True)
    sr = {"zarr_format": 3, "node_type": "array", "shape": [], "data_type": "uint8",
          "chunk_grid": {"name": "regular", "configuration": {"chunk_shape": []}}, "chunk_key_encoding": encoding,
          "fill_value": 0, "codecs": [{"name": "bytes"}], "attributes": dict(crs.to_cf()), "dimension_names": [],
          "storage_transformers": []}
    with open(os.path.join(var_dir, "zarr.json"), "w") as fh:
        json.dump(sr, fh)
    with open(os.path.join(var_dir, _v3_key(encoding, ())), "wb") as fh:
        fh.write(b"\x00")
    for item, meta in arrays.items():
        dims = v3_dimension_names(meta)
        if len(dims) >= 2 and dims[-2] == y_dim and dims[-1] == x_dim:
            meta["attributes"] = dict(meta.get("attributes") or {}, grid_mapping=crs_var_name)
            with open(os.path.join(store_path, item, "zarr.json"), "w") as fh:
                json.dump(meta, fh)
    consolidated = root.get("consolidated_metadata")
    if isinstance(consolidated, dict) and "metadata" in consolidated:
        entries = {}
        for dirpath, _dirs, files in os.walk(store_path):
            if "zarr.json" in files and dirpath != store_path:
                key = os.path.relpath(dirpath, store_path).replace(os.sep, "/")
                entries[key] = json.load(open(os.path.join(dirpath, "zarr.json")))
        consolidated["metadata"] = dict(sorted(entries.items()))
        with open(root_path, "w") as fh:
            json.dump(root, fh)
