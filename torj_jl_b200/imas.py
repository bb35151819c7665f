"""IMAS data-dictionary ingestion: equilibrium + core_profiles -> the eleven arrays ``Plasma(...)`` takes.

Follows the reference's test preamble, test/tests/setup.jl:31-62 (SURVEY.md §8(f) rank 3): that file reads an IMAS
JSON (`IMAS.json2imas`), sets `dd.global_time`, takes the equilibrium time slice and the core-profiles slice valid at
that time, normalises every psi with `(psi - psi_axis)/(psi_boundary - psi_axis)` and calls `TorJ.Plasma`.  Host-side
setup only; nothing here is on the device path.

PARITY UNPINNED: IMAS.jl is un-vendored and the reference's sample file lives in a remote artifact
(test/Artifacts.toml:4-7), so the two conventions this module has to assume could not be observed here:
  * 2-D arrays are nested lists with the OUTER index running over `grid.dim1` (R) — the OMAS/numpy `tolist()` layout
    that IMAS JSON files are written in; `matrix_order="dim2_outer"` reads the transposed layout, and for non-square
    grids the orientation is detected from the lengths;
  * `time_slice[]` / `profiles_1d[]` select the last slice whose time is <= `global_time` (IMAS.jl's causal lookup).
`solovev_dd` writes a dd of the synthetic equilibrium in the same layout, so the path can be exercised end to end.
"""
from __future__ import annotations

import json

import numpy as np

from .plasma import Plasma


def load_imas_json(path: str) -> dict:
    """IMAS.json2imas(path; error_on_missing_coordinates=false) — test/tests/setup.jl:31. Plain nested dicts/lists."""
    with open(path, "r") as fh:
        return json.load(fh)


def causal_index(times, global_time: float) -> int:
    """Index of the last entry of `times` that is <= global_time (IMAS.jl `time_slice[]` with dd.global_time,
    test/tests/setup.jl:32-34). Raises like IMAS.jl when global_time precedes the first slice."""
    t = np.asarray(times, dtype=np.float64)
    if t.size == 0:
        raise ValueError("no time slices")
    if np.any(np.diff(t) < 0):
        raise ValueError("time base is not sorted")
    i = int(np.searchsorted(t, global_time, side="right")) - 1
    if i < 0:
        raise ValueError(f"global_time {global_time} is before the first time slice {t[0]}")
    return i


def _times(ids: dict, slices: list) -> list:
    if len(slices) and all(isinstance(s, dict) and "time" in s for s in slices):
        return [s["time"] for s in slices]
    if "time" in ids and len(ids["time"]) == len(slices):
        return list(ids["time"])
    raise ValueError("IDS has neither per-slice `time` nor a matching `time` vector")


def _slice(ids: dict, key: str, global_time):
    slices = ids[key]
    if not slices:
        raise ValueError(f"{key} is empty")
    if global_time is None:
        if len(slices) != 1:
            raise ValueError(f"{key} has {len(slices)} slices: global_time is required")
        return slices[0]
    return slices[causal_index(_times(ids, slices), global_time)]


def _matrix(nested, n1: int, n2: int, matrix_order: str) -> np.ndarray:
    """Nested list -> array [dim1, dim2]."""
    a = np.asarray(nested, dtype=np.float64)
    if a.ndim != 2:
        raise ValueError("expected a 2-D array")
    if matrix_order not in ("dim1_outer", "dim2_outer", "auto"):
        raise ValueError("matrix_order must be 'dim1_outer', 'dim2_outer' or 'auto'")
    if n1 != n2:  # orientation is unambiguous on a non-square grid
        if a.shape == (n1, n2):
            return a
        if a.shape == (n2, n1):
            return np.ascontiguousarray(a.T)
        raise ValueError(f"2-D array of shape {a.shape} does not match the grid ({n1}, {n2})")
    if a.shape != (n1, n2):
        raise ValueError(f"2-D array of shape {a.shape} does not match the grid ({n1}, {n2})")
    return np.ascontiguousarray(a.T) if matrix_order == "dim2_outer" else a  # square: "auto" means dim1 outer


def plasma_arrays_from_dd(dd: dict, global_time=None, *, density_scale: float = 1.0, matrix_order: str = "auto") -> dict:
    """The keyword form of test/tests/setup.jl:34-55. `density_scale` is the factor of `plasma_low_density`
    (setup.jl:57-58)."""
    eq_slice = _slice(dd["equilibrium"], "time_slice", global_time)        # setup.jl:34
    p2d = eq_slice["profiles_2d"][0]                                      # setup.jl:35-36,39,53-54
    R_grid = np.asarray(p2d["grid"]["dim1"], dtype=np.float64)
    z_grid = np.asarray(p2d["grid"]["dim2"], dtype=np.float64)
    gq = eq_slice["global_quantities"]
    psi_axis, psi_boundary = float(gq["psi_axis"]), float(gq["psi_boundary"])
    if psi_boundary == psi_axis:
        raise ValueError("psi_boundary == psi_axis")
    norm = lambda psi: (np.asarray(psi, dtype=np.float64) - psi_axis) / (psi_boundary - psi_axis)
    nR, nZ = len(R_grid), len(z_grid)
    mat = lambda key: _matrix(p2d[key], nR, nZ, matrix_order)
    profiles_1d = _slice(dd["core_profiles"], "profiles_1d", global_time)  # setup.jl:38
    el = profiles_1d["electrons"]
    return dict(
        R_coords=R_grid, Z_coords=z_grid,
        psi_norm_data=norm(mat("psi")),                                    # setup.jl:39
        psi_prof=norm(profiles_1d["grid"]["psi"]),                         # setup.jl:41
        ne_prof=np.asarray(el["density"], dtype=np.float64) * density_scale,
        Te_prof=np.asarray(el["temperature"], dtype=np.float64),
        Br_data=mat("b_field_r"), Bz_data=mat("b_field_z"), Bphi_data=mat("b_field_tor"),
        eqt1d_psi_norm=norm(eq_slice["profiles_1d"]["psi"]),               # setup.jl:37
        eqt1d_volume=np.asarray(eq_slice["profiles_1d"]["volume"], dtype=np.float64))


def plasma_from_dd(dd: dict, global_time=None, *, density_scale: float = 1.0, matrix_order: str = "auto",
                   build: str = "host") -> Plasma:
    a = plasma_arrays_from_dd(dd, global_time, density_scale=density_scale, matrix_order=matrix_order)
    return Plasma(a["R_coords"], a["Z_coords"], a["psi_norm_data"], a["psi_prof"], a["ne_prof"], a["Te_prof"],
                  a["Br_data"], a["Bz_data"], a["Bphi_data"], a["eqt1d_psi_norm"], a["eqt1d_volume"], build=build)


def plasmas_from_dd(dd: dict, times=None, *, density_scale: float = 1.0, matrix_order: str = "auto",
                    build: str = "host") -> list:
    """One Plasma per equilibrium time slice — every slice (times=None) or the slice valid at each of `times` under the
    causal lookup — each with the core_profiles slice valid at that slice's time: the plasma set of
    trace_bundle / make_beams / make_beam_series. Raises ValueError when the slices' 2-D grids differ (a set shares one
    (R,Z) grid; resample the equilibria first)."""
    eq = dd["equilibrium"]
    if times is None:
        times = _times(eq, eq["time_slice"]) if eq["time_slice"] else []
    times = [float(t) for t in np.atleast_1d(times)]
    if not times:
        raise ValueError("no time slices")
    arrs = [plasma_arrays_from_dd(dd, t, density_scale=density_scale, matrix_order=matrix_order) for t in times]
    for t, a in zip(times, arrs):
        if not (np.array_equal(a["R_coords"], arrs[0]["R_coords"]) and np.array_equal(a["Z_coords"], arrs[0]["Z_coords"])):
            raise ValueError(f"the (R,Z) grid of the slice at t = {t} differs from that at t = {times[0]}: "
                             "a plasma set shares one grid")
    return [Plasma(a["R_coords"], a["Z_coords"], a["psi_norm_data"], a["psi_prof"], a["ne_prof"], a["Te_prof"], a["Br_data"],
                   a["Bz_data"], a["Bphi_data"], a["eqt1d_psi_norm"], a["eqt1d_volume"], build=build) for a in arrs]


def plasma_from_imas_json(path: str, global_time=None, **kw) -> Plasma:
    """test/tests/setup.jl:31-55 in one call."""
    return plasma_from_dd(load_imas_json(path), global_time, **kw)


def solovev_dd(arrays: dict, *, times=(2.0,), psi_axis: float = -0.35, psi_boundary: float = 0.85,
               ne_scale_per_slice=None) -> dict:
    """A minimal dd (nested dicts/lists as `json.dump` writes them) holding the arrays of
    `synthetic.solovev_arrays` at each of `times`, with un-normalised psi = psi_axis + psi_N (psi_boundary - psi_axis).
    `ne_scale_per_slice` scales the density of slice k, so that tests can tell the slices apart."""
    un = lambda pn: (psi_axis + np.asarray(pn) * (psi_boundary - psi_axis))
    scales = list(ne_scale_per_slice) if ne_scale_per_slice is not None else [1.0] * len(times)
    eq_slices, cp_slices = [], []
    for t, sc in zip(times, scales):
        eq_slices.append(dict(
            time=float(t),
            global_quantities=dict(psi_axis=psi_axis, psi_boundary=psi_boundary),
            profiles_1d=dict(psi=un(arrays["eqt1d_psi_norm"]).tolist(), volume=np.asarray(arrays["eqt1d_volume"]).tolist()),
            profiles_2d=[dict(grid_type=dict(index=1, name="rectangular"),
                              grid=dict(dim1=np.asarray(arrays["R_coords"]).tolist(), dim2=np.asarray(arrays["Z_coords"]).tolist()),
                              psi=un(arrays["psi_norm_data"]).tolist(),
                              b_field_r=np.asarray(arrays["Br_data"]).tolist(),
                              b_field_z=np.asarray(arrays["Bz_data"]).tolist(),
                              b_field_tor=np.asarray(arrays["Bphi_data"]).tolist())]))
        cp_slices.append(dict(
            time=float(t),
            grid=dict(psi=un(arrays["psi_prof"]).tolist()),
            electrons=dict(density=(np.asarray(arrays["ne_prof"]) * sc).tolist(),
                           temperature=np.asarray(arrays["Te_prof"]).tolist())))
    tl = [float(t) for t in times]
    return dict(equilibrium=dict(time=tl, time_slice=eq_slices), core_profiles=dict(time=tl, profiles_1d=cp_slices))
