"""pe_sphere_sums_atoms_and_groups: the per-atom and the grouped sphere sums in one call equal the two pe_sphere_sums calls
bit for bit, whether the per-atom sums run inside the grouped kernel or as a launch of their own."""
import ctypes
import io

import numpy as np
import pytest

from pdb_eda_b200 import _lib, ccp4, synthetic
from pdb_eda_b200._device import geom_from_header

ATOM_TYPE_RADII = np.array([0.78, 0.72, 0.66, 0.81, 0.84], dtype=np.float32)   # N, CA, C, O, CB of ALA
CELL = (48.0, 48.0, 48.0, 90, 90, 90)
N = (96, 96, 96)                                                               # a 0.5 A grid, as in bench.py's C2


def _structure_map(order, seed=5, crop=None):
    """(2Fo-Fc density map, float64 atom coordinates) of a poly-ALA structure; crop = (crsStart, (nc, nr, ns)) stores only
    part of the cell."""
    st = synthetic.polyAlaStructure(200, (0, 0, 0), CELL[:3], seed=seed)
    a, _ = synthetic.mapPair(st, N, CELL, seed=seed + 1, axisOrder=order)
    start = (0, 0, 0)
    if crop is not None:
        start, (nc, nr, ns) = crop
        a = np.ascontiguousarray(a[start[2]:start[2] + ns, start[1]:start[1] + nr, start[0]:start[0] + nc])
    dm = ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(a, CELL, N, crsStart=start, axisOrder=order)), "fused")
    xyz = np.array([at.coord for at in st.get_atoms()], dtype=np.float64)
    return dm.deviceMap, xyz


def _fused(dm, xyz, atom_r, group_r, start, cut_pos, cut_neg, max_r=None):
    """One call of the fused entry point; returns (atom rows, group rows, names of the kernels it launched)."""
    import torch
    from pdb_eda_b200._device import _ptr, _stream
    lib = _lib.load()
    n, ng = xyz.shape[0], len(start) - 1
    dev = dm.rho.device
    d_xyz = torch.as_tensor(xyz, dtype=torch.float64, device=dev).contiguous()
    d_ar = torch.as_tensor(atom_r, dtype=torch.float32, device=dev).contiguous()
    d_gr = torch.as_tensor(group_r, dtype=torch.float32, device=dev).contiguous()
    d_start = torch.as_tensor(start, dtype=torch.int32, device=dev).contiguous()
    out_a = torch.full((n, _lib.PE_SPHERE_NOUT), -7.0, dtype=torch.float64, device=dev)
    out_g = torch.full((ng, _lib.PE_SPHERE_NOUT), -7.0, dtype=torch.float64, device=dev)
    ws = torch.empty(max(int(lib.pe_sphere_workspace_bytes(n)), 256), dtype=torch.uint8, device=dev)
    max_r = float(np.max(atom_r)) if max_r is None else max_r
    torch.cuda.synchronize()
    _lib.profile(True, reset=True)
    rc = lib.pe_sphere_sums_atoms_and_groups(
        ctypes.byref(dm.geom), _ptr(dm.rho), n, _ptr(d_xyz), _ptr(d_ar), ctypes.c_float(max_r), _ptr(d_gr), ng, _ptr(d_start),
        ctypes.c_float(cut_pos), ctypes.c_float(cut_neg), _ptr(out_a), _ptr(out_g), _ptr(ws), _stream())
    _lib.check(rc, "pe_sphere_sums_atoms_and_groups")
    torch.cuda.synchronize()
    kernels = set(_lib.profile())
    _lib.profile(False)
    return out_a.cpu().numpy(), out_g.cpu().numpy(), kernels


def _check(dm, xyz, atom_r, group_r, start, cut_pos, cut_neg, fused_path):
    cut_pos, cut_neg = float(np.float32(cut_pos)), float(np.float32(cut_neg))
    got_a, got_g, kernels = _fused(dm, xyz, atom_r, group_r, start, cut_pos, cut_neg)
    want_a = dm.sphere_sums(xyz, atom_r, None, cut_pos, cut_neg).cpu().numpy()
    want_g = dm.sphere_sums(xyz, group_r, start, cut_pos, cut_neg).cpu().numpy()
    assert np.array_equal(got_a, want_a)
    assert np.array_equal(got_g, want_g)
    assert kernels >= {"sphere_union_kernel"}
    assert ("sphere_sums_kernel" not in kernels) == fused_path, kernels
    return want_a, want_g


@pytest.mark.gpu
@pytest.mark.parametrize("order", [(1, 2, 3), (1, 3, 2), (3, 1, 2)])   # z carried by the sections / rows / columns
@pytest.mark.parametrize("neg", [False, True])                         # with the negative class switched on
def test_c2_shaped_structure(order, neg):
    dm, xyz = _structure_map(order)
    n = xyz.shape[0]
    m, s = dm.mean_std()
    cut = m + 1.5 * s
    atom_r = np.tile(ATOM_TYPE_RADII, n // 5)
    start = np.arange(0, n + 1, 5, dtype=np.int32)
    want_a, want_g = _check(dm, xyz, atom_r, np.full(n, 3.5, np.float32), start, cut, -cut if neg else 0.0, True)
    assert want_a[:, 0].min() > 0 and want_a[:, 2].sum() > 0 and want_g[:, 0].min() > 0


@pytest.mark.gpu
def test_partial_map_with_atoms_over_its_edge():
    dm, xyz = _structure_map((1, 2, 3), seed=7, crop=((10, 20, 30), (60, 50, 40)))
    n = xyz.shape[0]
    atom_r = np.tile(ATOM_TYPE_RADII, n // 5)
    start = np.arange(0, n + 1, 5, dtype=np.int32)
    want_a, want_g = _check(dm, xyz, atom_r, np.full(n, 3.5, np.float32), start, 0.5, 0.0, True)
    for rows in (want_a, want_g):
        assert (rows[:, 6] == 0.0).any() and (rows[:, 6] == 1.0).any()


@pytest.mark.gpu
def test_ragged_atom_count_single_atom_and_empty_groups():
    dm, xyz = _structure_map((1, 3, 2), seed=9)
    xyz = xyz[:301]
    atom_r = np.resize(ATOM_TYPE_RADII, 301)
    start = np.array([0, 1, 2, 2] + list(range(7, 301, 6)) + [301], dtype=np.int32)
    want_a, want_g = _check(dm, xyz, atom_r, np.full(301, 3.0, np.float32), start, 0.4, -0.2, True)
    assert want_g[2, 0] == 0.0 and want_g[2, 6] == 1.0                    # the empty group


@pytest.mark.gpu
@pytest.mark.parametrize("radius, fused_path", [(1.74, True), (1.75, False), (1.76, False)])
def test_box_width_limit(radius, fused_path):
    """On a 0.5 A grid R = round(r / 0.5) and the box is 2 R + 2 wide: 8 up to r < 1.75 (round half to even takes 3.5 to 4)."""
    dm, xyz = _structure_map((3, 1, 2), seed=11)
    n = xyz.shape[0]
    atom_r = np.tile(ATOM_TYPE_RADII, n // 5)
    atom_r[::7] = radius
    start = np.arange(0, n + 1, 5, dtype=np.int32)
    _check(dm, xyz, atom_r, np.full(n, 3.5, np.float32), start, 0.5, 0.0, fused_path)


@pytest.mark.gpu
def test_a_radius_above_the_bound_gives_nan_rows():
    dm, xyz = _structure_map((1, 2, 3), seed=13)
    n = xyz.shape[0]
    start = np.arange(0, n + 1, 5, dtype=np.int32)
    group_r = np.full(n, 3.5, np.float32)
    got_a, got_g, kernels = _fused(dm, xyz, np.full(n, 2.5, np.float32), group_r, start, 0.5, 0.0, max_r=1.0)
    assert "sphere_sums_kernel" not in kernels
    assert np.isnan(got_a).all()
    assert np.array_equal(got_g, dm.sphere_sums(xyz, group_r, start, 0.5, 0.0).cpu().numpy())


def test_workspace_holds_what_the_entry_points_carve():
    """The atoms' boxes (6 int32 each) and distance thresholds (float64) in 256-byte aligned regions, then the grouped kernel's
    work-item counter (one int), which a grouped call writes even when it has no atoms."""
    lib = _lib.load()

    def aligned(nbytes):
        return (nbytes + 255) // 256 * 256

    assert lib.pe_sphere_workspace_bytes(0) >= 4
    for n in (1, 5, 40_000):
        assert lib.pe_sphere_workspace_bytes(n) >= aligned(24 * n) + aligned(8 * n) + 4, n


def test_argument_errors_match_pe_sphere_sums():
    """Checked on the host before anything is launched: the same status codes as pe_sphere_sums."""
    lib = _lib.load()
    dm = ccp4.parse(io.BytesIO(synthetic.ccp4Bytes(np.zeros((8, 8, 8), np.float32), (4.0, 4.0, 4.0, 90, 90, 90), (8, 8, 8))), "args")
    g = geom_from_header(dm.header)
    bad = _lib.PeGeom()
    fake = ctypes.c_void_p(16)   # never dereferenced: every call below fails its checks first

    def both(geom, n, ptr, ng, start, cp=0.0, cn=0.0):
        rg = lib.pe_sphere_sums(ctypes.byref(geom), ptr, n, ptr, ptr, ng, start, cp, cn, ptr, ptr, None)
        rf = lib.pe_sphere_sums_atoms_and_groups(ctypes.byref(geom), ptr, n, ptr, ptr, 1.0, ptr, ng, start, cp, cn, ptr, ptr, ptr, None)
        return rg, rf

    for args in ((bad, 4, fake, 4, fake),            # invalid geometry
                 (g, -1, fake, 4, fake),             # negative size
                 (g, 4, fake, -1, fake),
                 (g, 4, None, 2, fake),              # null pointers
                 (g, 4, fake, 3, None)):             # n_groups != n_atoms without group offsets
        want, got = both(*args)
        assert want == got == -1, args
    assert both(g, 4, fake, 2, fake, cp=-1.0) == (-1, -1)    # cut_pos < 0
    assert both(g, 4, fake, 2, fake, cn=1.0) == (-1, -1)     # cut_neg > 0
    assert both(g, 0, None, 0, None) == (0, 0)               # nothing to do
