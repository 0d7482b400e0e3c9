"""CPU checks of the oracle's exposed-point masks (tests/mask_oracle.py) and of surface_points: the masks are what the GPU
masks are compared with bit for bit, so they are checked here against the oracle's own counts and a float64 brute force."""
import numpy as np
import pytest

from tests.mask_oracle import exposed_masks

PROBE = 1.4


def popcount_rows(m):
    return np.unpackbits(np.ascontiguousarray(m, np.uint32).view(np.uint8), axis=1).sum(axis=1)


@pytest.mark.parametrize("lanes", [4, 8, 16])
@pytest.mark.parametrize("n_points", [100, 960])
def test_mask_popcounts_are_the_oracle_counts(oracle, golden, n_points, lanes):
    for name in golden.names:
        xyzr = golden.structure(name)["xyzr"]
        m = exposed_masks(oracle, xyzr, PROBE, n_points, lanes)
        assert m.shape == (xyzr.shape[0], (n_points + 31) // 32)
        c = oracle.calculate_sasa_internal(xyzr, PROBE, n_points, threads=0, lanes=lanes)["counts"]
        assert np.array_equal(popcount_rows(m), c), name
        if n_points % 32:
            assert not np.any(m[:, -1] >> np.uint32(n_points % 32)), name


def brute_force(oracle, xyzr, probe, n_points):
    """Per-point exposure in float64 (point p of atom i is occluded when it lies inside some other atom's probe-inflated
    sphere), and a mask of the points whose closest test lies within the 1e-5 A^2 boundary tolerance (|2R (dot - limit)|,
    where float32 rounding may decide either way)."""
    pts = oracle.sphere_points(n_points).astype(np.float64)
    x = xyzr.astype(np.float64)
    n = x.shape[0]
    exposed = np.ones((n, n_points), bool)
    near = np.zeros((n, n_points), bool)
    for i in range(n):
        r = x[i, 3] + probe
        v = x[i, :3] - x[:, :3]
        d2 = (v * v).sum(1)
        nb = np.nonzero((np.sqrt(d2) < x[i, 3] + x[:, 3] + 2 * probe + 0.1) & (np.arange(n) != i))[0]
        if nb.size == 0:
            continue
        limit = ((x[nb, 3] + probe) ** 2 - d2[nb] - r * r) / (2 * r)
        margin = 2 * r * (pts @ v[nb].T - limit[None, :])   # (n_points, k): squared distance to neighbour j minus its R_j^2
        exposed[i] = ~np.any(margin < 0, axis=1)
        near[i] = np.any(np.abs(margin) <= 1e-5, axis=1)
    return exposed, near


@pytest.mark.parametrize("name", ["example.cif", "2drt", "4xfj"])
def test_masks_agree_with_float64_brute_force(oracle, golden, name):
    xyzr = golden.structure(name)["xyzr"]
    for n_points, lanes in ((100, 8), (129, 16)):
        m = exposed_masks(oracle, xyzr, PROBE, n_points, lanes)
        bits = np.unpackbits(m.view(np.uint8), axis=1, bitorder="little")[:, :n_points].astype(bool)
        exposed, near = brute_force(oracle, xyzr, PROBE, n_points)
        decided = ~near
        assert decided.mean() > 0.99
        assert np.array_equal(bits[decided], exposed[decided]), (name, n_points)


def test_surface_points_lie_on_the_probe_spheres(oracle, golden):
    from rustsasa_b200 import surface_points
    xyzr = golden.structure("example.cif")["xyzr"]
    for n_points, probe in ((100, 1.4), (960, 0.0), (37, 3.0)):
        m = exposed_masks(oracle, xyzr, probe, n_points, 8)
        pts, atom = surface_points(xyzr, m, n_points, probe)
        assert pts.dtype == np.float32 and atom.dtype == np.int64
        assert pts.shape == (int(popcount_rows(m).sum()), 3) and atom.shape == (pts.shape[0],)
        assert np.all(np.diff(atom) >= 0)
        d = np.linalg.norm(pts.astype(np.float64) - xyzr[atom, :3].astype(np.float64), axis=1)
        R = xyzr[atom, 3].astype(np.float64) + probe
        assert np.all(np.abs(d - R) <= 1e-5 * np.maximum(R, 1.0) + 1e-5 * np.abs(xyzr[atom, :3]).max(axis=1)), n_points
        # the points of one atom are its exposed sphere points in the engine's order
        sphere = oracle.sphere_points(n_points)
        k = np.nonzero(np.unpackbits(m[atom[0]].view(np.uint8), bitorder="little")[:n_points])[0]
        want = xyzr[atom[0], :3] + (xyzr[atom[0], 3] + np.float32(probe)) * sphere[k]
        assert np.array_equal(pts[atom == atom[0]], want.astype(np.float32))
