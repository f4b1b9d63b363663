"""CPU tests of the oracle (test infrastructure): it must agree with the reference's golden vectors,
with the fixtures generated from the compiled reference, and with the reference's outputs on further meshes
(2-D, single-cell, renumbered, edge tables), stored as digests."""
import json
import os
import sys

import numpy as np
import pytest

from helpers import GOLDEN, GOLDEN_CASES, GRID_ARRAYS, GRID_SCALARS, check_against_golden, digest, load_golden

import oracle
from ninpol_b200 import meshgen

sys.path.insert(0, GOLDEN)
import make_golden  # noqa: E402


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_matches_golden_fixtures(name):
    """Fixtures = outputs of the compiled reference; the oracle calls the same scipy DGELS/DGEMV, so
    even GLS is compared bit-for-bit."""
    mesh, d = load_golden(name)
    O = oracle.OracleInterpolator().load_mesh(mesh)
    check_against_golden(O, d, exact_gls=True)


@pytest.mark.parametrize("case", ["QUAD", "FAN", "ALH"])
def test_oracle_reproduces_published_accuracy(case):
    """Known-answer test from the reference's own results (tests/results/yaml/accuracy.yaml, hexa rows)."""
    table = json.load(open(os.path.join(GOLDEN, "accuracy_hexa.json")))["table"][case]
    for method in ("gls", "idw", "ls"):
        for n, published in zip(table[method]["n"][:2], table[method]["published"][:2]):
            mesh, sol = make_golden.analytic_mesh(case, n)
            O = oracle.OracleInterpolator().load_mesh(mesh)
            W, _ = O.interpolate(case, method)
            err = make_golden.interior_l2(W, mesh, sol, case, O.grid.boundary_points)
            assert abs(err - published) <= 5e-13 * max(1.0, abs(published)) + 1e-15, (case, method, n, err, published)


def test_oracle_linear_exactness():
    """LIN rows of accuracy.yaml (:293-438): LS and GLS reproduce a linear field to rounding."""
    mesh, sol = make_golden.analytic_mesh("LIN", 6)
    O = oracle.OracleInterpolator().load_mesh(mesh)
    for method in ("ls", "gls"):
        W, _ = O.interpolate("LIN", method)
        assert make_golden.interior_l2(W, mesh, sol, "LIN", O.grid.boundary_points) < 1e-14


def _stored(section, kind, n, kw):
    with open(make_golden.DIGESTS) as f:
        doc = json.load(f)[section]
    d = doc[make_golden.case_key(kind, n, kw)]
    mesh = meshgen.make_case(kind, n, **kw)
    assert make_golden.mesh_digest(mesh) == d["mesh"], "the mesh generator no longer makes the stored mesh"
    return mesh, d


@pytest.mark.parametrize("kind,n,kw", make_golden.SMALL_CASES)
def test_oracle_matches_compiled_reference(kind, n, kw):
    """Every output of the oracle equals the compiled reference's (stored as digests, tests/golden/make_golden.py)."""
    mesh, d = _stored("small", kind, n, kw)
    O = oracle.OracleInterpolator().load_mesh(mesh)
    for s in GRID_SCALARS:
        assert getattr(O.grid, s) == d["grid_scalars"][s], s
    for a in GRID_ARRAYS:
        assert digest(getattr(O.grid, a)) == d["grid"][a], a
    for method in ("idw", "ls", "gls"):
        W, nv = O.interpolate("u", method)
        want = d[method]
        for name, got in (("indptr", W.indptr), ("indices", W.indices), ("data", W.data), ("neumann", nv)):
            assert digest(got) == want[name], (method, name)


def test_release_build_diffusion_magnitude():
    """SURVEY.md Q2: (1 - 3/tr K)^2, independent of det K."""
    K = meshgen.random_spd_permeability(50, seed=7)
    dm = oracle.diffusion_magnitude(K)
    tr = K[:, 0] + K[:, 4] + K[:, 8]
    assert np.array_equal(dm, (1 - 3 / tr) ** 2)


@pytest.mark.parametrize("kind,n,kw", make_golden.EDGE_CASES)
def test_oracle_edges_match_compiled_reference(kind, n, kw):
    mesh, d = _stored("edges", kind, n, kw)
    O = oracle.OracleInterpolator().load_mesh(mesh, build_edges=True)
    assert O.grid.n_edges == d["n_edges"]
    assert digest(O.grid.inedel) == d["inedel"]
    assert digest(O.grid.inpoed) == d["inpoed"]
