"""The point ILU(0) restatement (oracle/pilu_ref.py) that tests/test_pilu_gpu.py checks csrc/pilu.cu against, on its own (no GPU):
on oracle-assembled Jacobians L U equals A at every position of the pattern, which is what defines ILU(0)."""
import numpy as np
import pytest

import _pins as P
from oracle import colour_ref, pilu_ref
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M


def greedy_colouring(indptr, indices, is_p, pressure_first=False):
    """A proper colouring of the matrix graph: one class after the other (velocity first unless pressure_first), the second
    class's colours numbered after the first's."""
    n = len(is_p)
    colour = -np.ones(n, dtype=np.int64)
    base = 0
    for cls in ((True, False) if pressure_first else (False, True)):
        rows = np.flatnonzero(is_p == cls)
        for i in rows:
            nb = np.asarray(indices[indptr[i]:indptr[i + 1]])
            nb = nb[(nb < n) & (nb != i)]
            nb = nb[is_p[nb] == cls]
            used = set(colour[nb].tolist())
            c = base
            while c in used:
                c += 1
            colour[i] = c
        base = colour[rows].max() + 1
    return colour


def _assemble(oracle, m, space, bcs, **fk):
    sp = space
    form = oracle.Form(gdim=m.gdim, vdeg=sp.vdeg, **fk)
    marker, value, mult = oracle.bc_arrays(sp.n_dofs, [b[0] for b in bcs], [np.broadcast_to(b[1], (len(b[0]),)) for b in bcs])
    indptr, indices = oracle.build_pattern(sp.dofmap, sp.n_dofs)
    w = np.where(marker != 0, value, 0.0) + 0.01 * np.random.default_rng(2).standard_normal(sp.n_dofs)
    vals = oracle.assemble_jacobian(form, m.x, m.cells, sp.dofmap, w, indptr, indices, marker, mult)
    return indptr, indices, vals


def _cases(oracle):
    m = M.create_rectangle_tris(5, 5); sp = M.mixed_space(m, 1)
    yield "cavity_ugn", sp, _assemble(oracle, m, sp, M.cavity_bcs(sp), flavour=1, nu=0.01)
    m = M.duct_mesh(1, 3); sp = M.mixed_space(m, 2)
    yield "duct_stokes_beta0", sp, _assemble(oracle, m, sp, P.uniform_inlet_duct_bcs(sp), flavour=2, nu=1.0, alpha=1.0, sp=-1.0, beta=0.0)


def test_pilu_ref_lu_equals_a_on_the_pattern(oracle):
    for name, sp, (indptr, indices, vals) in _cases(oracle):
        n = sp.n_dofs
        is_p = sp.dof_comp == sp.mesh.gdim
        colour = greedy_colouring(indptr, indices, is_p)
        assert colour[~is_p].max() < colour[is_p].min()
        order, L, U, udiag = pilu_ref.pilu0(indptr, indices, vals, colour)
        Ld, Ud = np.eye(n), np.diag(udiag)
        for i in range(n):
            Ld[i, L[i][0]] = L[i][1]
            Ud[i, U[i][0]] = U[i][1]
        rows = np.repeat(np.arange(n), np.diff(indptr))
        err = np.abs((Ld @ Ud)[rows, indices] - vals).max()
        assert err <= 1e-12 * np.abs(vals).max(), (name, err)
        # the application is the solve with those factors
        r = np.random.default_rng(4).standard_normal(n)
        z = pilu_ref.apply((order, L, U, udiag), r)
        assert np.abs(Ld @ (Ud @ z) - r).max() <= 1e-10 * np.abs(r).max(), name


def test_pilu_ref_pressure_first_meets_a_zero_pivot(oracle):
    """Taylor-Hood Stokes with beta = 0: a pressure row has no diagonal of its own; eliminated before its velocity neighbours its
    pivot is zero.  Velocity first, the pivot is the local Schur complement (the test above)."""
    name, sp, (indptr, indices, vals) = list(_cases(oracle))[1]
    is_p = sp.dof_comp == sp.mesh.gdim
    colour = greedy_colouring(indptr, indices, is_p, pressure_first=True)
    with pytest.raises(ZeroDivisionError, match="zero pivot"):
        pilu_ref.pilu0(indptr, indices, vals, colour)


def test_colour_ref_is_a_proper_colouring_velocity_first(oracle):
    """The colouring restatement (oracle/colour_ref.py) that tests/test_ilu_gpu.py and tests/test_pilu_gpu.py hold the device colours
    to: no two neighbours share a colour, and every pressure colour comes after every velocity colour."""
    for name, sp, (indptr, indices, vals) in _cases(oracle):
        n = sp.n_dofs
        is_p = sp.dof_comp == sp.mesh.gdim
        colour = colour_ref.colour(indptr, indices, n, cls=is_p)
        rows = np.repeat(np.arange(n), np.diff(indptr))
        off = rows != indices
        assert colour.min() == 0 and np.all(colour[rows[off]] != colour[indices[off]]), name
        assert colour[~is_p].max() + 1 == colour[is_p].min(), name
        assert np.array_equal(np.unique(colour), np.arange(colour.max() + 1)), name
