"""Host-side mirror of the reference's assembly seam, on top of the C ABI (ctypes, NumPy in/out).

``NSAssembler`` owns one GPU context (= one MPI rank's partition) and exposes the five dolfinx calls the
reference makes per Newton iterate -- ``create_matrix``, ``assemble_vector`` + ``apply_lifting`` + ``set_bc``
(= ``residual``) and ``assemble_matrix`` (= ``jacobian``) -- plus ``mult`` (PETSc MatMult).
``NonlinearPDE_SNESProblem`` keeps the constructor role and the ``F(snes, x, F)`` / ``J(snes, x, J, P)``
callback signatures of NavierStokes/NavierStokesChannelFlow.py:40-75 so that ``snes.setFunction`` /
``snes.setJacobian`` (:278-279) can be pointed at it unchanged.
"""
import ctypes

import numpy as np

from . import _lib

GMETRIC, UGN, STOKES = 0, 1, 2


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class NSAssembler:
    def __init__(self, x, cells, dofmap, vdeg=1, n_dofs_owned=None, n_dofs_ghost=0, n_cells_owned=None, device=0, options=None):
        self.lib = _lib.load()
        self.ctx = ctypes.c_void_p()
        rc = self.lib.nsgpu_create(ctypes.byref(self.ctx), device)
        if rc != 0:
            raise _lib.NsgpuError(f"nsgpu_create failed ({rc}): {self.lib.nsgpu_last_error(None).decode()}")
        x = np.ascontiguousarray(x, dtype=np.float64)
        cells = np.ascontiguousarray(cells, dtype=np.int32)
        dofmap = np.ascontiguousarray(dofmap, dtype=np.int32)
        if x.ndim != 2 or x.shape[1] != 3:
            raise ValueError("x must be (n_nodes, 3) like mesh.geometry.x")
        self.gdim = cells.shape[1] - 1
        self.vdeg = vdeg
        self.n_cells_total = cells.shape[0]
        self.n_cells_owned = self.n_cells_total if n_cells_owned is None else int(n_cells_owned)
        if dofmap.shape[0] != self.n_cells_total:
            raise ValueError("dofmap and geometry dofmap must have one row per cell")
        self.ndofs_cell = dofmap.shape[1]
        n_total = int(dofmap.max()) + 1 if n_dofs_owned is None else int(n_dofs_owned) + int(n_dofs_ghost)
        self.n_owned = n_total - int(n_dofs_ghost) if n_dofs_owned is None else int(n_dofs_owned)
        self.n_ghost = int(n_dofs_ghost)
        self.n_dofs = self.n_owned + self.n_ghost
        for k, v in (options or {}).items():          # options that must be known before the space is set ("renumber", "renumber_order")
            self.set_option(k, v)
        self._check(self.lib.nsgpu_set_mesh(self.ctx, self.gdim, x.shape[0], _ptr(x), self.n_cells_owned, self.n_cells_total, _ptr(cells)), "set_mesh")
        self._check(self.lib.nsgpu_set_space(self.ctx, vdeg, _ptr(dofmap), self.n_owned, self.n_ghost), "set_space")
        self.n_cols = self.n_dofs
        self.nnz = None
        self.n_rows = None
        self.n_tags = 0

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc, what):
        _lib.check(self.ctx, rc, what)

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.nsgpu_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name, value):
        self._check(self.lib.nsgpu_set_option(self.ctx, name.encode(), int(value)), f"set_option({name})")

    # ------------------------------------------------------------------ problem definition
    def set_form(self, flavour=GMETRIC, nu=0.1, Ci=36.0, alpha=1.0, sp=1.0, beta=0.0):
        """define_navier_stokes_form(W, msh, Re) reduced to its parameters (nu = 1/Re)."""
        self._check(self.lib.nsgpu_set_form(self.ctx, int(flavour), float(nu), float(Ci), float(alpha), float(sp), float(beta)), "set_form")

    def set_bcs(self, bcs):
        """bcs: ordered list of (dofs, values), one pair per dirichletbc object."""
        ptr = np.zeros(len(bcs) + 1, dtype=np.int64)
        for k, (d, _) in enumerate(bcs):
            ptr[k + 1] = ptr[k] + len(d)
        dofs = np.ascontiguousarray(np.concatenate([np.asarray(d, dtype=np.int32) for d, _ in bcs]) if bcs else np.zeros(0, np.int32))
        vals = np.ascontiguousarray(np.concatenate([np.broadcast_to(np.asarray(v, dtype=np.float64), (len(d),)) for d, v in bcs]) if bcs else np.zeros(0))
        self._check(self.lib.nsgpu_set_bcs(self.ctx, len(bcs), _ptr(ptr), _ptr(dofs), _ptr(vals)), "set_bcs")

    def create_matrix(self, fetch=True):
        """create_matrix(problem.a): returns (indptr int64, indices int32) of the CSR pattern."""
        nnz = ctypes.c_int64()
        self._check(self.lib.nsgpu_build_pattern(self.ctx, ctypes.byref(nnz)), "build_pattern")
        self.nnz = nnz.value
        self.n_rows = self.n_dofs
        if not fetch:
            return None
        indptr = np.empty(self.n_rows + 1, dtype=np.int64)
        indices = np.empty(self.nnz, dtype=np.int32)
        self._check(self.lib.nsgpu_get_pattern(self.ctx, _ptr(indptr), _ptr(indices)), "get_pattern")
        return indptr, indices

    # ------------------------------------------------------------------ multi-GPU set-up hooks (distributed.py)
    def build_pattern(self, extra_rows=None, extra_cols=None, colx_leader=None, colx_slot=None, colx_size=None):
        """(Re)build the pattern; the optional arguments are what other ranks' ghost rows add to rows this rank owns."""
        nx = 0 if colx_leader is None else len(colx_leader)
        la = np.ascontiguousarray(colx_leader if nx else np.zeros(0), dtype=np.int32)
        sl = np.ascontiguousarray(colx_slot if nx else np.zeros(0), dtype=np.int32)
        sz = np.ascontiguousarray(colx_size if nx else np.zeros(0), dtype=np.int32)
        self._check(self.lib.nsgpu_set_col_ghosts(self.ctx, nx, _ptr(la), _ptr(sl), _ptr(sz)), "set_col_ghosts")
        self.n_cols = self.n_dofs + nx
        if extra_rows is not None and len(extra_rows):
            er = np.ascontiguousarray(extra_rows, dtype=np.int32)
            ec = np.ascontiguousarray(extra_cols, dtype=np.int32)
            self._check(self.lib.nsgpu_add_pattern_entries(self.ctx, len(er), _ptr(er), _ptr(ec)), "add_pattern_entries")
        self.create_matrix(fetch=False)

    def get_rows(self, rows):
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        n = len(rows)
        start = np.zeros(n, dtype=np.int64)
        ptr = np.zeros(n + 1, dtype=np.int64)
        self._check(self.lib.nsgpu_get_rows(self.ctx, n, _ptr(rows), _ptr(start), _ptr(ptr), None, 0), "get_rows")
        idx = np.zeros(int(ptr[-1]), dtype=np.int32)
        self._check(self.lib.nsgpu_get_rows(self.ctx, n, _ptr(rows), _ptr(start), _ptr(ptr), _ptr(idx), len(idx)), "get_rows")
        return start, ptr, idx

    def comm_init(self, rank, size, unique_id):
        buf = ctypes.create_string_buffer(bytes(unique_id), 128)
        self._check(self.lib.nsgpu_comm_init(self.ctx, rank, size, buf), "comm_init")

    @staticmethod
    def comm_unique_id():
        lib = _lib.load()
        buf = ctypes.create_string_buffer(128)
        rc = lib.nsgpu_comm_unique_id(buf, 128)
        if rc != 0:
            raise _lib.NsgpuError("nsgpu_comm_unique_id failed: " + lib.nsgpu_last_error(None).decode())
        return buf.raw

    def set_halo(self, neigh, send_ptr, send_idx, recv_ptr, recv_idx):
        a = [np.ascontiguousarray(neigh, dtype=np.int32), np.ascontiguousarray(send_ptr, dtype=np.int64),
             np.ascontiguousarray(send_idx, dtype=np.int32), np.ascontiguousarray(recv_ptr, dtype=np.int64),
             np.ascontiguousarray(recv_idx, dtype=np.int32)]
        self._check(self.lib.nsgpu_set_halo(self.ctx, len(a[0]), *[_ptr(v) for v in a]), "set_halo")

    def set_row_exchange(self, neigh, send_ptr, send_pos, recv_ptr, recv_pos):
        a = [np.ascontiguousarray(neigh, dtype=np.int32), np.ascontiguousarray(send_ptr, dtype=np.int64),
             np.ascontiguousarray(send_pos, dtype=np.int64), np.ascontiguousarray(recv_ptr, dtype=np.int64),
             np.ascontiguousarray(recv_pos, dtype=np.int64)]
        self._check(self.lib.nsgpu_set_row_exchange(self.ctx, len(a[0]), *[_ptr(v) for v in a]), "set_row_exchange")

    def owned_nnz(self):
        n = ctypes.c_int64()
        self._check(self.lib.nsgpu_owned_nnz(self.ctx, ctypes.byref(n)), "owned_nnz")
        return n.value

    # ------------------------------------------------------------------ the hot path
    def _state(self, x):
        """The C ABI reads n_owned + n_ghost values from x_local (it cannot see lengths): check here.  A vector that only
        holds the owned entries (a petsc4py ``Vec.array``) is padded -- the ghost part is refreshed by the forward halo inside."""
        x = np.ascontiguousarray(x, dtype=np.float64).ravel()
        if x.size >= self.n_dofs:
            return x
        if x.size == self.n_owned:
            xg = np.zeros(self.n_dofs)
            xg[: self.n_owned] = x
            return xg
        raise ValueError(f"state vector has {x.size} entries; expected n_owned = {self.n_owned} or n_owned + n_ghost = {self.n_dofs}")

    def _out(self, out, n, what):
        if out is None:
            return np.empty(n)
        if not isinstance(out, np.ndarray) or out.dtype != np.float64 or not out.flags.c_contiguous or out.size < n:
            raise ValueError(f"{what}: need a C-contiguous float64 array with at least {n} entries")
        return out

    def residual(self, x, out=None):
        """F of NavierStokesChannelFlow.py:51-67 (assemble_vector + apply_lifting + reverse halo + set_bc)."""
        x = self._state(x)
        out = self._out(out, self.n_dofs, "residual output")
        self._check(self.lib.nsgpu_residual(self.ctx, _ptr(x), _ptr(out)), "residual")
        return out

    def jacobian(self, x, out=None, fetch=True):
        """J of NavierStokesChannelFlow.py:69-75.  fetch=False keeps the values on the device (MatShell)."""
        x = self._state(x)
        if fetch:
            out = self._out(out, self.nnz, "Jacobian values")
        self._check(self.lib.nsgpu_jacobian(self.ctx, _ptr(x), _ptr(out) if fetch else None), "jacobian")
        return out

    def jacobian_residual(self, x, vals_out=None, F_out=None, fetch_vals=True):
        x = self._state(x)
        F_out = self._out(F_out, self.n_dofs, "residual output")
        if fetch_vals:
            vals_out = self._out(vals_out, self.nnz, "Jacobian values")
        self._check(self.lib.nsgpu_jacobian_residual(self.ctx, _ptr(x), _ptr(vals_out) if fetch_vals else None, _ptr(F_out)), "jacobian_residual")
        return vals_out, F_out

    def mult(self, x, out=None):
        """PETSc MatMult with the last assembled Jacobian: y_owned = J x."""
        x = self._state(x)
        out = self._out(out, self.n_owned, "MatMult output")
        self._check(self.lib.nsgpu_spmv(self.ctx, _ptr(x), _ptr(out)), "spmv")
        return out

    def tfqmr(self, b, x0=None, rtol=1e-8, atol=0.0, max_it=1000, pc=4):
        """KSPSolve with KSPTFQMR on the resident Jacobian (NavierStokesChannelFlow.py:77, :282-285), fully on the device.
        pc: 0 none, 1 Jacobi, 4 4x4 vertex-block Jacobi (P1-P1 tets, else 1), 5 multicolour block ILU(0) (P1-P1 tets only),
        6 multicolour point ILU(0) (any space; NsgpuError "zero pivot" when a pivot vanishes), 7 point ILU(0) in the caller's
        order of the dofs, PETSc's natural order (any space; NsgpuError "zero pivot" naming the first such row).
        Returns (x_owned, info) with info = dict(its, rnorm = true ||b - A x||, r0norm)."""
        b = np.ascontiguousarray(b, dtype=np.float64)
        x = np.zeros(self.n_owned) if x0 is None else np.array(x0[: self.n_owned], dtype=np.float64)
        its, rn, r0 = ctypes.c_int(), ctypes.c_double(), ctypes.c_double()
        self._check(self.lib.nsgpu_tfqmr(self.ctx, _ptr(b), _ptr(x), float(rtol), float(atol), int(max_it), int(pc), 1 if x0 is None else 0,
                                         ctypes.byref(its), ctypes.byref(rn), ctypes.byref(r0)), "tfqmr")
        return x, {"its": its.value, "rnorm": rn.value, "r0norm": r0.value}

    def tfqmr_dev(self, b_dev, x_dev, rtol=1e-8, atol=0.0, max_it=1000, pc=4, zero_guess=True):
        """``tfqmr`` on device vectors (b: n_owned, x: n_cols doubles); pc as in ``tfqmr``."""
        its, rn, r0 = ctypes.c_int(), ctypes.c_double(), ctypes.c_double()
        self._check(self.lib.nsgpu_tfqmr_dev(self.ctx, b_dev, x_dev, float(rtol), float(atol), int(max_it), int(pc), 1 if zero_guess else 0,
                                             ctypes.byref(its), ctypes.byref(rn), ctypes.byref(r0)), "tfqmr_dev")
        return {"its": its.value, "rnorm": rn.value, "r0norm": r0.value}

    def ilu_apply(self, r, refactor=True):
        """PCApply of the multicolour block ILU(0) (pc = 5) on a host vector: z = U^-1 L^-1 r (owned entries)."""
        r = np.ascontiguousarray(r, dtype=np.float64)
        if r.size < self.n_owned:
            raise ValueError(f"ilu_apply needs the {self.n_owned} owned entries")
        z = np.empty(self.n_owned)
        self._check(self.lib.nsgpu_ilu_apply(self.ctx, 1 if refactor else 0, _ptr(r), _ptr(z)), "ilu_apply")
        return z

    def ilu_colours(self):
        """(elimination colour per owned vertex in the internal vertex order, number of colours)"""
        n = ctypes.c_int32()
        col = np.empty(self.n_owned // 4, dtype=np.int32)
        self._check(self.lib.nsgpu_ilu_colours(self.ctx, _ptr(col), ctypes.byref(n)), "ilu_colours")
        return col, n.value

    def pilu_apply(self, r, refactor=True):
        """PCApply of the multicolour point ILU(0) (pc = 6) on a host vector in the caller's numbering: z = U^-1 L^-1 r (owned entries)."""
        r = np.ascontiguousarray(r, dtype=np.float64)
        if r.size < self.n_owned:
            raise ValueError(f"pilu_apply needs the {self.n_owned} owned entries")
        z = np.empty(self.n_owned)
        self._check(self.lib.nsgpu_pilu_apply(self.ctx, 1 if refactor else 0, _ptr(r), _ptr(z)), "pilu_apply")
        return z

    def pilu_colours(self):
        """(elimination colour per owned dof in the caller's numbering, number of colours, number of velocity colours); the
        velocity colours are 0 .. n_velocity_colours - 1, the pressure colours come after them."""
        n, nv = ctypes.c_int32(), ctypes.c_int32()
        col = np.empty(self.n_owned, dtype=np.int32)
        self._check(self.lib.nsgpu_pilu_colours(self.ctx, _ptr(col), ctypes.byref(n), ctypes.byref(nv)), "pilu_colours")
        return col, n.value, nv.value

    def nilu_apply(self, r, refactor=True):
        """PCApply of the point ILU(0) in the caller's order (pc = 7) on a host vector in the caller's numbering: z = U^-1 L^-1 r."""
        r = np.ascontiguousarray(r, dtype=np.float64)
        if r.size < self.n_owned:
            raise ValueError(f"nilu_apply needs the {self.n_owned} owned entries")
        z = np.empty(self.n_owned)
        self._check(self.lib.nsgpu_nilu_apply(self.ctx, 1 if refactor else 0, _ptr(r), _ptr(z)), "nilu_apply")
        return z

    def nilu_depth(self):
        """(levels of the forward sweep, levels of the backward sweep) of the caller's-order ILU(0): rows on the longest path of
        each dependency DAG."""
        lo, up = ctypes.c_int32(), ctypes.c_int32()
        self._check(self.lib.nsgpu_nilu_depth(self.ctx, ctypes.byref(lo), ctypes.byref(up)), "nilu_depth")
        return lo.value, up.value

    def axpy_dev(self, a, x_dev, y_dev):
        self._check(self.lib.nsgpu_axpy_dev(self.ctx, float(a), x_dev, y_dev), "axpy_dev")

    def norm_dev(self, x_dev):
        out = ctypes.c_double()
        self._check(self.lib.nsgpu_norm_dev(self.ctx, x_dev, ctypes.byref(out)), "norm_dev")
        return out.value

    def dot_dev(self, x_dev, y_dev):
        out = ctypes.c_double()
        self._check(self.lib.nsgpu_dot_dev(self.ctx, x_dev, y_dev, ctypes.byref(out)), "dot_dev")
        return out.value

    def newton_dev(self, w_dev, rtol=1e-8, atol=1e-8, max_it=30, ksp_rtol=1e-8, ksp_max_it=2000, pc=4, work=None, linesearch="bt"):
        """Device-resident Newton iteration with the SNES settings of the reference (snes_rtol / snes_atol 1e-8, max_it 30,
        NavierStokesChannelFlow.py:286-291): F and J from the assembly kernels, dw from TFQMR, w -= lambda dw.
        ``linesearch``: "bt" = PETSc's default for newtonls (SNESLineSearchBT: sufficient decrease alpha = 1e-4 on
        1/2 ||F||^2, quadratic then cubic backtracking, steps clipped to [0.1, 0.5] of the previous one, at most 40), or
        "basic" (full steps).  ``pc``: the preconditioner of the TFQMR solves, as in ``tfqmr`` (6 and 7, the point ILU(0)s, work on
        every space).  Nothing but a few scalars crosses PCIe.  w_dev: n_cols doubles (state in / solution out)."""
        nbytes = 8 * self.n_cols
        owns = work is None
        F_dev, dw_dev = (self.dev_alloc(nbytes), self.dev_alloc(nbytes)) if owns else work[:2]
        Jd_dev = None
        hist = []
        try:
            self.jacobian_residual_dev(w_dev, True, F_dev)
            fn = self.norm_dev(F_dev)
            for it in range(max_it + 1):
                hist.append({"it": it, "fnorm": fn})
                if fn <= atol or (it > 0 and fn <= rtol * hist[0]["fnorm"]) or it == max_it:
                    break
                info = self.tfqmr_dev(F_dev, dw_dev, rtol=ksp_rtol, max_it=ksp_max_it, pc=pc)
                hist[-1].update(ksp_its=info["its"], ksp_rnorm=info["rnorm"])
                if linesearch == "basic":
                    self.axpy_dev(-1.0, dw_dev, w_dev)
                    self.jacobian_residual_dev(w_dev, True, F_dev)
                    fn = self.norm_dev(F_dev)
                    continue
                # initial slope of phi(lambda) = 1/2 ||F(w - lambda dw)||^2 at 0:  -F . (J dw)   (PETSc: MatMult + VecDot)
                if Jd_dev is None:
                    Jd_dev = self.dev_alloc(nbytes)
                self.spmv_dev(dw_dev, Jd_dev)
                slope = -self.dot_dev(F_dev, Jd_dev)
                if slope > 0.0:
                    slope = -slope
                if slope == 0.0:
                    slope = -1.0
                f0 = 0.5 * fn * fn
                lam, lam_prev, g_prev, steps = 1.0, None, None, 0
                self.axpy_dev(-lam, dw_dev, w_dev)
                while True:
                    self.jacobian_residual_dev(w_dev, True, F_dev)
                    gn = self.norm_dev(F_dev)
                    g = 0.5 * gn * gn
                    if (np.isfinite(g) and g <= f0 + 1e-4 * lam * slope) or steps >= 40:
                        break
                    if lam_prev is None or not np.isfinite(g):                     # quadratic fit through phi(0), phi'(0), phi(lam)
                        lam_new = -slope * lam * lam / (2.0 * (g - f0 - lam * slope)) if np.isfinite(g) else 0.5 * lam
                    else:                                                          # cubic through the last two trial points
                        t1, t2 = g - f0 - lam * slope, g_prev - f0 - lam_prev * slope
                        ca = (t1 / lam ** 2 - t2 / lam_prev ** 2) / (lam - lam_prev)
                        cb = (-lam_prev * t1 / lam ** 2 + lam * t2 / lam_prev ** 2) / (lam - lam_prev)
                        if ca == 0.0:
                            lam_new = -slope / (2.0 * cb)
                        else:
                            disc = cb * cb - 3.0 * ca * slope
                            lam_new = 0.5 * lam if disc < 0.0 else ((-cb + np.sqrt(disc)) / (3.0 * ca) if cb <= 0.0 else -slope / (cb + np.sqrt(disc)))
                    lam_new = min(max(lam_new, 0.1 * lam), 0.5 * lam)
                    lam_prev, g_prev = lam, g
                    self.axpy_dev(lam - lam_new, dw_dev, w_dev)                    # w = w0 - lam_new dw
                    lam = lam_new
                    steps += 1
                hist[-1].update(lam=lam, ls_steps=steps)
                fn = gn
        finally:
            if owns:
                self.dev_free(F_dev); self.dev_free(dw_dev)
            if Jd_dev is not None:
                self.dev_free(Jd_dev)
        return hist

    # ------------------------------------------------------------------ point evaluation / non-matching interpolation
    def eval(self, w, points, tol=1e-12, padding=0.0):
        """Function.eval of the mixed function w (caller numbering) at points (n, 3): returns (values (n, gdim + 1) = velocity
        components then pressure, cells (n,) int32).  cells: c inside cell c (lowest-numbered cell with every barycentric coordinate
        >= -tol), -2 - c extrapolated from the nearest cell c within ``padding``, -1 outside (values 0).

        On a context with a communicator the call is collective: every rank passes its own points (any number, also none) and the
        same tol and padding; only owned cells hold points.  A point inside an owned cell of the calling rank stays there; otherwise
        the lowest rank with an owned cell holding it answers; otherwise (padding > 0) the nearest owned cell over all ranks within
        ``padding`` (ties to the lower rank).  Cell numbers are those of the answering rank."""
        w = self._state(w)
        p = np.ascontiguousarray(points, dtype=np.float64)
        if p.ndim != 2 or p.shape[1] != 3:
            raise ValueError("points must be (n, 3)")
        values = np.empty((p.shape[0], self.gdim + 1))
        cells = np.empty(p.shape[0], dtype=np.int32)
        self._check(self.lib.nsgpu_eval(self.ctx, _ptr(w), p.shape[0], _ptr(p), float(tol), float(padding), _ptr(values), _ptr(cells)), "eval")
        return values, cells

    def eval_dev(self, w_dev, n, points_dev, values_dev, cells_dev=None, tol=1e-12, padding=0.0):
        """``eval`` on device arrays (w: n_owned + n_ghost, points: n x 3, values: n x (gdim + 1) doubles, cells: n int32 or None);
        asynchronous on the context's stream on one rank; collective and synchronous on several (see ``eval``)."""
        self._check(self.lib.nsgpu_eval_dev(self.ctx, w_dev, int(n), points_dev, float(tol), float(padding), values_dev, cells_dev), "eval_dev")

    def interpolate_nonmatching(self, src, w_src, tol=1e-12, padding=0.0):
        """Function.interpolate_nonmatching onto this (destination) space: every dof gets the source function ``w_src`` of the
        NSAssembler ``src`` (another mesh of the same gdim, any velocity degree) evaluated at the dof's node, with the location rule
        of ``eval``.  Returns (w (n_owned + n_ghost), info = dict(n_extrapolated, n_outside) counted over destination nodes).

        On several ranks (both contexts with communicators of the same size, the destination with its halo plan) the call is
        collective: each rank's owned destination nodes are evaluated over the source's ranks, the ghost entries are refreshed from
        their owners, and the counts are summed over the ranks."""
        w_src = src._state(w_src)
        w = np.empty(self.n_dofs)
        ne, no = ctypes.c_int64(), ctypes.c_int64()
        self._check(self.lib.nsgpu_interpolate(src.ctx, _ptr(w_src), self.ctx, _ptr(w), float(tol), float(padding), ctypes.byref(ne), ctypes.byref(no)),
                    "interpolate")
        return w, {"n_extrapolated": ne.value, "n_outside": no.value}

    def interpolate_nonmatching_dev(self, src, w_src_dev, w_dev, tol=1e-12, padding=0.0, counts_dev=None):
        """``interpolate_nonmatching`` on device vectors, asynchronous on this context's stream (which first waits for src's);
        counts_dev: None or a device pointer to two int64 (extrapolated, outside).  Synchronous on several ranks."""
        ne = no = None
        if counts_dev is not None:
            base = counts_dev.value if isinstance(counts_dev, ctypes.c_void_p) else int(counts_dev)
            ne, no = ctypes.c_void_p(base), ctypes.c_void_p(base + 8)
        self._check(self.lib.nsgpu_interpolate_dev(src.ctx, w_src_dev, self.ctx, w_dev, float(tol), float(padding), ne, no), "interpolate_dev")

    # ------------------------------------------------------------------ boundary functionals over tagged facets
    def set_facets(self, cells, local_facets, tags):
        """Integration domain of ``ds(subdomain_data=facet_tags)``: one (cell, local facet, tag) per exterior facet (dolfinx's
        compute_integration_domains; local facet i is opposite vertex i; ``gmsh_io.facet_integration_domain`` builds them from
        tagged facets).  Tags in [0, 64).  Facets of ghost cells are integrated by the owning rank.  Returns n_tags = max tag + 1."""
        c = np.ascontiguousarray(cells, dtype=np.int32).ravel()
        lf = np.ascontiguousarray(local_facets, dtype=np.int32).ravel()
        t = np.ascontiguousarray(tags, dtype=np.int32).ravel()
        if not (len(c) == len(lf) == len(t)):
            raise ValueError("cells, local_facets and tags must have the same length")
        n = ctypes.c_int32()
        self._check(self.lib.nsgpu_set_facets(self.ctx, len(c), _ptr(c), _ptr(lf), _ptr(t), ctypes.byref(n)), "set_facets")
        self.n_tags = n.value
        return self.n_tags

    def facet_integrals(self, w):
        """Per tag: [area, int u.n, int p n (gdim), int (grad u) n (gdim), int (grad u)^T n (gdim)] with n the outward unit normal,
        (grad u)_ij = du_i/dx_j, no viscosity applied; returns (n_tags, 2 + 3 gdim).  The force of the fluid on the tagged
        boundary by the Cauchy stress is -(nu (row[2+g:2+2g] + row[2+2g:]) - row[2:2+g])."""
        w = self._state(w)
        out = np.empty((self.n_tags, 2 + 3 * self.gdim))
        self._check(self.lib.nsgpu_facet_integrals(self.ctx, _ptr(w), _ptr(out)), "facet_integrals")
        return out

    def facet_integrals_dev(self, w_dev, out_dev):
        """``facet_integrals`` on device arrays (out: n_tags x (2 + 3 gdim) doubles); asynchronous on the context's stream."""
        self._check(self.lib.nsgpu_facet_integrals_dev(self.ctx, w_dev, out_dev), "facet_integrals_dev")

    def reaction(self, w):
        """Per tag and velocity component: the unconstrained residual of the current form (no lifting, no set_bc) summed over the
        velocity dofs of the tagged facets (vertices, plus edges for P2); returns (n_tags, gdim).  The force of the fluid on the
        tagged boundary is -reaction (the consistent drag / lift)."""
        w = self._state(w)
        out = np.empty((self.n_tags, self.gdim))
        self._check(self.lib.nsgpu_reaction(self.ctx, _ptr(w), _ptr(out)), "reaction")
        return out

    def reaction_dev(self, w_dev, out_dev):
        """``reaction`` on device arrays (out: n_tags x gdim doubles); asynchronous on the context's stream."""
        self._check(self.lib.nsgpu_reaction_dev(self.ctx, w_dev, out_dev), "reaction_dev")

    def values_norm(self):
        """Frobenius norm of the resident Jacobian over all ranks' owned rows (a partition-independent checksum)."""
        out = ctypes.c_double()
        self._check(self.lib.nsgpu_values_norm(self.ctx, ctypes.byref(out)), "values_norm")
        return out.value

    def set_values(self, vals):
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        self._check(self.lib.nsgpu_set_values(self.ctx, _ptr(vals)), "set_values")

    def get_values(self):
        out = np.empty(self.nnz)
        self._check(self.lib.nsgpu_get_values(self.ctx, _ptr(out)), "get_values")
        return out

    def values_dev(self):
        """Device pointer of the CSR values in the caller's order (the resident array itself unless the library renumbered)."""
        p = ctypes.c_void_p()
        self._check(self.lib.nsgpu_values_dev(self.ctx, ctypes.byref(p)), "values_dev")
        return p

    def get_value_range(self, start, n, vals_dev=None):
        """CSR values [start, start + n) of the resident matrix (rows of huge matrices without fetching 16 GB)."""
        p = self.values_dev() if vals_dev is None else vals_dev
        out = np.empty(int(n))
        self.d2h(out, ctypes.c_void_p(p.value + 8 * int(start)))
        return out

    def timers(self):
        ms = (ctypes.c_double * 8)()
        self._check(self.lib.nsgpu_timers(self.ctx, ms, 8), "timers")
        keys = ["jacobian_residual", "residual", "spmv", "halo", "h2d", "d2h", "pattern", "spare"]
        return dict(zip(keys, list(ms)))

    def last_kernel_name(self):
        return self.lib.nsgpu_last_kernel_name(self.ctx).decode()

    def last_spmv_name(self):
        return self.lib.nsgpu_last_spmv_name(self.ctx).decode()

    def fp64_peak(self):
        """Measured DFMA TFLOP/s of this GPU (live micro-benchmark)."""
        out = ctypes.c_double()
        self._check(self.lib.nsgpu_fp64_peak(self.ctx, ctypes.byref(out)), "fp64_peak")
        return out.value

    def launch_count(self):
        return int(self.lib.nsgpu_launch_count(self.ctx))

    # ------------------------------------------------------------------ device-resident variants
    def dev_alloc(self, nbytes):
        p = ctypes.c_void_p()
        self._check(self.lib.nsgpu_dev_alloc(self.ctx, int(nbytes), ctypes.byref(p)), "dev_alloc")
        return p

    def dev_free(self, p):
        self._check(self.lib.nsgpu_dev_free(self.ctx, p), "dev_free")

    def h2d(self, dptr, arr):
        arr = np.ascontiguousarray(arr)
        self._check(self.lib.nsgpu_memcpy_h2d(self.ctx, dptr, _ptr(arr), arr.nbytes), "h2d")

    def d2h(self, arr, dptr):
        self._check(self.lib.nsgpu_memcpy_d2h(self.ctx, _ptr(arr), dptr, arr.nbytes), "d2h")

    def jacobian_residual_dev(self, x_dev, want_jacobian=True, F_dev=None):
        self._check(self.lib.nsgpu_jacobian_residual_dev(self.ctx, x_dev, 1 if want_jacobian else 0, F_dev), "jacobian_residual_dev")

    def spmv_dev(self, x_dev, y_dev):
        self._check(self.lib.nsgpu_spmv_dev(self.ctx, x_dev, y_dev), "spmv_dev")

    def sync(self):
        self._check(self.lib.nsgpu_sync(self.ctx), "sync")

    def timer_start(self):
        self._check(self.lib.nsgpu_timer_start(self.ctx), "timer_start")

    def timer_stop(self):
        ms = ctypes.c_double()
        self._check(self.lib.nsgpu_timer_stop(self.ctx, ctypes.byref(ms)), "timer_stop")
        return ms.value

    def pinned_empty(self, n, dtype=np.float64):
        """NumPy array backed by page-locked host memory (cudaMallocHost)."""
        nbytes = int(n) * np.dtype(dtype).itemsize
        p = ctypes.c_void_p()
        rc = self.lib.nsgpu_host_alloc_pinned(nbytes, ctypes.byref(p))
        if rc != 0:
            raise _lib.NsgpuError("cudaMallocHost failed")
        buf = (ctypes.c_char * nbytes).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(n))
        self._pinned = getattr(self, "_pinned", []) + [p]
        return arr

    def last_kernel_ms(self):
        ms = ctypes.c_double()
        self._check(self.lib.nsgpu_last_kernel_ms(self.ctx, ctypes.byref(ms)), "last_kernel_ms")
        return ms.value


def _as_array(v):
    """NumPy view of a NumPy array or of a petsc4py Vec.  A ghosted Vec is opened through its local form (owned + ghost
    entries, what dolfinx's ``x.localForm()`` gives, NavierStokesChannelFlow.py:57-60); a plain Vec through ``.array``."""
    if isinstance(v, np.ndarray):
        return v
    gl = getattr(v, "getLocalForm", None) or getattr(v, "localForm", None)
    if gl is not None:
        try:
            loc = gl()
            arr = getattr(loc, "array", None)
            if arr is None and hasattr(loc, "__enter__"):
                arr = loc.__enter__().array
            if arr is not None:
                return arr
        except Exception:
            pass
    return v.array


def _fill_matrix(J, asm, pattern, vals, local_to_global=None):
    """Hand the owned rows of the CSR triple to a petsc4py-like Mat.  Column indices of the pattern are LOCAL (owned, then
    ghosts, then column ghosts): ``setValuesLocalCSR`` takes them as they are (dolfinx's create_matrix installs the
    local-to-global maps); ``setValuesCSR`` wants global columns, so a map is required as soon as ghosts exist."""
    indptr, indices = pattern
    n = asm.n_owned
    if int(indptr[n]) > np.iinfo(np.int32).max:
        raise OverflowError(f"{int(indptr[n])} entries in the owned rows do not fit PETSc's 32-bit PetscInt row pointers; "
                            "use more ranks or the MatShell mode (values stay on the device)")
    ip = indptr[: n + 1].astype(np.int32)
    ix, v = indices[: indptr[n]], vals[: indptr[n]]
    J.zeroEntries()
    if hasattr(J, "setValuesLocalCSR") and local_to_global is None:
        J.setValuesLocalCSR(ip, ix, v)
    else:
        if local_to_global is not None:
            ix = np.asarray(local_to_global)[ix].astype(np.int32)
        elif getattr(asm, "n_cols", asm.n_dofs) > asm.n_owned:
            raise ValueError("Mat.setValuesCSR needs global column indices: pass local_to_global (owned + ghost + column ghosts)")
        J.setValuesCSR(ip, ix, v)
    J.assemble()


class NonlinearPDE_SNESProblem:
    """Same role and callback signatures as the class of that name in
    NavierStokes/NavierStokesChannelFlow.py:40-75.  ``F``/``J`` accept NumPy arrays or petsc4py objects:
    a Vec is accessed through its ghosted local form (or ``.array``); a Mat is filled with ``setValuesLocalCSR`` /
    ``setValuesCSR``, otherwise ``J`` is treated as the CSR value array itself."""

    def __init__(self, assembler, u=None, fuse=True, local_to_global=None):
        self.asm = assembler
        self.u = u                       # optional mirror of the state vector (self.u of the reference)
        self.pattern = None
        self.local_to_global = local_to_global
        # SNES evaluates F and then J at the same iterate: with fuse the residual call assembles the Jacobian in the same
        # pass (it stays on the device) and the Jacobian call that follows recognises the state and reuses it.
        self.asm.set_option("fuse_fj", 1 if fuse else 0)

    def create_matrix(self):
        self.pattern = self.asm.create_matrix()
        return self.pattern

    def F(self, snes, x, F):
        """Assemble residual vector (x.ghostUpdate, assemble_vector, apply_lifting, F.ghostUpdate, set_bc)."""
        xa = _as_array(x)
        if self.u is not None:
            ua = _as_array(self.u)
            ua[: xa.size] = xa[: ua.size]     # x.copy(self.u.x.petsc_vec)
        Fa = _as_array(F)
        res = self.asm.residual(xa)
        Fa[: self.asm.n_owned] = res[: self.asm.n_owned]
        if Fa.size > self.asm.n_owned:
            Fa[self.asm.n_owned:] = 0.0   # ghost part of F is zero after the reverse scatter

    def J(self, snes, x, J, P=None):
        """Assemble Jacobian matrix (zeroEntries, assemble_matrix with bcs, assemble)."""
        xa = _as_array(x)
        vals = self.asm.jacobian(xa)
        if hasattr(J, "setValuesCSR") or hasattr(J, "setValuesLocalCSR"):
            _fill_matrix(J, self.asm, self.pattern if self.pattern is not None else self.create_matrix(), vals, self.local_to_global)
        else:
            _as_array(J)[:] = vals


class NonlinearProblem:
    """The three callbacks dolfinx.nls.petsc.NewtonSolver takes from dolfinx.fem.petsc.NonlinearProblem
    (LidDrivenFlow/LidDrivenNavierStokesFlow.py:150-153): ``form(x)`` (ghost update before an assembly), ``F(x, b)``
    (assemble_vector + apply_lifting(x0 = x, alpha = -1) + ghost reverse-add + set_bc(x0 = x, alpha = -1)) and ``J(x, A)``
    (zeroEntries + assemble_matrix(bcs) + assemble).  ``x`` / ``b``: NumPy arrays or petsc4py Vecs; ``A``: a petsc4py-like
    Mat or the CSR value array.  ``solver.setF(problem.F, b); solver.setJ(problem.J, A); solver.set_form(problem.form)``."""

    def __init__(self, assembler, u=None, local_to_global=None):
        self.asm = assembler
        self.u = u
        self.local_to_global = local_to_global
        self.pattern = None
        self.asm.set_option("fuse_fj", 1)      # NewtonSolver calls F then J at the same iterate

    def create_matrix(self):
        self.pattern = self.asm.create_matrix()
        return self.pattern

    def form(self, x):
        """x.ghostUpdate(INSERT, FORWARD): the library refreshes the ghost entries itself inside F / J (halo over NCCL), so
        there is nothing to do beyond keeping the state mirror in step."""
        if self.u is not None:
            xa, ua = _as_array(x), _as_array(self.u)
            ua[: xa.size] = xa[: ua.size]

    def F(self, x, b):
        ba = _as_array(b)
        res = self.asm.residual(_as_array(x))
        ba[: self.asm.n_owned] = res[: self.asm.n_owned]
        if ba.size > self.asm.n_owned:
            ba[self.asm.n_owned:] = 0.0

    def J(self, x, A):
        vals = self.asm.jacobian(_as_array(x))
        if hasattr(A, "setValuesCSR") or hasattr(A, "setValuesLocalCSR"):
            _fill_matrix(A, self.asm, self.pattern if self.pattern is not None else self.create_matrix(), vals, self.local_to_global)
        else:
            _as_array(A)[:] = vals


def newton_solve(problem, x, linear_solve, rtol=1e-9, atol=1e-10, max_it=50, relaxation=1.0, criterion="incremental", A=None, b=None):
    """The iteration dolfinx's NewtonSolver runs on a NonlinearProblem (LidDrivenNavierStokesFlow.py:152-169):
    form, F, J, solve J dx = F, x -= relaxation dx, until the incremental (||dx|| < rtol ||dx_0|| or < atol) or residual
    criterion holds.  ``linear_solve(A_values, b_owned) -> dx_owned`` stands for the KSP (preonly + LU in the lid-driven
    script).  x: NumPy array (owned + ghost); returns (iterations, converged)."""
    asm = problem.asm
    b = np.zeros(asm.n_dofs) if b is None else b
    A = np.zeros(asm.nnz) if A is None else A
    r0 = None
    for it in range(1, max_it + 1):
        problem.form(x)
        problem.F(x, b)
        problem.J(x, A)
        dx = linear_solve(A, b[: asm.n_owned])
        x[: asm.n_owned] -= relaxation * dx
        r = float(np.linalg.norm(dx)) if criterion == "incremental" else float(np.linalg.norm(b[: asm.n_owned]))
        r0 = r if r0 is None else r0
        if r < atol or (r0 > 0 and r / r0 < rtol):
            return it, True
    return max_it, False
