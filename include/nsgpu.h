/*
 * nsgpu.h -- C ABI of libnsgpu.so: B200-native (sm_100a) residual / Jacobian assembly of the
 * stabilized incompressible Navier-Stokes weak forms, CSR sparsity construction, CSR SpMV and
 * ghost (halo) exchange.  Plain pointers and sizes only; no C++ / torch types cross this boundary.
 *
 * Each entry point names the reference interface it replaces (file:line into the reference
 * repository mungerct/Stabilized_Navier_Stokes_Flow_FEniCSx).  "dolfinx" below means the un-vendored
 * fenics-dolfinx 0.9.0 the reference scripts call.
 *
 * Conventions
 *   - every function returns 0 on success or a negative NSGPU_E* code; the message is available
 *     from nsgpu_last_error().  Nothing throws or aborts across the ABI.
 *   - one context per GPU per host thread/process (= one MPI rank = one mesh partition).  Calls on a
 *     context are serialised on its CUDA stream and are synchronous on return unless noted.
 *   - the caller owns every host array; set_* calls copy to the device; x / F / vals arguments of the
 *     compute calls are borrowed for the duration of the call.
 *   - *_dev variants take device pointers (zero-copy; used by the device-resident Krylov loop and the
 *     throughput benchmark).
 *   - array layout is exactly what dolfinx exposes: geometry x (n_nodes x 3, padded), geometry dofmap
 *     (cells x nodes_per_cell int32), W.dofmap.list (cells x ndofs_cell int32, block size 1), owned
 *     dofs first then ghosts; owned cells first then ghost cells.
 */
#ifndef NSGPU_H
#define NSGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nsgpu_ctx nsgpu_ctx;

enum {
  NSGPU_OK = 0,
  NSGPU_EINVAL = -1,   /* bad argument / call order */
  NSGPU_ECUDA = -2,    /* CUDA runtime error (no device, OOM, launch failure) */
  NSGPU_EUNSUPPORTED = -3,
  NSGPU_ENCCL = -4,
  NSGPU_EPATTERN = -5, /* element entry outside the sparsity pattern / row too long */
  NSGPU_ENONFINITE = -6, /* the assembled residual holds NaN / Inf (diverged state or degenerate cell); see option "check_finite" */
  NSGPU_EZEROPIVOT = -7  /* the point ILU(0) factorisation met a zero or non-finite pivot (PETSc: factor zero-pivot failure) */
};

/* weak-form flavours (nsgpu_set_form) */
enum {
  NSGPU_FORM_GMETRIC = 0, /* G-metric SUPG/PSPG/LSIC NS: NavierStokes/NavierStokesChannelFlow.py:220-251 */
  NSGPU_FORM_UGN = 1,     /* h-based UGN SUPG/PSPG/LSIC NS: LidDrivenFlow/LidDrivenNavierStokesFlow.py:112-143 */
  NSGPU_FORM_STOKES = 2   /* alpha grad u:grad v + sp(-p div v + q div u) + beta h^2 grad p.grad q:
                             NavierStokesChannelFlow.py:160-172, LidDrivenNavierStokesFlow.py:86-99,
                             StokesFlow/DuctStokesFlow.py:188-192 */
};

/* assembly kernel selection (nsgpu_set_option "kernel") */
enum {
  NSGPU_KERNEL_AUTO = 0,
  NSGPU_KERNEL_GENERIC = 1,  /* one thread per (cell, test dof), direct quadrature, any element/form */
  NSGPU_KERNEL_FAST = 2      /* factorised P1-P1 tet G-metric kernels */
};

int nsgpu_version(void);

/* Lifetime.  device = CUDA ordinal. */
int nsgpu_create(nsgpu_ctx** out, int device);
int nsgpu_destroy(nsgpu_ctx* ctx);
/* Last error text of ctx (or of the failed nsgpu_create when ctx == NULL). Never NULL. */
const char* nsgpu_last_error(const nsgpu_ctx* ctx);

/* mesh.geometry.x / mesh.geometry.dofmap of the rank-local mesh produced by
 * gmshio.model_to_mesh (NavierStokesChannelFlow.py:111) or create_rectangle
 * (LidDrivenNavierStokesFlow.py:29-30).  gdim = 2 (triangles) or 3 (tetrahedra); affine cells. */
int nsgpu_set_mesh(nsgpu_ctx* ctx, int gdim, int64_t n_nodes, const double* x /* n_nodes*3 */,
                   int64_t n_cells_owned, int64_t n_cells_total, const int32_t* x_dofmap /* n_cells_total*(gdim+1) */);

/* W = functionspace(msh, mixed_element([P_vdeg^gdim, P1])) (NavierStokesChannelFlow.py:128-129):
 * W.dofmap.list (block size 1; cell-local order = velocity node-major, components interleaved, then
 * pressure) and the index-map sizes.  vdeg = 1 (stabilized P1-P1) or 2 (Taylor-Hood P2-P1). */
int nsgpu_set_space(nsgpu_ctx* ctx, int vdeg, const int32_t* dofmap /* n_cells_total*ndofs_cell */,
                    int64_t n_dofs_owned, int64_t n_dofs_ghost);

/* The UFL form text of define_navier_stokes_form (NavierStokesChannelFlow.py:220-266) reduced to its
 * parameters: nu = 1/Re (:223), Ci = 36 (:237).  alpha/sp/beta are used by NSGPU_FORM_STOKES only.
 * May be called again at any time (Reynolds sweep of run_all_RE.sh) without rebuilding anything. */
int nsgpu_set_form(nsgpu_ctx* ctx, int flavour, double nu, double Ci, double alpha, double sp, double beta);

/* bcs = [bc_wall, bc_inlet_1, bc_inlet_2, bc_outlet] (NavierStokesChannelFlow.py:134-146): one
 * (dofs, values) segment per dirichletbc object, in list order; a dof may appear in several objects
 * (multiplicity is preserved: assemble_matrix adds 1.0 on the diagonal per object). */
int nsgpu_set_bcs(nsgpu_ctx* ctx, int n_bc, const int64_t* bc_ptr /* n_bc+1 */, const int32_t* bc_dofs, const double* bc_vals);

/* create_matrix(problem.a) (NavierStokesChannelFlow.py:272): CSR sparsity = union over owned cells of
 * dofs x dofs, rows = owned + ghost dofs, columns sorted by local index.  nnz_out may be NULL. */
int nsgpu_build_pattern(nsgpu_ctx* ctx, int64_t* nnz_out);
int nsgpu_get_pattern(nsgpu_ctx* ctx, int64_t* indptr /* n_rows+1 */, int32_t* indices /* nnz */);
int nsgpu_pattern_sizes(nsgpu_ctx* ctx, int64_t* n_rows, int64_t* nnz);
/* Entries held in the rows this rank owns (= indptr[n_dofs_owned]); what MatMult streams. */
int nsgpu_owned_nnz(nsgpu_ctx* ctx, int64_t* nnz_owned);

/* NonlinearPDE_SNESProblem.F (NavierStokesChannelFlow.py:51-67): forward halo of x, zero F,
 * assemble_vector(F, L), apply_lifting(F, [a], [bc], [x], -1.0), reverse halo-add, set_bc(F, bc, x, -1.0).
 * x_local: n_owned + n_ghost values (ghost part is overwritten by the forward halo when a communicator
 * is attached).  F_local: n_owned + n_ghost values out (owned part meaningful). */
int nsgpu_residual(nsgpu_ctx* ctx, const double* x_local, double* F_local);

/* NonlinearPDE_SNESProblem.J (NavierStokesChannelFlow.py:69-75): J.zeroEntries(),
 * assemble_matrix(J, a, bcs=bc) incl. BC diagonals, J.assemble() (ghost rows shipped to owners).
 * vals (nnz, CSR order of nsgpu_get_pattern) may be NULL: the matrix then stays on the device for
 * nsgpu_spmv (MatShell use). */
int nsgpu_jacobian(nsgpu_ctx* ctx, const double* x_local, double* vals);

/* One pass producing both (what SNES needs at every Newton iterate).  The Jacobian is always assembled;
 * vals == NULL keeps it on the device, F_local == NULL skips the residual. */
int nsgpu_jacobian_residual(nsgpu_ctx* ctx, const double* x_local, double* vals, double* F_local);

/* MatMult inside KSPTFQMR (snes.getKSP().setType('tfqmr'), NavierStokesChannelFlow.py:282):
 * y_owned = J x with the Jacobian of the last nsgpu_jacobian*; x: n_owned (+ghost, refreshed by the halo). */
int nsgpu_spmv(nsgpu_ctx* ctx, const double* x_local, double* y_owned);

/* KSPSolve with KSPTFQMR (snes_ksp_type 'tfqmr', NavierStokesChannelFlow.py:77, :282-283; KSP rtol :285) on the
 * Jacobian of the last nsgpu_jacobian*: transpose-free QMR, right-preconditioned, every vector and scalar
 * device-resident; two MatMults per iteration, dot products reduced over all ranks (ncclAllReduce).
 *   pc: 0 none, 1 Jacobi, 4 = 4x4 block Jacobi over the dofs of one P1-P1 vertex (falls back to 1 elsewhere),
 *       5 = multicolour 4x4-block ILU(0), block Jacobi over the ranks (P1-P1 tets; NSGPU_EUNSUPPORTED elsewhere),
 *       6 = multicolour point ILU(0), block Jacobi over the ranks, any space (velocity dofs eliminated before pressure dofs;
 *           NSGPU_EZEROPIVOT on a zero pivot).
 *   zero_guess != 0 ignores the incoming x (PETSc's default initial guess).
 * Stops when the quasi-residual bound tau*sqrt(m+1) <= max(rtol * ||b||, atol) (PETSc's default test) or after max_it iterations;
 * *its_out = iterations done, *rnorm_out = TRUE residual norm ||b - A x|| at exit, *r0norm_out = ||b - A x0||.
 * b: n_owned values; x: host variant n_owned in/out, device variant n_owned + n_ghost (+ column ghosts) values. */
int nsgpu_tfqmr(nsgpu_ctx* ctx, const double* b_owned, double* x_owned, double rtol, double atol, int max_it, int pc, int zero_guess,
                int* its_out, double* rnorm_out, double* r0norm_out);
int nsgpu_tfqmr_dev(nsgpu_ctx* ctx, const double* b_owned_dev, double* x_local_dev, double rtol, double atol, int max_it, int pc,
                    int zero_guess, int* its_out, double* rnorm_out, double* r0norm_out);
/* The two vector operations a device-resident Newton loop needs besides F, J and the solve (VecAXPY / VecNorm on
 * the owned entries; the norm is reduced over all ranks): y += a x, *out = ||x||_2. */
/* Multicolour 4x4-block ILU(0) of the resident Jacobian (pc = 5 of nsgpu_tfqmr*; the class of PETSc's default PC for
 * snes_ksp_type = 'tfqmr', NavierStokesChannelFlow.py:282-291: ILU(0), block Jacobi over the ranks).  nsgpu_ilu_apply = PCApply on
 * host vectors (owned entries): z = U^-1 L^-1 r; refactor != 0 factorises the current values first (always done when there is no
 * factorisation yet).  nsgpu_ilu_colours: the elimination colour of every owned vertex in the library's internal vertex order
 * (= the caller's order when its numbering is vertex-blocked, dof = 4 vertex + component) and the number of colours; for tests. */
int nsgpu_ilu_apply(nsgpu_ctx* ctx, int refactor, const double* r_owned, double* z_owned);
int nsgpu_ilu_colours(nsgpu_ctx* ctx, int32_t* colour /* n_owned / 4, may be NULL */, int32_t* n_colours);
/* Multicolour point ILU(0) of the resident Jacobian (pc = 6 of nsgpu_tfqmr*): PETSc's default PC on the AIJ matrix of the mixed space
 * (block size 1), block Jacobi over the ranks.  The owned dofs are coloured on the graph of the CSR pattern, velocity dofs first and
 * pressure dofs with colours numbered after every velocity colour, and eliminated in the order (colour, row): every pressure pivot
 * then carries the local Schur complement, so the unstabilised Taylor-Hood Stokes operator (zero pressure diagonal) factorises.
 * nsgpu_pilu_apply = PCApply on host vectors in the caller's numbering: z = U^-1 L^-1 r; refactor != 0 factorises the current values
 * first (always done when there is no factorisation yet); NSGPU_EZEROPIVOT names the row of a zero pivot.  nsgpu_pilu_colours: the
 * elimination colour of every owned dof in the caller's numbering, the number of colours and how many of them are velocity colours
 * (within a colour the order does not change the factor); for tests. */
int nsgpu_pilu_apply(nsgpu_ctx* ctx, int refactor, const double* r_owned, double* z_owned);
int nsgpu_pilu_colours(nsgpu_ctx* ctx, int32_t* colour /* n_owned, may be NULL */, int32_t* n_colours, int32_t* n_velocity_colours);
int nsgpu_axpy_dev(nsgpu_ctx* ctx, double a, const double* x_dev, double* y_dev);
int nsgpu_norm_dev(nsgpu_ctx* ctx, const double* x_dev, double* out);
/* VecDot over the owned entries, reduced over all ranks (the initial slope F . J dx of SNES' backtracking line search). */
int nsgpu_dot_dev(nsgpu_ctx* ctx, const double* x_dev, const double* y_dev, double* out);

/* Frobenius norm of the resident Jacobian over the rows owned by all ranks (MatNorm(NORM_FROBENIUS)); a partition-independent
 * checksum of an assembly.  Collective. */
int nsgpu_values_norm(nsgpu_ctx* ctx, double* out);

/* Replace the matrix values (e.g. to use nsgpu_spmv with a matrix assembled elsewhere). */
int nsgpu_set_values(nsgpu_ctx* ctx, const double* vals);
int nsgpu_get_values(nsgpu_ctx* ctx, double* vals);

/* Device-pointer variants: same semantics, pointers are device memory of ctx's GPU; asynchronous on
 * ctx's stream (use nsgpu_sync or the stream). */
int nsgpu_jacobian_residual_dev(nsgpu_ctx* ctx, double* x_local_dev, int want_jacobian, double* F_local_dev);
int nsgpu_spmv_dev(nsgpu_ctx* ctx, double* x_local_dev, double* y_owned_dev);
int nsgpu_values_dev(nsgpu_ctx* ctx, double** vals_dev);
int nsgpu_sync(nsgpu_ctx* ctx);
void* nsgpu_stream(nsgpu_ctx* ctx); /* cudaStream_t */

/* Device memory helpers for hosts without a CUDA binding (ctypes). */
int nsgpu_dev_alloc(nsgpu_ctx* ctx, int64_t bytes, void** out);
int nsgpu_dev_free(nsgpu_ctx* ctx, void* p);
int nsgpu_memcpy_h2d(nsgpu_ctx* ctx, void* dst_dev, const void* src_host, int64_t bytes);
int nsgpu_memcpy_d2h(nsgpu_ctx* ctx, void* dst_host, const void* src_dev, int64_t bytes);
int nsgpu_host_alloc_pinned(int64_t bytes, void** out);
int nsgpu_host_free_pinned(void* p);

/* Options: "kernel" (NSGPU_KERNEL_*); for the factorised P1-P1 kernels "ws" (1, default: warp-specialised kernel -- two
 * compute warpgroups and a gather warpgroup per SM, tables by cp.async.bulk) and "pipe" (1: software-pipelined 2-CTA kernel
 * when "ws" is off or does not apply; both 0: plain tile kernel); "rowown" (atomics-free row-owner kernel for the spaces /
 * forms without a factorised kernel: 0 never, 1 default: P2-P1 spaces, 2 every such space) and "rowown_lean" (1, default: the
 * G-metric form on tetrahedra through row-side records + a short mixed part; 0: unsplit entity blocks); "fuse_fj", "stream_host",
 * "stream_chunks", "spmv_blocks", "spmv_wide" (1, default: 256-bit loads in the vertex-blocked MatMult when rows and vectors are
 * 32-byte aligned); "overlap" (0, default: ghost-row / ghost-residual exchanges after the assembly kernel; 1: ghost tiles first,
 * exchanges on a second stream beside the interior tiles) and "sm_reserve" (SMs left to the exchange kernels when "overlap" is on);
 * "check_finite" (1, default: NaN / Inf scan of every assembled residual, status NSGPU_ENONFINITE);
 * "renumber" (0 never, 1 default: internal vertex-blocked numbering when the caller's W.dofmap.list is not vertex-blocked,
 * 2 always) and "renumber_order" (1 leader-dof order, 2 default: Morton order of the vertices) -- both before nsgpu_set_space. */
int nsgpu_set_option(nsgpu_ctx* ctx, const char* name, int64_t value);

/* Which assembly kernel variant the last residual / Jacobian call ran: "p1tet_ws", "p1tet_ws (streamed host vectors)",
 * "p1tet_pipe", "p1tet_pipe (streamed host vectors)", "p1tet_tiles", "rowown", "generic_coop", "generic_row", "trace_rk45"
 * (static string, never NULL). */
const char* nsgpu_last_kernel_name(const nsgpu_ctx* ctx);
/* Which MatMult kernel the last nsgpu_spmv* / Krylov product ran: "spmv_block4" (vertex-blocked 4x4 blocks, one column index
 * per block) or "spmv_csr". */
const char* nsgpu_last_spmv_name(const nsgpu_ctx* ctx);

/* Time on ctx's stream, CUDA events: ms of the last call of each phase.
 * 0 jacobian+residual kernel(s), 1 residual-only kernel(s), 2 spmv kernel, 3 halo, 4 h2d, 5 d2h, 6 pattern build, 7 streamline kernel. */
int nsgpu_timers(nsgpu_ctx* ctx, double* ms, int n);
/* Measured FP64 ceiling of ctx's GPU: DFMA TFLOP/s of a register-resident loop (8 chains/thread, 64 warps/SM), the
 * denominator of the benchmark's fp64 fraction (SURVEY 8d asks for a measured DFMA peak). Takes ~20 ms. */
int nsgpu_fp64_peak(nsgpu_ctx* ctx, double* tflops);
/* Kernel launches issued by this context since creation (bench.py's "gpu_launches"). */
int64_t nsgpu_launch_count(nsgpu_ctx* ctx);
/* Device time (ms) of the main kernel(s) of the last *_dev call; synchronises on that call's end event. */
int nsgpu_last_kernel_ms(nsgpu_ctx* ctx, double* ms);
/* CUDA-event stopwatch on ctx's stream (the stream every kernel of ctx is launched on). */
int nsgpu_timer_start(nsgpu_ctx* ctx);
int nsgpu_timer_stop(nsgpu_ctx* ctx, double* ms);

/* ---- multi-GPU: x.ghostUpdate(INSERT, FORWARD) / F.ghostUpdate(ADD, REVERSE) / J.assemble()
 *      (NavierStokesChannelFlow.py:57-60, :66, :75) over NCCL ------------------------------------- */
int nsgpu_comm_unique_id(void* out, int64_t nbytes /* >= 128 */);
int nsgpu_comm_init(nsgpu_ctx* ctx, int rank, int nranks, const void* unique_id);
/* Vector halo plan.  For neighbour k: forward sends x[send_idx[send_ptr[k]..send_ptr[k+1])] (owned dofs
 * ghosted by neigh_rank[k]) and receives into x[recv_idx[recv_ptr[k]..]] (local ghost dofs owned by it);
 * the reverse (ADD) exchange uses the same lists with the roles swapped. */
int nsgpu_set_halo(nsgpu_ctx* ctx, int n_neigh, const int32_t* neigh_rank, const int64_t* send_ptr, const int32_t* send_idx,
                   const int64_t* recv_ptr, const int32_t* recv_idx);
/* Ghost-row plan for J.assemble().  For neighbour k: this rank sends the CSR values of its ghost rows
 * owned by neigh_rank[k], positions send_pos[send_ptr[k]..], and adds what it receives at recv_pos[...]. */
int nsgpu_set_row_exchange(nsgpu_ctx* ctx, int n_neigh, const int32_t* neigh_rank, const int64_t* send_ptr, const int64_t* send_pos,
                           const int64_t* recv_ptr, const int64_t* recv_pos);
/* Extra (row, col) entries contributed by other ranks' ghost rows (dolfinx SparsityPattern::finalize);
 * must be called before nsgpu_build_pattern. */
int nsgpu_add_pattern_entries(nsgpu_ctx* ctx, int64_t n, const int32_t* rows, const int32_t* cols);
/* Column ghosts that are dofs of no local cell but appear in rows this rank owns through other ranks' ghost
 * rows (dolfinx SparsityPattern::finalize appends them to the column index map).  They get local column
 * indices n_owned + n_ghost + k.  leader_local / slot / size describe which of them live on one mesh entity
 * (leader = local index of the entity's first dof, slot = position in the entity, size = dofs on it).
 * After this call every x_local vector has n_owned + n_ghost + n_extra entries (nsgpu_local_sizes). */
int nsgpu_set_col_ghosts(nsgpu_ctx* ctx, int64_t n_extra, const int32_t* leader_local, const int32_t* slot, const int32_t* size);
int nsgpu_local_sizes(nsgpu_ctx* ctx, int64_t* n_owned, int64_t* n_ghost, int64_t* n_cols);
/* Rows of the pattern by local row index (used to build the J.assemble() plan without fetching the whole
 * pattern): start_out[k] = position of the row's first entry in the CSR arrays, ptr_out has n+1 offsets into
 * idx_out; idx_out == NULL only fills start_out / ptr_out (size query). */
int nsgpu_get_rows(nsgpu_ctx* ctx, int64_t n, const int32_t* rows, int64_t* start_out, int64_t* ptr_out, int32_t* idx_out,
                   int64_t idx_capacity);

/* ---- streamline tracing (SURVEY 8f rank 4; NavierStokes/streamtrace.py) -------------------------------------------------
 * One GPU thread integrates one seed with scipy's RK45 algorithm (solve_ivp(..., method='RK45', events=..., max_step=...)),
 * locating the point in the tetrahedral mesh of nsgpu_set_mesh and evaluating the P1 velocity there; zero outside the mesh.
 *
 * nsgpu_trace_setup  builds the point locator (first call / new tol) and loads the nodal velocity u_nodes (n_nodes x 3, the
 *                    geometry-node order of nsgpu_set_mesh; NULL keeps the previous field).  Replaces geometry.bb_tree(mesh, 3)
 *                    (streamtrace.py:397) and the Function uh filled by read_mesh_and_function (:57-129).  tol: a point is inside
 *                    a cell when every barycentric coordinate is >= -tol.
 * nsgpu_trace_velocity = velfunc (streamtrace.py:144-158) on n points: vel (n x 3), cell (n, -1 outside; may be NULL).
 * nsgpu_trace_run    = streamtrace_pool (:198-218, reverse = 0: events |u| - speed_min falling, x - x_stop rising) or
 *                    reverse_streamtrace_pool (:357-384, reverse = 1: velocity negated, x - x_stop falling) for n seeds at once.
 *                    end_xyz (n x 3) = sol.y[:, -1]; status per seed: 0 reached t_end, 1 position event, 2 speed event,
 *                    -1 step size underflow, -2 max_steps accepted steps; t_final / n_steps may be NULL.  The reference's values:
 *                    x_stop 3.7 / 0.13, speed_min 1e-6, t_end 20, max_step 0.125, rtol 1e-3, atol 1e-6 (scipy defaults). */
int nsgpu_trace_setup(nsgpu_ctx* ctx, const double* u_nodes, double tol);
int nsgpu_trace_velocity(nsgpu_ctx* ctx, int64_t n, const double* points, double* vel, int32_t* cell);
int nsgpu_trace_run(nsgpu_ctx* ctx, int64_t n, const double* seeds, int reverse, double x_stop, double speed_min, double t_end,
                    double max_step, double rtol, double atol, int64_t max_steps, double* end_xyz, int32_t* status, double* t_final,
                    int32_t* n_steps);

#ifdef __cplusplus
}
#endif
#endif /* NSGPU_H */
