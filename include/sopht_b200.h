/*
 * sopht_b200.h -- C ABI of libsophtb200.so
 *
 * B200-native (sm_100a) implementation of the per-timestep Eulerian/Lagrangian
 * hot path of sopht-mpi.  The reference (pure Python: pystencils / numba /
 * mpi4py-fft JITs) has no FFI; the boundary a maintainer binds is its Python
 * operator API.  Each entry point below names the reference callable it
 * replaces (paths relative to the reference tree, sopht_mpi/...).
 *
 * Conventions
 *  - every function returns 0 on success, a negative value on error;
 *    sb200_last_error() returns a message for the calling thread.
 *  - all field pointers are DEVICE pointers (owned by the caller, e.g. a torch
 *    tensor); `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *  - fields are C-ordered (z,y,x) / (ncomp,z,y,x), padded with `gs` ghost
 *    cells on every side of every axis, exactly the reference's local arrays
 *    (simulator/flow/flow_simulators_mpi_3d.py:170-196).  2D: (y,x), n[0] = 1.
 *  - no torch / C++ types cross this boundary.
 */
#ifndef SOPHT_B200_H
#define SOPHT_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB200_F32 0
#define SB200_F64 1

/* local (per rank / per GPU) grid description */
typedef struct sb200_grid {
  int32_t dim;     /* 2 or 3 */
  int32_t dtype;   /* SB200_F32 / SB200_F64 */
  int32_t gs;      /* ghost size */
  int32_t n[3];    /* local interior size (z,y,x); 2D: n[0] = 1 */
  int32_t phys[6]; /* z_prev,z_next,y_prev,y_next,x_prev,x_next: 1 = neighbour is
                      PROC_NULL (physical boundary), utils/mpi_utils_3d.py:70-74 */
} sb200_grid_t;

const char* sb200_last_error(void);
int sb200_version(void);

/* ---- pointwise ops over `count` contiguous reals (whole padded arrays) ----
 * replace the un-vendored sopht elementwise kernels called at
 * simulator/flow/flow_simulators_mpi_3d.py:267-269,303-318,397-401,422-424 and
 * numeric/eulerian_grid_ops/stencil_ops_3d/laplacian_filter_mpi_3d.py:102-107 */
int sb200_set_fixed_val(int dtype, void* field, int64_t count, double value, void* stream);
int sb200_elementwise_sum(int dtype, void* sum, const void* a, const void* b, int64_t count, void* stream);
int sb200_elementwise_copy(int dtype, void* dst, const void* src, int64_t count, void* stream);
int sb200_elementwise_saxpby(int dtype, void* sum, const void* a, double pa, const void* b, double pb,
                             int64_t count, void* stream);
/* result/field_1/field_2 are (3,count) */
int sb200_elementwise_cross_product(int dtype, void* result, const void* f1, const void* f2,
                                    int64_t count, void* stream);
/* field (ncomp,count) += vals[c] */
int sb200_add_fixed_val(int dtype, void* field, int ncomp, int64_t count, const double* vals, void* stream);

/* ---- stencils: interior + six boundary slabs + physical-ring zeroing ------ */
/* stencil_ops_3d/update_vorticity_from_velocity_forcing_mpi_3d.py:27-176 and
 * stencil_ops_2d/update_vorticity_from_velocity_forcing_mpi_2d.py:8-123
 * (3D: omega(3), F(3); 2D: omega scalar, F(2)) */
int sb200_update_vorticity_from_velocity_forcing(const sb200_grid_t* g, void* vorticity,
                                                 const void* velocity_forcing, double prefactor, void* stream);
/* The same update for a forcing field that is zero almost everywhere (immersed-boundary forcing):
 * F is read once to flag the 1024-cell chunks of the padded array that hold a non-zero value
 * (`tile_flags`: a device work buffer of sb200_tile_flag_count(g) BYTES, zero-initialised once by the
 * caller: per-chunk flags and the compact lists of flagged / active chunks),
 * omega is only touched on chunks whose stencil reaches a flagged chunk.  sb200_clear_flagged_tiles
 * zeroes `field` on the flagged chunks and clears the flags: the `set_field(F, 0)` that ends the reference step
 * (simulator/flow/flow_simulators_mpi_3d.py:422-424, flow_simulators_mpi_2d.py:291-293) at a cost
 * proportional to the support of F. */
int64_t sb200_tile_flag_count(const sb200_grid_t* g);
int sb200_update_vorticity_from_sparse_forcing(const sb200_grid_t* g, void* vorticity,
                                               const void* velocity_forcing, double prefactor,
                                               void* tile_flags, void* stream);
int sb200_clear_flagged_tiles(const sb200_grid_t* g, void* field, int ncomp, void* tile_flags, void* stream);
/* stencil_ops_3d/curl_mpi_3d.py:29-194; 2D: stencil_ops_2d/outplane_field_curl_mpi_2d.py:10-141 */
int sb200_curl(const sb200_grid_t* g, void* curl, const void* field, double prefactor, void* stream);
/* stencil_ops_3d/diffusion_flux_mpi_3d.py:35-192 (scalar field) */
int sb200_diffusion_flux(const sb200_grid_t* g, void* diffusion_flux, const void* field, double prefactor,
                         void* stream);
/* stencil_ops_3d/diffusion_timestep_mpi_3d.py:41-90: ncomp sequential scalar
 * steps sharing one scalar flux buffer */
int sb200_diffusion_timestep(const sb200_grid_t* g, void* field, int ncomp, void* diffusion_flux,
                             double nu_dt_by_dx2, void* stream);
/* stencil_ops_3d/advection_flux_mpi_3d.py:25-193 (ENO3, kernel support 2) */
int sb200_advection_flux_eno3(const sb200_grid_t* g, void* advection_flux, const void* field,
                              const void* velocity, double inv_dx, void* stream);
/* stencil_ops_3d/advection_timestep_mpi_3d.py:40-93 */
int sb200_advection_timestep_eno3(const sb200_grid_t* g, void* field, int ncomp, void* advection_flux,
                                  const void* velocity, double dt_by_dx, void* stream);
/* stencil_ops_3d/divergence_mpi_3d.py:31-198 */
int sb200_divergence(const sb200_grid_t* g, void* divergence, const void* field, double inv_dx, void* stream);
/* stencil_ops_3d/laplacian_filter_mpi_3d.py:267-419; filter_type 0 = multiplicative, 1 = convolution */
int sb200_laplacian_filter(const sb200_grid_t* g, void* field, int ncomp, int filter_order, int filter_type,
                           void* filter_flux_buffer, void* field_buffer, void* stream);
/* The order-1 multiplicative filter (the rod examples' setting, flow_past_rod_case.py:114-115) of a
 * vector field in ONE pass, out of place: out = field - Fz(Fy(Fx(field))) with the wrappers' masks and ring
 * zeroing (laplacian_filter_mpi_3d.py:267-319), for a block whose six faces are all physical (one rank).
 * filter_flux_buffer and field_buffer end up as the reference leaves them (the last component's flux). */
int sb200_laplacian_filter_order1_out_of_place(const sb200_grid_t* g, void* out, const void* field, int ncomp,
                                               void* filter_flux_buffer, void* field_buffer, void* stream);
/* one axis pass of the filter incl. the ring clearing that follows it
 * (laplacian_filter_mpi_3d.py:145-264,118-143); axis = ARRAY axis counted from the
 * last one: 0 = x, 1 = y, 2 = z.  Lets the host exchange halos between passes. */
int sb200_laplacian_filter_axis(const sb200_grid_t* g, void* filter_flux, const void* field_buffer,
                                int axis, void* stream);
/* One stage of the filter chain with the wrapper bookkeeping folded in (out of place):
 *   out = ring ? 0 : written ? 0.25 (-in(+1) - in(-1) + 2 in) : (first ? out : in);  field -= out if field
 * (reference laplacian_filter_mpi_3d.py:145-385: seven-region filter + ring clear + buffer copy per
 * stage, `field -= filter_flux` after the last).  The distributed path calls it between halo
 * exchanges of `in`; sb200_laplacian_filter chains it on one rank. */
int sb200_laplacian_filter_stage(const sb200_grid_t* g, void* out, const void* in, int axis, void* field,
                                 int first, void* stream);
/* zero the physical-boundary ring of width gs+width (laplacian_filter_mpi_3d.py:118-143) */
int sb200_clear_physical_ring(const sb200_grid_t* g, void* field, int ncomp, int width, void* stream);
/* stencil_ops_3d/penalise_field_boundary_mpi_3d.py:185-267.  `factors` is a
 * DEVICE array [2*dim][gs+width] of the sine factors in real_t, ordered
 * (3D) z_front,z_back,y_front,y_back,x_front,x_back, each indexed by the
 * distance-ordered position inside its slab (index 0 = outermost ghost cell
 * for *_front, = first slab cell for *_back, i.e. array order). */
int sb200_penalise_field_boundary(const sb200_grid_t* g, void* field, int ncomp, int width,
                                  const void* factors, void* stream);

/* ---- operators of the reference API that no simulator path uses (arithmetic in the un-vendored `sopht`
 * package, published forms restated):
 * stencil_ops_3d/brinkmann_penalise_mpi_3d.py:7-21: penalised = (field + lambda chi target) / (1 + lambda chi),
 * pointwise over `count` cells, `ncomp` components sharing one characteristic function;
 * stencil_ops_3d/char_func_from_level_set_mpi_3d.py:8-30: smooth sine Heaviside of a level set;
 * stencil_ops_3d/update_vorticity_from_velocity_forcing_mpi_3d.py:181-330:
 * omega += prefactor * curl(penalised_velocity - velocity) on the cells the wrapper writes. */
int sb200_brinkmann_penalise(int dtype, void* penalised, double penalty_factor, const void* char_func,
                             const void* penalty_field, const void* field, int ncomp, int64_t count, void* stream);
int sb200_char_func_from_level_set(int dtype, void* char_func, const void* level_set, double blend_width,
                                   int64_t count, void* stream);
int sb200_update_vorticity_from_penalised_velocity(const sb200_grid_t* g, void* vorticity,
                                                   const void* penalised_velocity, const void* velocity,
                                                   double prefactor, void* stream);

/* ---- reductions over the interior; result written as ONE double at `out`
 * (device pointer, 8 bytes) ------------------------------------------------ */
/* max over interior of sum_c |u_c| : simulator/flow/flow_simulators_mpi_3d.py:429-442 */
int sb200_max_abs_sum(const sb200_grid_t* g, const void* field, int ncomp, void* out, void* stream);
/* signed max over interior of all components: flow_simulators_mpi_3d.py:471-476 */
int sb200_max(const sb200_grid_t* g, const void* field, int ncomp, void* out, void* stream);
/* sum of squares over interior: flow_simulators_mpi_3d.py:461-464 */
int sb200_sum_squares(const sb200_grid_t* g, const void* field, int ncomp, void* out, void* stream);

/* ---- fused hot path -------------------------------------------------------
 * u = prefactor*curl(psi), zero physical ring, u += U_inf, F = 0 and
 * max_abs_sum(u) in one sweep: flow_simulators_mpi_3d.py:388-393,422-424,429-442.
 * `forcing` may be NULL, `max_out` may be NULL. */
int sb200_velocity_from_stream_function(const sb200_grid_t* g, void* velocity, const void* stream_func,
                                        double prefactor, const double* free_stream, void* forcing,
                                        void* max_out, void* stream);
/* omega <- omega + p*curl(F); omega <- omega + p*curl(u x omega); omega <- omega + c*lap(omega)
 * flow_simulators_mpi_3d.py:395-411,416-420 in one streaming pass.
 * `forcing` may be NULL (flow_type "navier_stokes"); `out` must not alias `vorticity`. */
int sb200_vorticity_rhs_fused_3d(const sb200_grid_t* g, void* out, const void* vorticity,
                                 const void* velocity, const void* forcing, double curl_prefactor,
                                 double nu_dt_by_dx2, void* stream);

/* The same sweep restricted to the output planes [z_begin, z_end) (it reads the input planes z_begin - 2
 * ... z_end + 1): lets the caller run the planes that do not depend on ghost planes while the halo
 * exchange is in flight, and the remaining ones afterwards (the reference's interior -> Waitall ->
 * boundary slabs structure, e.g. stencil_ops_3d/curl_mpi_3d.py:41-194). */
int sb200_vorticity_rhs_fused_3d_range(const sb200_grid_t* g, void* out, const void* vorticity,
                                       const void* velocity, double curl_prefactor, double nu_dt_by_dx2,
                                       int z_begin, int z_end, void* stream);

/* ---- unbounded Poisson solver ---------------------------------------------
 * poisson_solver_3d/UnboundedPoissonSolverMPI3D.py:22-187 (+ fft_mpi_3d.py),
 * poisson_solver_2d/UnboundedPoissonSolverMPI2D.py:12-153.
 * nz,ny,nx: GLOBAL interior grid; this handle serves rank `rank` of `nranks`
 * z-slabs (y-slabs in 2D).  With nranks > 1 the caller performs the two
 * transposes between sb200_poisson_forward_local / _backward_local. */
typedef struct sb200_poisson sb200_poisson_t;
int sb200_poisson_create(sb200_poisson_t** out, int dim, int dtype, int nz, int ny, int nx, int gs,
                         double x_range, int rank, int nranks, int backend, void* stream);
int sb200_poisson_destroy(sb200_poisson_t* p);
/* single-rank solve of `ncomp` components: psi interior <- solve(rhs interior) */
int sb200_poisson_solve(sb200_poisson_t* p, void* solution, const void* rhs, int ncomp, void* stream);
int64_t sb200_poisson_workspace_bytes(const sb200_poisson_t* p);
/* z-slab decomposition.  Served by distributed handles (nranks > 1, 3D) of either backend: backend 1
 * on 2, 4 or 8 ranks for power-of-two grids, backend 0 (cuFFT) on any rank count that divides nz, for
 * any grid size.  Both use the same buffers and layout.  mpi4py-fft's distributed transform
 * (poisson_solver_3d/fft_mpi_3d.py:27-48) and MPIDomainDoublingCommunicator3D
 * (UnboundedPoissonSolverMPI3D.py:190-382) become
 *   slab_forward  (x r2c of the local planes -> send_buf, blocked by destination rank: each rank
 *                  receives ceil((nx+1)/nranks) kx bins, rounded up to a multiple of 4, of every plane)
 *   all-to-all  send_buf -> recv_buf                       (caller: NCCL)
 *   slab_spectral (y and z forward on the zero-padded doubled plane x Green x inverse, cropped;
 *                  result back in recv_buf)
 *   all-to-all  recv_buf -> send_buf
 *   slab_backward (x c2r of the local planes -> solution interior)
 * The transposes act on the x-pass output, the smallest array of the pipeline (2 reals per cell
 * instead of 4 after the y pass).  Both buffers hold sb200_poisson_slab_buffer_bytes(p, ncomp)
 * bytes and must be ZERO-INITIALISED once by the caller (the padding bins of the last kx block are
 * never written). */
int64_t sb200_poisson_slab_buffer_bytes(const sb200_poisson_t* p, int ncomp);
int sb200_poisson_slab_forward(sb200_poisson_t* p, const void* rhs, int ncomp, void* send_buf, void* stream);
int sb200_poisson_slab_spectral(sb200_poisson_t* p, void* recv_buf, int ncomp, void* stream);
int sb200_poisson_slab_backward(sb200_poisson_t* p, void* solution, int ncomp, const void* send_buf,
                                void* stream);
/* Per-kernel device times of a single-rank solve of the fft backend: with profiling on, CUDA events
 * are recorded on the solve's stream around its five launches; sb200_poisson_last_stage_ms
 * synchronises on the last event and writes n <= 5 times in milliseconds,
 * {x r2c, y forward, fused z (forward x Green x inverse), y inverse, x c2r}.  bench.py uses it to
 * time the dominant kernel live, inside its timed region. */
int sb200_poisson_set_profiling(sb200_poisson_t* p, int enable);
int sb200_poisson_last_stage_ms(sb200_poisson_t* p, float* ms_out, int n);
/* NVLink peer copies for the transposes (replace the MPI Alltoallw inside mpi4py-fft,
 * poisson_solver_3d/fft_mpi_3d.py:27-48): `dst` is a pointer into another rank's exchange buffer,
 * mapped into this process through CUDA IPC by the caller.  enable_peer_access is called once per
 * device pair; peer_copy enqueues a copy-engine transfer on `stream`. */
int sb200_enable_peer_access(int device, int peer_device);
int sb200_peer_copy(void* dst, int dst_device, const void* src, int src_device, int64_t bytes, void* stream);
int sb200_peer_copy_blocks(int n, void* const* dst, const int* dst_device, const void* const* src,
                           int src_device, int64_t bytes, void* stream);
/* The exchange as one kernel: block k (bytes, a multiple of 16) is copied from src[k] (local) to dst[k] (an
 * IPC-mapped pointer into rank k's buffer, or a local pointer) by blocks_per_peer thread blocks of
 * 512 threads each (<= 0: default), all n <= 8 destinations concurrently over NVLink.  With
 * signal_flags != NULL, signal_flags[k] (an int32 in rank k's memory, IPC-mapped) is set to `epoch` once
 * block k has landed completely (done_counters: n zero-initialised device int32 of the caller);
 * sb200_peer_wait_flags makes the stream wait until the n flags of the local buffer have reached
 * `epoch` (bounded spin: *error_flag, a device int32, is raised after ~2 s).  Together they replace the
 * collective barrier behind the MPI Alltoallw of mpi4py-fft (poisson_solver_3d/fft_mpi_3d.py:27-48). */
int sb200_peer_push_blocks(int n, void* const* dst, const void* const* src, int64_t bytes, int blocks_per_peer,
                           void* const* signal_flags, int epoch, void* done_counters, void* stream);
int sb200_peer_wait_flags(const void* flags, int n, int epoch, void* error_flag, void* stream);
/* Exchange buffers shared between the ranks of a node: plain device allocations (zero-initialised) whose
 * CUDA IPC handle (64 bytes) another process opens while its own device is current, so that its kernels
 * can store through the mapping over NVLink (cudaIpcMemLazyEnablePeerAccess). */
int sb200_peer_alloc(int64_t bytes, void** ptr_out);
int sb200_peer_free(void* ptr);
int sb200_ipc_export(const void* ptr, void* handle_out_64);
int sb200_ipc_open(const void* handle_64, void** ptr_out);
int sb200_ipc_close(void* ptr);
/* 1 when the pruned in-kernel FFT backend (backend = 1, power-of-two grids) is built in */
int sb200_poisson_fft_available(void);

/* ---- immersed boundary ------------------------------------------------------
 * numeric/immersed_boundary_ops/EulerianLagrangianGridCommunicatorMPI3D.py:116-589
 * (+ 2D twin) and VirtualBoundaryForcingMPI.py:278-406.  Lagrangian arrays are
 * (dim,n) device arrays of lag_dtype; substart_xyz = local interior start index
 * in x,y,z order. */
typedef struct sb200_ib_params {
  int32_t lag_dtype;      /* SB200_F32 / SB200_F64 */
  int32_t kernel_type;    /* 0 = cosine, 1 = peskin */
  int32_t width;          /* interp_kernel_width (2) */
  int32_t substart_xyz[3];
  double dx;              /* value of real_t(dx) */
  double coord_shift;     /* eul_grid_coord_shift */
  double stiffness;       /* virtual_boundary_stiffness_coeff (already rescaled) */
  double damping;
} sb200_ib_params_t;
/* steps 1-5 of compute_interaction_force_on_lag_grid (VirtualBoundaryForcingMPI.py:357-397):
 * nearest index, weights, E->L interpolation of u, velocity mismatch, penalty force.
 * nearest (dim,n) int64; weights ((2w)^dim, n) lag_dtype, may be NULL. */
int sb200_ib_interact_lag(const sb200_grid_t* g, const sb200_ib_params_t* p, int64_t n,
                          const void* eul_velocity, const void* lag_position, const void* lag_velocity,
                          const void* position_mismatch, void* nearest, void* weights,
                          void* flow_velocity, void* velocity_mismatch, void* forcing, void* stream);
/* L->E spreading without ghost sum: ...MPI3D.py:329-427 */
int sb200_ib_spread(const sb200_grid_t* g, const sb200_ib_params_t* p, int64_t n, void* eul_forcing,
                    const void* lag_forcing, const void* lag_position, void* stream);
/* Lagrangian rank ownership on the device: utils/mpi_utils_3d.py:1352-1384 (`_compute_lag_nodes_rank_address`),
 * mpi_utils_2d.py:611-637.  rank_address[i] (int32, device) = row-major Cartesian rank of the block
 * coordinates ((pos - shift) / sub_dx).astype(int32) of point i; sub_dx_zyx = eul_grid_dx * local grid
 * size per ARRAY axis (z,y,x; 2D: entry 0 unused), topo_zyx the grid topology in the same order (host
 * arrays of 3).  *out_of_domain_flag (device int32, may be NULL) is set to 1 if a block coordinate falls
 * outside the topology (the reference logs an error and aborts). */
int sb200_ib_rank_address(int lag_dtype, int dim, int64_t n, const void* lag_position, double coord_shift,
                          const double* sub_dx_zyx, const int32_t* topo_zyx, void* rank_address,
                          void* out_of_domain_flag, void* stream);
/* sb200_ib_interact_lag / sb200_ib_spread over GLOBAL (replicated) Lagrangian arrays, restricted to the
 * points with rank_address[i] == my_rank (rank_address NULL: all points); the interaction writes zeros
 * for the other points so that one SUM all-reduce assembles the global arrays: replaces
 * MPILagrangianFieldCommunicator3D.scatter_global_field / gather_local_field
 * (utils/mpi_utils_3d.py:1410-1459) and VirtualBoundaryForcingMPI.update_buffers (:238-276). */
int sb200_ib_interact_owned(const sb200_grid_t* g, const sb200_ib_params_t* p, int64_t n,
                            const void* eul_velocity, const void* lag_position, const void* lag_velocity,
                            const void* position_mismatch, void* nearest, void* weights, void* flow_velocity,
                            void* velocity_mismatch, void* forcing, const void* rank_address, int my_rank,
                            void* stream);
int sb200_ib_spread_owned(const sb200_grid_t* g, const sb200_ib_params_t* p, int64_t n, void* eul_forcing,
                          const void* lag_forcing, const void* lag_position, const void* rank_address,
                          int my_rank, void* stream);
/* zero all ghost cells: ...MPI3D.py:786-792 */
int sb200_clear_ghost_cells(const sb200_grid_t* g, void* field, int ncomp, void* stream);
/* dst interior-adjacent layers += src slab (ghost-sum receive side): ...MPI3D.py:689-784 */
int sb200_ghost_sum_add_z(const sb200_grid_t* g, void* field, int ncomp, const void* from_prev,
                          const void* from_next, void* stream);
/* generic E->L interpolation of an n_components field (the communicator's public kernel) */
int sb200_ib_interpolate(const sb200_grid_t* g, const sb200_ib_params_t* p, int64_t n, int ncomp,
                         const void* eul_field, const void* lag_position, void* lag_field, void* stream);
/* position_mismatch += dt * velocity_mismatch: VirtualBoundaryForcingMPI.py:293-307 */
int sb200_ib_update_position_mismatch(int lag_dtype, void* position_mismatch, const void* velocity_mismatch,
                                      int64_t count, double dt, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SOPHT_B200_H */
