/* pamg.h — C ABI of the B200-native AMG-PCG solve phase (libpamg.so).
 *
 * This is the drop-in boundary for the path tirtho109/parallel_AMG applies through
 * PartitionedArrays.jl.  The reference snapshot defines NO interface of its own
 * (/root/reference/README.md:1-2 is the whole repository), so every entry point below cites
 * the PartitionedArrays.jl / PartitionedSolvers.jl call it stands in for as recalled in
 * SURVEY.md Appendix A [RECALL-UNVERIFIED]; the Julia `ccall` stubs are in julia/PAMG.jl and
 * INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers and sizes only; caller owns every host array, the library copies on
 *     entry and never retains a host pointer; the library owns all device memory.
 *   - every function returns PAMG_OK (0) or a negative pamg_status; nothing throws or aborts
 *     across the ABI; pamg_last_error() gives the CUDA / argument error text.
 *   - ids are 0-based (the Julia shim subtracts 1); global ids int64, local ids int32.
 *   - local order of a part = own ids (ascending global id) then ghost ids (ascending
 *     (owner part, global id)).
 *   - vectors cross the ABI as `nparts` host pointers to OWN values (n_own doubles each);
 *     entries for parts that are not device-resident in this process may be NULL.
 *   - not thread-safe per context; distinct contexts are independent.
 */
#ifndef PAMG_H
#define PAMG_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct pamg_ctx pamg_ctx;

typedef enum {
  PAMG_OK = 0,
  PAMG_ERR_ARG = -1,      /* bad argument / call order */
  PAMG_ERR_CUDA = -2,     /* CUDA runtime error (text in pamg_last_error) */
  PAMG_ERR_NOGPU = -3,    /* no usable CUDA device: there is NO CPU fallback */
  PAMG_ERR_COMM = -4,     /* peer mapping / halo time-out */
  PAMG_ERR_NOTCONV = -5,  /* pcg hit maxiter (x still holds the last iterate) */
  PAMG_ERR_ALLOC = -6
} pamg_status;

enum { PAMG_SMOOTHER_JACOBI = 0, PAMG_SMOOTHER_L1JACOBI = 1, PAMG_SMOOTHER_CHEBYSHEV = 2 };
enum { PAMG_CYCLE_V = 0, PAMG_CYCLE_W = 1 };
/* kernel family for the own-own blocks: CSR = sub-warp "vector per row" (1..32 lanes chosen from the
 * mean nnz/row; 32 = warp per row); STREAM = CSR-stream (block-cooperative 128-bit coalesced loads of
 * the contiguous val/col ranges, products staged in shared memory); the storage is plain CSR for both.
 * SELL = SELL-C-sigma (C = 32 x sell_rows_per_thread rows per slice, column-major slices, rows sorted by
 * length inside windows of sell_sigma rows), one thread per row, no row pointers.  AUTO decides per
 * operator from the nnz/row distribution (padding of the SELL layout; row length vs. the STREAM buffer).
 * A SELL block (2 rows per thread) with at most 255 distinct values -- stencil matrices, their prolongators -- is stored
 * VALUE-INDEXED: int32 column + one byte into a dictionary of the original doubles (two bytes up to 4095 values), four
 * interleaved rows per lane in slices of 128 rows: 5 (6) instead of 12 bytes per entry, bit-identical products and sums
 * (pamg_stats.value_indexed, pamg_layout_sell_values; env PAMG_VALUE_INDEX=0 keeps fp64 values).
 * Under AUTO an A block of at least 200000 rows whose rows hold their entries at row + off[j] for at most 32 fixed offsets
 * (stencil matrices; strictly ascending columns, ndiag x rows <= 1.25 nnz, <= 254 distinct non-zero values) is stored with
 * IMPLIED COLUMNS: one index byte per (row, offset) slot and no column (pamg_stats.value_indexed bit 64, pamg_layout_sell_diag;
 * pamg_stats.format still reads SELL).  SELL_DIAG takes that layout for every qualifying A block at any size and handles all
 * other blocks as SELL; an explicit SELL never takes it. */
enum { PAMG_FORMAT_AUTO = 0, PAMG_FORMAT_CSR = 1, PAMG_FORMAT_STREAM = 2, PAMG_FORMAT_SELL = 3, PAMG_FORMAT_SELL_DIAG = 4 };
/* blocks of the split (own/ghost) storage of a level, PSparseMatrix own_own_values /
 * own_ghost_values (SURVEY.md App. A "PSparseMatrix") */
enum { PAMG_A_OO = 0, PAMG_A_OG = 1, PAMG_P_OO = 2, PAMG_P_OG = 3, PAMG_R_OO = 4, PAMG_R_OG = 5 };

/* PartitionedSolvers `amg(; fine_params, coarse_params)` keyword set (App. A) + kernel knobs */
typedef struct {
  int32_t struct_size;    /* = sizeof(pamg_options), checked */
  double eps_strength;    /* smoothed_aggregation(; epsilon): 0 => structural strength */
  int32_t coarse_size;    /* amg_coarse_params(; coarse_size) */
  int32_t max_levels;     /* amg_fine_params(; n_fine_levels)+1 */
  int32_t smoother;       /* PAMG_SMOOTHER_* : jacobi(; iters, omega) / l1 / chebyshev */
  double omega_jacobi;    /* jacobi(; omega) */
  int32_t nu_pre;         /* pre_smoother iters */
  int32_t nu_post;        /* pos_smoother iters */
  int32_t cheb_degree;
  double cheb_lo_frac;    /* Chebyshev interval [lo_frac*rho, hi_frac*rho] of D^-1 A */
  double cheb_hi_frac;
  int32_t spmv_format;    /* PAMG_FORMAT_* ; AUTO decides per level and per operator (A, P, R) */
  int32_t use_graph;      /* 1: replay the V-cycle / PCG iteration as CUDA graphs */
  int32_t lanes_per_row;  /* 0: auto (from mean nnz/row); else 1,2,4,8,16,32 for CSR */
  int32_t tail_rows;      /* coarse-level agglomeration: levels (>= 1) whose global rows <= this are merged over all
                             parts and run replicated on every GPU without halos (0: only the coarsest level) */
  int32_t sell_sigma;     /* SELL sorting window in rows; 0: auto (1 = no sorting when the padding is small) */
  int32_t sell_rows_per_thread; /* 1 or 2 (C = 32 or 64; 2 => 128-bit value loads); 0: auto */
  int32_t fuse_halo;      /* 1: halo pack / wait / boundary rows run inside the consuming kernel whenever every local
                             part has a GPU of its own; 0: always three launches (env PAMG_FUSE_HALO overrides) */
  int32_t cycle;          /* PAMG_CYCLE_V (0) or PAMG_CYCLE_W (1): amg_level_params(; cycle = v_cycle | w_cycle) */
} pamg_options;

typedef struct {
  int64_t n_global;       /* rows of A_level over all parts */
  int64_t n_own, n_ghost; /* this part */
  int64_t n_own_coarse;   /* own rows of the next level (0 on the coarsest) */
  int64_t nnz[6];         /* PAMG_A_OO .. PAMG_R_OG */
  int32_t n_recv_nbrs, n_send_nbrs;
  int64_t n_send;         /* total entries of the send lists */
  double rho;             /* Gershgorin bound of rho(D^-1 A) on this level */
  double omega_p;         /* prolongator smoothing weight 4/(3 rho_F) (0 on the coarsest) */
} pamg_level_info;

typedef struct {
  int32_t iters;
  int32_t converged;
  double r0_norm, r_norm;
  double solve_ms;        /* device time of the last pamg_pcg (CUDA events, max over local parts) */
  double vcycle_ms;       /* device time of the last pamg_vcycle */
  int64_t kernel_launches;/* kernels launched (or graph kernel nodes replayed) by the last call */
  int32_t n_levels;
  int32_t format[16];     /* PAMG_FORMAT_* chosen per level for A */
  int32_t lanes[16];      /* lanes per row chosen per level for A (CSR) */
  int32_t format_p[16];   /* PAMG_FORMAT_* chosen per level for P and R (part 0 of this process) */
  int32_t format_r[16];
  double sell_fill[16];   /* stored entries / nnz of A's SELL layout (1.0 when A is not SELL) */
  int32_t fused_halo;     /* 1 when the halo roles run inside the consuming kernels */
  int32_t tail_level;     /* first level of the replicated coarse tail (n_levels - 1: coarsest only) */
  int32_t value_indexed[16]; /* per level, bit mask 1 A / 2 P / 4 R: the SELL block stores one byte per entry into a dictionary of its
                             <= 256 distinct fp64 values instead of the values (same products, same order, same bits); 8 / 16 / 32:
                             two index bytes (wide dictionary); 64: A is stored with implied columns (pamg_layout_sell_diag) */
} pamg_stats;

void pamg_default_options(pamg_options* o);

/* ---- context ---------------------------------------------------------------------------
 * nparts = length of the PartitionedArrays `ranks` array (`distribute(LinearIndices((np,)))`). */
int pamg_create(int32_t nparts, pamg_ctx** out);
void pamg_destroy(pamg_ctx* c);
const char* pamg_last_error(const pamg_ctx* c);

/* ---- problem input (host) --------------------------------------------------------------
 * pamg_set_part_rows: one call per part = the assembled rows of a PSparseMatrix held by that
 * part (`psparse(I,J,V,rows,cols) |> fetch`, own rows, GLOBAL column ids), CSR by own row in
 * own_to_global order.  Julia's SparseMatrixCSC of a symmetric A is a valid CSR of A. */
int pamg_set_part_rows(pamg_ctx* c, int32_t part, int64_t n_own, const int64_t* own_to_global,
                       const int64_t* rowptr, const int64_t* col_gid, const double* val);
/* whole matrix + owner[gid] (one call; equivalent to nparts pamg_set_part_rows calls) */
int pamg_set_matrix_global(pamg_ctx* c, int64_t n, const int64_t* rowptr, const int64_t* col,
                           const double* val, const int32_t* owner);
/* gallery (PartitionedArrays `laplacian_fdm(nodes_per_dir, parts_per_dir, ranks)`) with
 * `uniform_partition(ranks, parts_per_dir, nodes_per_dir)` ownership */
int pamg_gallery_poisson(pamg_ctx* c, int32_t ndim, const int64_t* nodes_per_dir,
                         const int32_t* parts_per_dir);
/* -div(K grad u), K = diag(k,k,eps_z k), k in {1,kmax} on a blocks^d checkerboard (config 5) */
int pamg_gallery_diffusion_jump(pamg_ctx* c, int32_t ndim, const int64_t* nodes_per_dir,
                                const int32_t* parts_per_dir, int32_t blocks, double kmax,
                                double eps_z);
/* 3-D linear elasticity (BASELINE.json configs[3]): trilinear hexahedra on unit cubes, nodes_per_dir FREE nodes
 * with 3 DOFs each (gid = 3 node + component), the node layer at i = -1 clamped and eliminated; also installs
 * the 6 rigid-body modes as near-nullspace (PartitionedArrays `linear_elasticity_fem` +
 * `nullspace_linear_elasticity`).  Nodes, not DOFs, are partitioned. */
int pamg_gallery_elasticity(pamg_ctx* c, const int64_t* nodes_per_dir, const int32_t* parts_per_dir, double E,
                            double nu);
/* near-nullspace B (row-major n x k, GLOBAL row order) and the number of DOFs per node: the setup then
 * aggregates nodes and builds the tentative prolongator by per-aggregate QR of B (PartitionedSolvers
 * `smoothed_aggregation(; tentative_prolongator = ... with_block_size / near nullspace)`); k <= 0 or B == NULL
 * restores scalar smoothed aggregation.  Call after the matrix is set, before pamg_setup. */
int pamg_set_near_nullspace(pamg_ctx* c, int32_t block_size, int32_t k, const double* B);
int pamg_get_near_nullspace(pamg_ctx* c, int32_t* block_size, int32_t* k, double* B /* may be NULL */);
int pamg_uniform_partition(int32_t ndim, const int64_t* nodes_per_dir,
                           const int32_t* parts_per_dir, int32_t* owner_out);
/* y = A x on the global host matrix (builds right-hand sides b = A*1 without a second copy) */
int pamg_host_matvec_global(pamg_ctx* c, const double* x, double* y);
int pamg_global_size(pamg_ctx* c, int64_t* n, int64_t* nnz);

/* ---- AMG setup on the host (PartitionedSolvers `setup(amg(...), x, A, b)`) ------------- */
/* OpenMP threads for the host-side setup (launchers such as torchrun export OMP_NUM_THREADS=1);
 * n <= 0 restores the hardware default.  Process-wide. */
void pamg_set_num_threads(int32_t n);
int pamg_setup(pamg_ctx* c, const pamg_options* o);
/* external hierarchy (built by the caller, e.g. PartitionedSolvers itself), level by level,
 * part by part, in the split format; any block pointer triple may be NULL when empty */
int pamg_hierarchy_begin(pamg_ctx* c, int32_t n_levels, const pamg_options* o);
int pamg_level_upload(pamg_ctx* c, int32_t level, int32_t part, int64_t n_own, int64_t n_ghost,
                      const int64_t* own_to_global, const int64_t* ghost_to_global,
                      const int32_t* ghost_to_owner, int64_t n_own_coarse, int64_t n_ghost_coarse,
                      const int64_t* const rowptr[6], const int32_t* const col[6],
                      const double* const val[6], double rho);
int pamg_coarse_upload(pamg_ctx* c, int64_t n, const double* inverse_row_major);
int pamg_hierarchy_end(pamg_ctx* c);

/* One process per GPU: the rank that ran pamg_setup saves the hierarchy (e.g. under /dev/shm) and the other
 * ranks load it instead of repeating the setup.  keep_part >= 0 loads only that part's matrices in full (plus
 * every part on the small levels of the replicated coarse tail) and metadata for the rest; keep_part < 0 loads
 * everything.  The loading context must have been created with the same number of parts. */
int pamg_hierarchy_save(pamg_ctx* c, const char* path);
int pamg_hierarchy_load(pamg_ctx* c, const char* path, int32_t keep_part);

/* ---- hierarchy queries (bit-exact parity of maps / aggregates / CSR structure) --------- */
int pamg_num_levels(pamg_ctx* c, int32_t* n_levels);
int pamg_get_level_info(pamg_ctx* c, int32_t level, int32_t part, pamg_level_info* info);
int pamg_get_index_maps(pamg_ctx* c, int32_t level, int32_t part, int64_t* own_to_global,
                        int64_t* ghost_to_global, int32_t* ghost_to_owner);
int pamg_get_block(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int64_t* rowptr,
                   int32_t* col, double* val);
int pamg_get_aggregates(pamg_ctx* c, int32_t level, int32_t part, int32_t* agg_local);
/* nbr_part/slot0/count have n_*_nbrs entries; send_idx has n_send entries (own local ids,
 * concatenated per neighbour in nbr order) */
int pamg_get_halo_plan(pamg_ctx* c, int32_t level, int32_t part, int32_t* recv_part,
                       int32_t* recv_slot0, int32_t* recv_count, int32_t* send_part,
                       int32_t* send_slot0, int32_t* send_count, int32_t* send_idx);
int pamg_get_coarse_inverse(pamg_ctx* c, int64_t* n, double* inverse_row_major /* may be NULL */);
int pamg_get_diag(pamg_ctx* c, int32_t level, int32_t part, double* diag, double* diag_l1);

/* ---- device layouts of one own-own block (which = PAMG_A_OO / PAMG_P_OO / PAMG_R_OO), computed on the host exactly
 * as the upload does, so that their invariants can be checked without a GPU.  Output arrays may be NULL; call once
 * with NULL arrays to get the sizes.
 * SELL-C-sigma: slice sl holds rows perm[sl*C .. sl*C+C); entry j of slot q is at (slice_off[sl] + j) * C + q;
 *   stored = slice_off[n_slices] * C entries; padding is (0.0, a valid column).  sigma = -R (rows_per_slice = 32 R) gives the interleaved
 *   layout of the value-indexed kernel with R rows per lane: position lane * R + k of a full slice holds its row k * 32 + lane.
 * CSR-stream: n_blocks + 1 {first_row, first_entry} pairs (the last one = {nrows, nnz}); n_blocks = -1 when a row
 *   does not fit max_entries.
 * boundary rows: rows that also have own-ghost entries, stored whole (own-column entries [ptr[k], mid[k]), ghost-column
 *   entries [mid[k], ptr[k+1])); skip[row] = 1 marks them (nrows bytes). */
int pamg_layout_sell(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int32_t rows_per_slice, int32_t sigma,
                     int64_t* n_slices, int64_t* stored, int32_t* permuted, int32_t* slice_off, int32_t* col,
                     double* val, int32_t* perm);
/* value-indexed SELL storage of the same block: *indexed = 1 when it has at most 255 distinct non-zero values (bit patterns), 2 when at
 * most 4095 (two index bytes, little endian), else 0.  dict[4096] (dict[0] = +0.0, the padding value; ascending bit pattern behind it;
 * unused entries 0.0) and vidx[*indexed x stored] with dict[index k] == val[k] bit for bit in the layout of pamg_layout_sell.  The device
 * stores such blocks as int32 column + index byte(s) per entry (kernels.cuh k_spmv_sell_vi4); env PAMG_VALUE_INDEX=0 keeps fp64 values. */
int pamg_layout_sell_values(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int32_t rows_per_slice, int32_t sigma,
                            int32_t* indexed, int64_t* stored, double* dict, uint8_t* vidx);
/* SELL with implied columns of the same block (which = PAMG_A_OO): *ndiag = 0 when the block does not qualify (see
 * PAMG_FORMAT_SELL_DIAG).  Else off[*ndiag] (<= 32, ascending column offsets), dict[256] as pamg_layout_sell_values, and
 * idx[*stored] with *stored = ceil(rows / 128) x ndiag x 128 bytes: slice sl, offset j, byte 4 lane + k (k < 4) at
 * (sl ndiag + j) 128 + 4 lane + k holds the dictionary index of the entry (row, row + off[j]) for row = 128 sl + 32 k + lane (a full
 * slice) or 128 sl + 4 lane + k (the partial last slice); 255 = no such entry. */
int pamg_layout_sell_diag(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int32_t* ndiag, int32_t* off, int64_t* stored,
                          double* dict, uint8_t* idx);
int pamg_layout_stream(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int32_t max_rows, int32_t max_entries,
                       int64_t* n_blocks, int32_t* first_row, int32_t* first_entry);
int pamg_layout_boundary(pamg_ctx* c, int32_t level, int32_t part, int32_t which, int64_t* n_rows, int64_t* n_entries,
                         int32_t* lanes, int32_t* rows, int32_t* ptr, int32_t* mid, int32_t* col, double* val,
                         uint8_t* skip);

/* ---- device residency ------------------------------------------------------------------
 * Upload the parts this process drives.  One part per GPU is the production layout; several
 * parts may share one device (PartitionedArrays "debug backend" on one GPU).  With
 * nlocal < nparts the remaining parts live in other processes (one process per GPU) and
 * are wired up through the export/import/connect calls: the caller all-gathers the opaque
 * handle blobs (torch.distributed / MPI.Allgather), nothing else crosses processes on the host. */
int pamg_device_init(pamg_ctx* c, int32_t nlocal, const int32_t* local_parts,
                     const int32_t* device_ids);
/* change the kernel-side knobs (spmv_format, lanes_per_row, use_graph, sell_*, fuse_halo, tail_rows) of an existing hierarchy;
 * takes effect at the next pamg_device_init.  Numerical options are ignored. */
int pamg_set_kernel_options(pamg_ctx* c, const pamg_options* o);
int32_t pamg_comm_handle_bytes(void);
int pamg_comm_export(pamg_ctx* c, int32_t local_part, void* blob);
int pamg_comm_import(pamg_ctx* c, int32_t remote_part, const void* blob);
int pamg_comm_connect(pamg_ctx* c);

/* ---- operators on device-resident levels (host vectors in, host vectors out) -----------
 * x, y: arrays of nparts pointers to own values of the level's row partition. */
int pamg_spmv(pamg_ctx* c, int32_t level, const double* const* x, double* const* y); /* mul!(y,A,x) */
/* v: nparts pointers to LOCAL values (own then ghost); ghosts are overwritten */
int pamg_consistent(pamg_ctx* c, int32_t level, double* const* v);                  /* consistent!(v) |> wait */
/* owners += ghost copies (ascending neighbour part, ascending slot), ghosts <- 0 */
int pamg_assemble(pamg_ctx* c, int32_t level, double* const* v);                    /* assemble!(v) |> wait */
/* x <- nu sweeps of the configured smoother on A_level x = b (x is in/out) */
int pamg_smooth(pamg_ctx* c, int32_t level, int32_t nu, const double* const* b, double* const* x);
/* bc = R (b - A x); r (may be NULL) receives b - A x.  Two launches: the residual sweep (one pass over A, r written once)
 * and the restriction (one pass over R; its epilogue also writes the coarse level's zero-guess first smoothing step).  A
 * single-pass fusion would need every coarse row to recompute or stage the residuals of its R-support; DESIGN.md "a3" has
 * the traffic count and the measurement behind keeping r in HBM. */
int pamg_residual_restrict(pamg_ctx* c, int32_t level, const double* const* b,
                           const double* const* x, double* const* r, double* const* bc);
/* x += P ec (prolongation and correction in one pass over P: the row epilogue adds into x) */
int pamg_prolong_correct(pamg_ctx* c, int32_t level, const double* const* ec, double* const* x);
int pamg_dot(pamg_ctx* c, int32_t level, const double* const* u, const double* const* v, double* out);
/* x = V-cycle(b) from x = 0 (the preconditioner apply, `ldiv!(x, P, b)` / `solve!(x,S,b)`) */
int pamg_vcycle(pamg_ctx* c, const double* const* b, double* const* x);
/* AMG-preconditioned CG from x = 0 to ||r|| <= rtol ||r0||.  resid_hist (may be NULL) gets
 * hist[0]=||r0||, hist[k]=||r_k||, capacity maxiter+1.  precond=0 runs plain CG. */
int pamg_pcg(pamg_ctx* c, const double* const* b, double* const* x, double rtol, int32_t maxiter,
             int32_t precond, int32_t* iters, double* resid_hist);

/* Flexible AMG-preconditioned CG (Notay): beta = z_{k+1}.(r_{k+1} - r_k) / (z_k.r_k).  Same arguments and results as
 * pamg_pcg with precond = 1; it tolerates a preconditioner that is not a fixed SPD operator (W-cycles, truncated cycles).
 * PartitionedSolvers has no separate entry point for it [RECALL-UNVERIFIED]; the oracle restatement is
 * oracle/amg_oracle.py pcg(flexible=True) / pamg_oracle.c orc_pcg(precond = 2). */
int pamg_fcg(pamg_ctx* c, const double* const* b, double* const* x, double rtol, int32_t maxiter, int32_t* iters,
             double* resid_hist);

/* Restarted flexible GMRES, FGMRES(restart), right-preconditioned by one multigrid cycle (precond = 0: plain restarted
 * GMRES), from x = 0: Arnoldi with modified Gram-Schmidt on w = A M^-1 v_j, Givens rotations; resid_hist[0] = ||b||,
 * resid_hist[k] = the residual estimate |g_k| after inner step k (capacity maxiter + 1); stops at estimate <= rtol ||b|| or
 * after maxiter inner steps.  For operators or cycles that are not symmetric (PartitionedSolvers / IterativeSolvers `gmres`
 * [RECALL-UNVERIFIED]); oracle: amg_oracle.py fgmres / pamg_oracle.c orc_fgmres.  Device memory: (2 restart + 1) vectors. */
int pamg_fgmres(pamg_ctx* c, const double* const* b, double* const* x, double rtol, int32_t maxiter, int32_t restart,
                int32_t precond, int32_t* iters, double* resid_hist);

/* ---- several right-hand sides with one matrix (k solve! calls sharing one setup) ----------
 * The multi calls run k independent single-vector computations, sharing one launch per operation where the block's kernel has a
 * k-wide form (value-indexed and implied-column SELL).  Column j of every result is bit-identical to the single-vector call on
 * column j run with fuse_halo = 0 (which is what one GPU runs anyway).  Vectors: k * nparts pointers, column j of part p at
 * [j * nparts + p] (NULL for parts that are not local).  Multi calls always exchange halos with separate launches. */
#define PAMG_MAX_RHS 8
/* columns of device state the next pamg_device_init allocates (1..PAMG_MAX_RHS, default 1); every process of a job must set the
 * same value (pamg_comm_connect refuses a mismatch) */
int pamg_set_rhs_capacity(pamg_ctx* c, int32_t kmax);
int pamg_spmv_multi(pamg_ctx* c, int32_t level, int32_t k, const double* const* x, double* const* y);
int pamg_vcycle_multi(pamg_ctx* c, int32_t k, const double* const* b, double* const* x);
/* mode 0 CG, 1 AMG-PCG, 2 flexible AMG-PCG; each column has its own scalars, history, count and convergence decision, and a
 * converged column stays frozen while the others continue.  iters[k], converged[k] (may be NULL); resid_hist k x (maxiter + 1),
 * row j = column j, may be NULL.  PAMG_OK when every column converged, else PAMG_ERR_NOTCONV.  pamg_stats: iters = max over
 * columns, r0_norm / r_norm of column 0. */
int pamg_pcg_multi(pamg_ctx* c, int32_t k, const double* const* b, double* const* x, double rtol, int32_t maxiter,
                   int32_t mode, int32_t* iters, int32_t* converged, double* resid_hist);
/* pamg_time_kernel over k columns (kinds 0, 1, 2, 3, 6, 7): the time of the launches that serve all k columns at once, for a
 * comparison of a k-wide launch with k single ones */
int pamg_time_kernel_multi(pamg_ctx* c, int32_t k, int32_t kind, int32_t level, int32_t reps, int32_t flush_l2, float* ms_out);

/* ---- device-resident benchmarking hooks (inputs already in HBM) ------------------------
 * pamg_load_rhs copies b to the device once; pamg_pcg_resident re-solves from x=0 with the
 * resident b and leaves x on the device (pamg_read_solution fetches it). */
int pamg_load_rhs(pamg_ctx* c, const double* const* b);
int pamg_pcg_resident(pamg_ctx* c, double rtol, int32_t maxiter, int32_t precond, int32_t* iters,
                      double* resid_hist);
int pamg_read_solution(pamg_ctx* c, double* const* x);
/* time `reps` launches of one level-`level` kernel with CUDA events on the launching stream,
 * L2 flushed before each when flush_l2 != 0.  kind: 0 spmv, 1 smoother sweep,
 * 2 residual+restrict, 3 prolong+correct, 4 dot, 5 whole V-cycle, 6 spmv + fused dot, 7 smoother sweep + fused dot,
 * 8 reference stream (read + write of a 256 MiB buffer; needs flush_l2).
 * ms_out[reps]. */
int pamg_time_kernel(pamg_ctx* c, int32_t kind, int32_t level, int32_t reps, int32_t flush_l2,
                     float* ms_out);
int pamg_get_stats(pamg_ctx* c, pamg_stats* s);
/* tracing: after pamg_trace_enable(capacity > 0) CTA 0 of every kernel launched for a local part appends its
 * start time (device globaltimer, ns); pamg_trace_read copies and clears the record of one local part;
 * pamg_trace_names returns the newline-separated kernel names of one PCG iteration in launch order. */
int pamg_trace_enable(pamg_ctx* c, int32_t capacity);
int pamg_trace_read(pamg_ctx* c, int32_t part, uint64_t* out, int32_t cap, int32_t* n);
int pamg_trace_names(pamg_ctx* c, char* buf, int32_t cap);

#ifdef __cplusplus
}
#endif
#endif /* PAMG_H */
