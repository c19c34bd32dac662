/*
 * ccqp_b200.h -- C ABI of the B200-native CCQP projected-gradient hot path.
 *
 * This is the drop-in boundary for the path BASELINE.json's north_star names: the loop bodies of
 * the reference's solvers (the per-iteration fp64 A@x mat-vec, the convex projection, the
 * step-length dot products and residual reductions).  The reference is pure Python; each entry
 * point below names the reference interface it replaces (file:line under /root/reference) and
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Rules of the boundary
 *   - extern "C", plain pointers and sizes, no C++/torch types, no exceptions: every call returns a
 *     ccqp_status; ccqp_status_string() gives text.
 *   - Every data pointer is either a HOST or a DEVICE pointer, named by a ccqp_memtype argument.
 *     Host buffers are copied by the library (pinned host memory gives asynchronous copies).
 *   - All reals are IEEE fp64 (a dense Hessian may be stored as fp32: ccqp_set_matrix_f32).  Matrices are row-major
 *     (C order) with leading dimension lda.
 *   - One handle per host thread; a handle owns one CUDA device, one stream and its workspaces.
 *   - There is no CPU fallback: with no usable device ccqp_create() fails with
 *     CCQP_ERR_NO_DEVICE.
 */
#ifndef CCQP_B200_H
#define CCQP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCQP_ABI_VERSION 3

typedef enum ccqp_status {
    CCQP_OK = 0,
    CCQP_ERR_INVALID_ARG = 1,            /* bad shape / null pointer / unknown id                   */
    CCQP_ERR_NO_DEVICE = 2,              /* no CUDA device, or not an sm_100 part                   */
    CCQP_ERR_CUDA = 3,                   /* a CUDA runtime call failed (see ccqp_last_error)        */
    CCQP_ERR_UNSUPPORTED = 4,            /* valid request that this build does not implement        */
    CCQP_ERR_NOT_READY = 5,              /* solve before set_matrix / set_projection                */
    CCQP_ERR_NORMAL_NOT_IMPLEMENTED = 6, /* MPRGP reached normal_vector of a reference Cone block:
                                            the reference raises NotImplementedError there
                                            (solution_spaces.py:465)                                */
    CCQP_ERR_UNIFORMS_EXHAUSTED = 7,     /* SPG consumed every supplied uniform sample              */
    CCQP_ERR_RANGE = 8,                  /* SPG step bound is NaN: np.random.uniform raises
                                            OverflowError there (solvers.py:959)                    */
    CCQP_ERR_DEVICE_TIMEOUT = 9,         /* an in-kernel barrier timed out (~4 s): the kernel trapped.
                                            A trap is a sticky CUDA error: the process's CUDA context
                                            is gone, this handle AND every other handle / CUDA user of
                                            the process are dead; the process has to be restarted      */
    CCQP_ERR_COMM = 10                   /* multi-GPU exchange setup failed                         */
} ccqp_status;

typedef enum ccqp_memtype { CCQP_MEM_HOST = 0, CCQP_MEM_DEVICE = 1 } ccqp_memtype;

/* Leaf projection operators.  One block == one leaf operator of the reference; a table with
 * several blocks is the reference's DisjointProjOp (solution_spaces.py:495-560).             */
typedef enum ccqp_block_kind {
    CCQP_BLOCK_IDENTITY = 0, /* IdentityProjOp   solution_spaces.py:77   params: none               */
    CCQP_BLOCK_LOWER = 1,    /* LowerBoundProjOp solution_spaces.py:128  params: lb[dim]            */
    CCQP_BLOCK_UPPER = 2,    /* UpperBoundProjOp solution_spaces.py:204  params: ub[dim]            */
    CCQP_BLOCK_BOX = 3,      /* BoxProjOp        solution_spaces.py:280  params: lb[dim], ub[dim]   */
    CCQP_BLOCK_SPHERE = 4,   /* SphereProjOp     solution_spaces.py:369  params: radius             */
    CCQP_BLOCK_CONE_REF = 5, /* ConeProjOp       solution_spaces.py:438  params: aspect ratio mu;
                                bug-compatible with the reference ("this projection op is bugged") */
    CCQP_BLOCK_SOC = 6       /* extension: the correct second-order-cone projection {|u| <= mu z};
                                not in the reference, parity unpinned                               */
} ccqp_block_kind;

typedef struct ccqp_block {
    int32_t kind;      /* ccqp_block_kind                                  */
    int32_t reserved;  /* must be 0                                        */
    int64_t offset;    /* first element of the block; blocks tile [0,n)    */
    int64_t dim;       /* embedded_dimension of the leaf operator          */
    int64_t param_off; /* offset of the block's parameters in params[]     */
} ccqp_block;

/* Solvers.  The ids are the rows of SURVEY.md section 8(a). */
typedef enum ccqp_solver {
    CCQP_SOLVER_PGD = 0,     /* CCQPSolverPGD.solve                 solvers.py:94-170    */
    CCQP_SOLVER_APGD = 1,    /* CCQPSolverAPGD.solve                solvers.py:220-343   */
    CCQP_SOLVER_APGD_AR = 2, /* CCQPSolverAPGDAntiRelaxation.solve  solvers.py:393-533   */
    CCQP_SOLVER_BBPGD = 3,   /* CCQPSolverBBPGD.solve               solvers.py:583-669   */
    CCQP_SOLVER_BBPGDF = 4,  /* CCQPSolverBBPGDf.solve              solvers.py:719-819   */
    CCQP_SOLVER_SPG = 5,     /* CCQPSolverSPG.solve                 solvers.py:878-975   */
    CCQP_SOLVER_MPRGP = 6    /* CCQPSolverMPRGP.solve               solvers.py:1026-1200 */
} ccqp_solver;

/* Constructor arguments of the reference's solver classes (solvers.py:81, :208, :571, :856). */
typedef struct ccqp_params {
    double tol;       /* desired_residual_tol                                                   */
    double max_mv;    /* max_matrix_vector_multiplications; +inf allowed (the reference default) */
    double step_size; /* PGD only (solvers.py:81), default 0.01                                  */
    double tau;       /* SPG (solvers.py:856), default 0.5                                       */
    double sigma1;    /* SPG, default 0.01                                                       */
    double sigma2;    /* SPG, default 0.5                                                        */
    int32_t m;        /* SPG non-monotone window, default 5 (1..64)                              */
    int32_t reserved;
} ccqp_params;

/* Result fields of the reference (solvers.py:163-168) plus accounting for the roofline. */
typedef struct ccqp_result {
    double residual;       /* solution_residual (NaN where the reference would raise NameError) */
    double gpu_seconds;    /* device time of the solve, CUDA events on the handle's stream       */
    double hbm_bytes;      /* algorithmic bytes moved: gemv_count * (8 n_rows n + 8 n + 8 n_rows);
                              an fp32 Hessian (ccqp_set_matrix_f32): gemv_count * (4 n_rows n + 8 n + 8 n_rows) */
    int64_t mv_count;      /* solution_num_matrix_vector_multiplications (the REPORTED count)    */
    int64_t gemv_count;    /* mat-vec products actually executed on the device                   */
    int64_t iterations;    /* outer iterations completed                                         */
    int64_t uniforms_used; /* SPG: samples consumed from uniforms[]                              */
    int32_t converged;     /* solution_converged = mv_count < max_mv                             */
    int32_t status;        /* ccqp_status raised inside the kernel (0 = none)                    */
    int64_t kernel_launches; /* kernels launched by the call                                     */
} ccqp_result;

typedef struct ccqp_handle ccqp_handle;

/* ---- lifetime ------------------------------------------------------------------------------ */
int ccqp_abi_version(void);
const char* ccqp_status_string(int status);
/* Text of the last CUDA error seen by this handle (empty string if none). */
const char* ccqp_last_error(const ccqp_handle* h);

/* Create a handle on CUDA device `device` (-1 = current device).  Fails with
 * CCQP_ERR_NO_DEVICE when there is none: there is no CPU path behind this ABI. */
ccqp_status ccqp_create(ccqp_handle** out, int device);
ccqp_status ccqp_destroy(ccqp_handle* h);
/* Use an existing cudaStream_t (e.g. torch's current stream) instead of the handle's own. */
ccqp_status ccqp_set_stream(ccqp_handle* h, void* cuda_stream);
/* Number of SMs of the handle's device and its memory clock/bus derived peak are not exposed;
 * the kernel grid the dense solver will use is. */
ccqp_status ccqp_get_info(const ccqp_handle* h, int32_t* sm_count, int32_t* dense_grid,
                          int32_t* dense_threads, int64_t* dense_smem_bytes);

/* ---- problem data -------------------------------------------------------------------------- */
/* The Hessian.  Replaces the `A` argument of solve() (solvers.py:94); the reference touches A
 * only through A.dot(v) (26 call sites, SURVEY.md section 8b).  `A` points at rows
 * [row_begin, row_begin+n_rows) of the n x n matrix (row shard; single GPU: row_begin = 0,
 * n_rows = n).  A DEVICE matrix is borrowed, not copied, and must outlive the solves.  A HOST
 * matrix is copied on the handle's stream: from pinned memory that copy is asynchronous, so the
 * buffer must stay valid until the next ccqp_solve() / ccqp_solve_wait() on the handle returns. */
ccqp_status ccqp_set_matrix(ccqp_handle* h, const double* A, int64_t n, int64_t lda,
                            int64_t row_begin, int64_t n_rows, int memtype);

/* What the last ccqp_set_matrix() from HOST memory moved.  A whole matrix (row_begin = 0, n_rows = n, n >= 2048) that is
 * symmetric crosses PCIe as its upper block triangle only (row blocks of ccqp_upload_block_rows() rows, each from its first
 * column on): the copies are enqueued first, host threads then compare A[i][j] with A[j][i] for every entry below the block
 * diagonal while the copy engine works, and a device kernel mirrors the uploaded part -- the device copy is bit-identical to
 * a full upload.  (The test runs only where the process has at least 12 hardware threads: it reads all of A.)  A matrix that is not symmetric (or holds a NaN, or a -0.0 / +0.0 pair) gets its remaining blocks uploaded
 * after all.  The reference takes any square A (solvers.py:94, A.dot(v) at :133); the solver sees exactly that matrix
 * either way.  CCQP_SYM_UPLOAD=0 in the environment turns the scheme off. */
ccqp_status ccqp_get_upload_info(ccqp_handle* h, int64_t* bytes, int32_t* mirrored);
/* ccqp_set_matrix() for a whole matrix the CALLER declares symmetric (the dsymv('U') contract at the granularity of
 * ccqp_upload_block_rows() rows): from host memory only the upper block triangle is read and uploaded, no test is made, and
 * the solver works on that triangle mirrored -- which is A itself when the declaration is true.  Device memory: the same as
 * ccqp_set_matrix (A is used in place, both triangles are read).  Saves the host-side test, which reads all of A and competes
 * with the copy engine for host memory bandwidth (n = 32768: a stream of solves at ~80 ms per solve instead of ~140). */
ccqp_status ccqp_set_matrix_symmetric(ccqp_handle* h, const double* A, int64_t n, int64_t lda, int memtype);
/* The host-side test of that scheme (pure host code, usable without a GPU): 1 if every entry below the block diagonal
 * equals its mirror image bit for bit and is not a NaN, 0 if not, -1 for invalid arguments.  threads <= 0: all the
 * process may run on. */
int32_t ccqp_host_matrix_is_block_symmetric(const double* A, int64_t n, int64_t lda, int32_t threads);
int32_t ccqp_upload_block_rows(void);

/* ccqp_set_matrix() for a Hessian STORED as IEEE fp32 (lda counted in floats).  The arithmetic stays fp64: every entry is
 * widened exactly in a register in front of its fma, which is what NumPy does for the reference's A.dot(v) with a float32 A
 * (solvers.py:133), and the mat-vec keeps the fp64 kernels' summation order -- a solve returns the same bits as the fp64
 * solve of the widened matrix (same lda parity: rows with 16-byte aligned starts and lda % 4 == 0 take the vector loop,
 * like 32-byte aligned fp64 rows; others the scalar loop).  A DEVICE matrix is borrowed, neither copied nor widened; a
 * HOST matrix is copied into padded fp32 rows (asynchronous from pinned memory, same lifetime rule as ccqp_set_matrix).
 * Half the HBM bytes per mat-vec (result.hbm_bytes counts 4 per entry), half the PCIe bytes of an upload
 * (ccqp_get_upload_info: 4 * n_rows * n, never mirrored).  Replaces any previous matrix of the handle. */
ccqp_status ccqp_set_matrix_f32(ccqp_handle* h, const float* A, int64_t n, int64_t lda, int64_t row_begin, int64_t n_rows,
                                int memtype);

/* Operator-form Hessian in CSR.  The reference accepts any `A` with a .dot (solvers.py:133), in particular
 * scipy.sparse matrices (contact-style Hessians D^T M^-1 D are sparse); this is that case.  indptr has
 * n_rows + 1 entries RELATIVE to the shard (indptr[0] = 0, indptr[n_rows] = nnz), indices are column ids
 * in [0, n).  DEVICE arrays are borrowed, HOST arrays are copied.  Replaces a previous ccqp_set_matrix(). */
ccqp_status ccqp_set_matrix_csr(ccqp_handle* h, const int64_t* indptr, const int32_t* indices, const double* values,
                                int64_t n, int64_t nnz, int64_t row_begin, int64_t n_rows, int memtype);

/* The feasible set.  Replaces the `convex_proj_op` argument of solve() (solvers.py:94) and the
 * operator classes of solution_spaces.py.  blocks must tile [0,n) in order.  Host pointers. */
ccqp_status ccqp_set_projection(ccqp_handle* h, const ccqp_block* blocks, int64_t n_blocks,
                                const double* params, int64_t n_params);

/* ---- the hot path -------------------------------------------------------------------------- */
/* One whole solve on the device: replaces CCQPSolver{PGD,APGD,APGDAntiRelaxation,BBPGD,BBPGDf,
 * SPG,MPRGP}.solve (solvers.py:94,220,393,583,719,878,1026).  b, x0 (nullable = zeros), uniforms
 * and x_out use `memtype`.  uniforms[] is the U[0,1) stream SPG's np.random.uniform (solvers.py:959)
 * would consume; ignored by the other solvers. */
ccqp_status ccqp_solve(ccqp_handle* h, int solver, const ccqp_params* params, const double* b,
                       const double* x0, const double* uniforms, int64_t n_uniforms, double* x_out,
                       int memtype, ccqp_result* result);

/* The same solve split in two, so that a caller with several handles (each has its own stream) can
 * overlap the host->device copy of the NEXT problem's Hessian with the solve of the current one:
 * ccqp_solve_async() enqueues the input copies, the solver kernel and the result copies on the
 * handle's stream and returns; ccqp_solve_wait() synchronises and fills `result`.  Host buffers
 * (b, x0, uniforms, x_out, and a host matrix given to ccqp_set_matrix) must stay valid -- and be
 * pinned, for the copies to be asynchronous -- until the wait.  One solve in flight per handle. */
ccqp_status ccqp_solve_async(ccqp_handle* h, int solver, const ccqp_params* params, const double* b,
                             const double* x0, const double* uniforms, int64_t n_uniforms, double* x_out,
                             int memtype);
ccqp_status ccqp_solve_wait(ccqp_handle* h, ccqp_result* result);

/* Many small independent box-constrained QPs, one CTA per problem, whole solver loop on the
 * device.  Problem i is defined to equal
 *     CCQPSolverX(tol,max_mv).solve(A[i], b[i], x0[i], BoxProjOp(n, lb[i], ub[i]))
 * (solvers.py:94.. with solution_spaces.py:280).  A is [batch][n][n]; b, x0 (nullable), lb, ub,
 * x_out are [batch][n]; uniforms is [batch][n_uniforms] (SPG); results is [batch] in HOST memory.
 * Supported n: 1..128; all seven solvers.  n <= 64 (the tuned case): 64 threads per problem, up to 6 problems in flight per SM;
 * 64 < n <= 128: 256 threads per problem, one problem per SM; larger n: CCQP_ERR_UNSUPPORTED (use ccqp_solve). */
ccqp_status ccqp_solve_batched(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch,
                               int64_t n, const double* A, const double* b, const double* x0,
                               const double* lb, const double* ub, const double* uniforms,
                               int64_t n_uniforms, double* x_out, int memtype,
                               ccqp_result* results, ccqp_result* summary);

/* The same for a caller that declares every A[i] SYMMETRIC (the reference's objective 0.5 x'Ax + b'x has the gradient Ax + b
 * its solvers iterate with, solvers.py:133, only for such an A).  Where the one-warp-per-problem kernels apply -- n <= 64 and
 * solver PGD / BBPGD / BBPGDf / SPG -- only the upper block triangle of A[i] is read: entries A[i][r][c] with c >= 8 * (r / 8),
 * the dsymv('U') contract at 8 x 8 granularity; the blocks below are never touched (18 KB instead of 32 KB of HBM traffic per
 * problem at n = 64, eight problems in flight per SM instead of six).  Every other case runs ccqp_solve_batched's kernels
 * on the full matrix -- the same answer for a symmetric A.  Results equal ccqp_solve_batched's up to the summation order of
 * the mat-vec (last-bit differences). */
ccqp_status ccqp_solve_batched_sym(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch,
                                   int64_t n, const double* A, const double* b, const double* x0,
                                   const double* lb, const double* ub, const double* uniforms,
                                   int64_t n_uniforms, double* x_out, int memtype,
                                   ccqp_result* results, ccqp_result* summary);

/* The same with ONE feasible set shared by all problems of the batch, given as a block table (any block kinds:
 * DisjointProjOp of Box / Lower / Upper / Identity / Sphere / reference Cone / SOC leaves, solution_spaces.py:77-560) --
 * the contact-style case: every problem has the same friction-disc structure.  Problem i equals
 *     CCQPSolverX(tol,max_mv).solve(A[i], b[i], x0[i], op)        with op described by blocks / block_params
 * (host pointers, as for ccqp_set_projection).  All solvers except MPRGP (CCQP_ERR_UNSUPPORTED). */
ccqp_status ccqp_solve_batched_table(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch,
                                     int64_t n, const double* A, const double* b, const double* x0,
                                     const ccqp_block* blocks, int64_t n_blocks, const double* block_params,
                                     int64_t n_params, const double* uniforms, int64_t n_uniforms, double* x_out,
                                     int memtype, ccqp_result* results, ccqp_result* summary);

/* The same block STRUCTURE for all problems, each problem with its own parameter VALUES (bounds, radii, aspect ratios) --
 * a batch of contact problems: k friction discs in every scene, disc radius mu * f_n of each contact.  Problem i equals
 *     CCQPSolverX(tol,max_mv).solve(A[i], b[i], x0[i], op_i)
 * where op_i is the table `blocks` (HOST pointer, shared) with the parameter array block_params + i * n_params: block_params
 * is [batch][n_params], row i laid out as op_i's own parameter array, and lives where A lives (`memtype`: a device array is
 * read in place, a host array is copied with the other inputs).  Argument checks as ccqp_solve_batched_table; n > 128:
 * CCQP_ERR_UNSUPPORTED; all solvers except MPRGP (CCQP_ERR_UNSUPPORTED).  result.hbm_bytes counts the 8 * n_params bytes
 * of each problem's row. */
ccqp_status ccqp_solve_batched_tables(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch,
                                      int64_t n, const double* A, const double* b, const double* x0,
                                      const ccqp_block* blocks, int64_t n_blocks, const double* block_params,
                                      int64_t n_params, const double* uniforms, int64_t n_uniforms, double* x_out,
                                      int memtype, ccqp_result* results, ccqp_result* summary);

/* The four batched calls for a Hessian batch STORED as IEEE fp32: A is float [batch][n][n], contiguous; every other argument,
 * check and status code is that of the fp64 function of the same name without _f32.  The arithmetic stays fp64: every
 * entry is widened exactly in a register when the problem's A is loaded, which is what NumPy does for the reference's
 * A.dot(v) with a float32 A (solvers.py:133), and nothing after that load depends on the storage type -- on every path
 * (host or device A, any alignment, any n, symmetric or general kernels, box or table) the solutions, residuals, counts,
 * converged flags and statuses equal bit for bit those of the fp64 call on A widened to double.  A DEVICE batch is read in
 * place (any 4-byte alignment: a base off a 16-byte boundary, or n % 4 != 0, loads entry by entry instead of by bulk row
 * copies); a HOST batch is copied to the device at 4 bytes per entry (asynchronous from pinned memory).  Half the HBM and
 * PCIe bytes of A: result.hbm_bytes and summary.hbm_bytes count 4 bytes per entry of A read (ccqp_solve_batched_sym_f32:
 * per entry of the upper block triangle, where that kernel runs). */
ccqp_status ccqp_solve_batched_f32(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch,
                                   int64_t n, const float* A, const double* b, const double* x0,
                                   const double* lb, const double* ub, const double* uniforms,
                                   int64_t n_uniforms, double* x_out, int memtype,
                                   ccqp_result* results, ccqp_result* summary);
ccqp_status ccqp_solve_batched_sym_f32(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch,
                                       int64_t n, const float* A, const double* b, const double* x0,
                                       const double* lb, const double* ub, const double* uniforms,
                                       int64_t n_uniforms, double* x_out, int memtype,
                                       ccqp_result* results, ccqp_result* summary);
ccqp_status ccqp_solve_batched_table_f32(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch,
                                         int64_t n, const float* A, const double* b, const double* x0,
                                         const ccqp_block* blocks, int64_t n_blocks, const double* block_params,
                                         int64_t n_params, const double* uniforms, int64_t n_uniforms, double* x_out,
                                         int memtype, ccqp_result* results, ccqp_result* summary);
ccqp_status ccqp_solve_batched_tables_f32(ccqp_handle* h, int solver, const ccqp_params* params, int64_t batch,
                                          int64_t n, const float* A, const double* b, const double* x0,
                                          const ccqp_block* blocks, int64_t n_blocks, const double* block_params,
                                          int64_t n_params, const double* uniforms, int64_t n_uniforms, double* x_out,
                                          int memtype, ccqp_result* results, ccqp_result* summary);

/* ---- unit-test hooks for the pieces of the path ---------------------------------------------- */
/* y = A v for the handle's row shard (y has n_rows entries).  A.dot(v), solvers.py:133 etc. */
ccqp_status ccqp_gemv(ccqp_handle* h, const double* v, double* y, int memtype);
/* Measurement hook: `repeats` back-to-back mat-vec kernels on device-resident v (n entries, padded
 * by the caller to n+64 zeros) and y; returns the mean device time per launch (CUDA events). */
ccqp_status ccqp_gemv_timed(ccqp_handle* h, const double* v_dev, double* y_dev, int repeats, double* seconds);
/* out = P(x): ProjOp.__call__, solution_spaces.py:125,200,276,363,431,484,553. */
ccqp_status ccqp_project(ccqp_handle* h, const double* x, double* out, int memtype);
/* out = normal_vector(x): solution_spaces.py:92,146,222,306,389,459,512. */
ccqp_status ccqp_normal(ccqp_handle* h, const double* x, double* out, int memtype);

/* (free, chopped) = projected_gradient(x, g): solution_spaces.py:162-184 (Lower), :238-260 (Upper), :324-347 (Box, its
 * activity test as written), :527-538 (Disjoint: leaf by leaf, each with its own leaf's normal_vector).  Elementwise
 * kinds only: a table with a Sphere / SOC leaf returns CCQP_ERR_UNSUPPORTED (the reference raises NotImplementedError,
 * :415), one with a reference Cone leaf CCQP_ERR_NORMAL_NOT_IMPLEMENTED; Identity leaves come back as (g, 0) -- the
 * host mirror reproduces the reference's None / TypeError for them. */
ccqp_status ccqp_projected_gradient(ccqp_handle* h, const double* x, const double* g, double* free_out,
                                    double* chopped_out, int memtype);

/* q_k[i] = a_k[i] / b[i], k = 0..2, evaluated with the shared-reciprocal routine the batched SPG kernel uses
 * for its three divisions by d.Ad (solvers.py:954,955,966); must equal IEEE division bit for bit. DEVICE pointers. */
ccqp_status ccqp_debug_divide(ccqp_handle* h, const double* a0, const double* a1, const double* a2, const double* b,
                            double* q0, double* q1, double* q2, int64_t count);

/* ---- measurement hooks (roofline denominators; nothing here is on the solve path) -------------
 * Measured FP64 throughput of the handle's device in TFLOP/s (2 flops per DFMA): every thread of
 * blocks_per_sm x threads_per_block resident threads per SM runs 8 independent DFMA chains.  With
 * the SM full (8 x 256) this is the fp64 term of the batched mode's roofline,
 * max(HBM bytes / BW, 2 n^2 * mat-vecs / FP64 peak) (BASELINE.md section 4); with 6 x 64 it is what
 * the batched kernel's own occupancy could issue if it executed nothing but its mat-vec DFMAs. */
ccqp_status ccqp_fp64_peak(ccqp_handle* h, int blocks_per_sm, int threads_per_block, double* tflops);
/* SM cycles per dependent operation, one warp, in the order DFMA, DADD, DMUL, SHFL.64+DADD, IEEE
 * division+DADD, sqrt+DADD, LDS.128 (all lanes one address)+DADD, LDS.128 (distinct)+DADD,
 * STS+bar+LDS+DADD+bar, bar.sync (64 threads), DSETP+select+DADD, then the FP64 tensor path (DMMA.884 dependent,
 * 8 independent, a 32-lane sum as DMMA+DADD+DMMA against 5 shuffle stages, DMMA mixed with DFMA), then the issue interval of
 * INDEPENDENT DFMAs per instruction: 8 chains with one fresh register operand, with two, and the 8 x 8 register-block mat-vec of
 * the batched kernels (two fresh operands, 64 distinct multiplicands).  n_out >= 19.  Feeds the cycle model of the batched
 * kernel in DESIGN.md. */
ccqp_status ccqp_microbench(ccqp_handle* h, double* cycles_per_op, int32_t n_out);

/* ---- multi-GPU (row-sharded dense solves, one process per GPU) --------------------------------
 * Nothing in the reference corresponds to this (it is single-process NumPy).  A is row-sharded:
 * every rank calls ccqp_set_matrix() with its rows [row_begin, row_begin+n_rows) and the FULL
 * projection table; the vectors are kept in full on every rank.  Setup, once per problem size:
 *   1. ccqp_comm_export(): allocate this rank's exchange buffer, get an opaque descriptor (CUDA IPC)
 *   2. the host all-gathers the descriptors (torch.distributed / MPI / files: the ABI does not care)
 *   3. ccqp_comm_attach(): map every peer's buffer over NVLink
 * Per solve: ccqp_comm_prepare() (clears the buffer), a HOST barrier across ranks, then ccqp_solve()
 * on every rank with the same arguments.  Inside the solver kernel each rank writes the rows of
 * every mat-vec result it computes straight into the peers' buffers (the all-gather, fused into the
 * mat-vec epilogue) and the sync that closes the mat-vec phase exchanges the scalar partial sums and
 * synchronises the ranks through 8-byte {data, epoch} packets in peer memory: no collective
 * launches inside the loop.  Every rank returns the full solution and identical result fields. */
#define CCQP_COMM_DESC_BYTES 128
ccqp_status ccqp_comm_export(ccqp_handle* h, int rank, int world, int64_t n, void* desc);
ccqp_status ccqp_comm_attach(ccqp_handle* h, const void* all_descs /* world * CCQP_COMM_DESC_BYTES */);
ccqp_status ccqp_comm_prepare(ccqp_handle* h);
ccqp_status ccqp_comm_detach(ccqp_handle* h);


/* ---- test vehicle: the ranks of a row-sharded solve emulated on ONE device --------------------
 * `world` handles created on the same device play ranks 0..world-1: ccqp_debug_emulate_ranks() gives each
 * 1/world of the SMs and wires the "peer" buffers to each other (no IPC); after ccqp_set_matrix() (each
 * handle its own row shard) and ccqp_set_projection() on every handle, ccqp_debug_solve_emulated() runs all
 * ranks inside ONE cooperative launch (CTAs [r*G,(r+1)*G) are rank r).  The kernel code executed is that of
 * a real sharded solve (fused all-gather into the peers' buffers, {data, epoch} packet all-reduce, the
 * cross-rank barrier); only the stores do not cross NVLink.  It exists so that the exchange protocol is
 * covered on single-GPU test boxes.  x_out holds world * n entries (every rank's copy of the solution),
 * results has world entries. */
ccqp_status ccqp_debug_emulate_ranks(ccqp_handle* const* handles, int world, int64_t n);
ccqp_status ccqp_debug_solve_emulated(ccqp_handle* const* handles, int world, int solver, const ccqp_params* params,
                                      const double* b, const double* x0, const double* uniforms, int64_t n_uniforms,
                                      double* x_out, int memtype, ccqp_result* results);

#ifdef __cplusplus
}
#endif
#endif /* CCQP_B200_H */
