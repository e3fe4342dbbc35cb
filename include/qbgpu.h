/* include/qbgpu.h -- C ABI of the B200-native H*v path (libqbgpu.so).
 *
 * Drop-in boundary for wztzjhn/quantum_basis.  The reference keeps its sparse backend behind an opaque MKL
 * inspector-executor handle (`sparse_matrix_t handle`, src/qbasis.h:985): created in csr_mat's constructors
 * (src/sparse.cc:129,258), used by csr_mat<T>::MultMv2 (src/sparse.cc:262-289) and destroyed in destroy()/dtor
 * (src/sparse.cc:165,185).  This header declares the same quartet (create / mv / destroy) for a B200, plus the
 * device-resident Krylov loops that replace the bodies of lanczos(), eigenvec_CG() and energy_scale()
 * (src/lanczos.cc:134-341, src/kpm.cc:45-88) so that one Krylov step makes one pass over H and the vectors.
 *
 * Conventions
 *   - plain C: pointers and sizes only; complex numbers are interleaved (re,im) doubles, layout-compatible with
 *     std::complex<double> / MKL_Complex16; indices on the host side are int64 (MKL_INT under -DMKL_ILP64).
 *   - every function returns 0 on success, non-zero on failure; qbgpu_last_error() gives the message (the C++
 *     adaptor include/qbgpu_csr_mat.hpp turns it into std::runtime_error like src/sparse.cc:130,259,288).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with QBGPU_ERR_CUDA.
 *   - `where` says where vector pointers live: QBGPU_HOST (the reference's calling convention: std::vector /
 *     ARPACK workd) or QBGPU_DEVICE (already resident, e.g. a torch tensor's data_ptr).
 *   - all work is issued on one CUDA stream per thread context (qbgpu_set_stream to adopt the caller's).
 *   - device vectors: complex vectors 16-byte aligned (read as double2), fp64 vectors 8-byte aligned.  Any such pointer
 *     works, e.g. a window of a larger vector; an fp64 x that is also 16-byte aligned lets pass 1 of a species-order
 *     product copy each block of x with one bulk copy instead of thread by thread.
 */
#ifndef QBGPU_H
#define QBGPU_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define QBGPU_OK            0
#define QBGPU_ERR_ARG       1
#define QBGPU_ERR_CUDA      2
#define QBGPU_ERR_ALLOC     3
#define QBGPU_ERR_STATE     4
#define QBGPU_ERR_NUMERIC   5   /* breakdown, non-Hermitian input, ... */

#define QBGPU_HOST   0
#define QBGPU_DEVICE 1

/* create flags */
#define QBGPU_KEEP_COMPLEX   1   /* do not demote an all-real complex matrix to fp64 values */
#define QBGPU_NO_AUTOTUNE    2   /* skip the kernel-variant timing pass at create */
#define QBGPU_FORMAT_CSR     4   /* force the expanded-CSR kernels  */
#define QBGPU_FORMAT_SELL    8   /* force the sliced-jagged kernels (32-row slices, jagged diagonals, no padding); refused
                                    for a row of 2^24 or more entries */
#define QBGPU_FORMAT_MATFREE 32  /* (info only) matrix-free handle: rows are regenerated inside the product */
#define QBGPU_MATFREE_TERMS 64  /* qbgpu_create_matfree_*: also store one byte per entry naming the Hamiltonian term that
                                  * produces it (directed bond x spin), so the product replays each row -- column from the
                                  * Lin tables, sign from the occupancy words -- without searching for applicable terms */
#define QBGPU_SPECIES_ORDER 128 /* qbgpu_build_hubbard / qbgpu_create_matfree_hubbard: keep the vectors INTERNALLY in the order
                                  * (rank of the up configuration, rank of the down configuration) and multiply in two passes
                                  * (see "species order" below); results and calling convention are unchanged */
#define QBGPU_VALUE_DICT    16   /* opt-in: store fp64 values as 1-byte codes into a table of the distinct values when there
                                    are at most 256 of them (lossless; products are bit-identical); implies FORMAT_SELL, and
                                    like it refuses a row of 2^24 or more entries (default create keeps such a matrix in the
                                    CSR layout).  Stored species-order handles pack their values without it (see "species order") */

typedef struct qbgpu_matrix *qbgpu_matrix_t;     /* replaces `sparse_matrix_t handle` (src/qbasis.h:985) */

typedef struct {
    int64_t n;              /* global dimension                                                    */
    int64_t row_lo, row_hi; /* rows held by this handle ([0,n) unless created as a shard)          */
    int64_t nnz_stored;     /* entries in the device layout (full expanded Hermitian rows)         */
    int64_t nnz_input;      /* entries of the host CSR it was created from (upper triangle if sym) */
    int     val_is_real;    /* 1: values stored as fp64 (input was real or all imaginary parts == 0) */
    int     value_dict;     /* > 0: number of dictionary entries; values are stored as 1-byte codes (QBGPU_VALUE_DICT)
                               or, on a stored species-order handle, as codes packed beside the columns */
    int     api_is_complex; /* 1: created through a z entry point                                  */
    int     format;         /* QBGPU_FORMAT_CSR or QBGPU_FORMAT_SELL                               */
    int     lanes;          /* threads per row chosen for the CSR-vector kernel                    */
    int64_t device_bytes;   /* HBM held by the matrix                                              */
    double  upload_seconds, convert_seconds, autotune_seconds;
} qbgpu_matrix_info;

/* ------------------------------------------------------------------------------------------- context */
int         qbgpu_init(int device);              /* binds the calling thread to `device`; idempotent          */
int         qbgpu_finalize(void);
int         qbgpu_device_count(int *count);
int         qbgpu_set_stream(void *cuda_stream); /* NULL: back to the context's own stream                    */
int         qbgpu_synchronize(void);
const char *qbgpu_last_error(void);
const char *qbgpu_version(void);

/* --------------------------------------------------------------------------- matrix create / destroy
 * Replaces mkl_sparse_{d,z}_create_csr as called by create_handle (src/sparse.cc:24-40): 4-array zero-based CSR,
 * row i = [row_start[i], row_end[i]).  sym_upper != 0 is csr_mat::sym (src/qbasis.h:981): only col >= row is
 * stored and (i,j>i,v) stands for v at (i,j) and conj(v) at (j,i).  The device copy is independent of the host
 * arrays (they may be freed, cf. HamMat_csr_repr[0].destroy() in the reference's examples).
 * PRECONDITION (checked; QBGPU_ERR_ARG otherwise): the referenced columns of every row are strictly ascending -- what
 * csr_mat(lil_mat&) always produces (src/sparse.cc:202-233: the LIL rows are sorted lists).  With sym_upper the entries
 * below the diagonal are not referenced (FILL_UPPER) and may be in any order.
 * The *_shard variants keep only rows [row_lo,row_hi) of the expanded matrix (multi-GPU row partition). */
int qbgpu_create_dcsr(qbgpu_matrix_t *A, int64_t n, const int64_t *row_start, const int64_t *row_end,
                      const int64_t *col, const double *val, int sym_upper, int flags);
int qbgpu_create_zcsr(qbgpu_matrix_t *A, int64_t n, const int64_t *row_start, const int64_t *row_end,
                      const int64_t *col, const void *val, int sym_upper, int flags);
int qbgpu_create_dcsr_shard(qbgpu_matrix_t *A, int64_t n, const int64_t *row_start, const int64_t *row_end,
                            const int64_t *col, const double *val, int sym_upper, int flags,
                            int64_t row_lo, int64_t row_hi);
int qbgpu_create_zcsr_shard(qbgpu_matrix_t *A, int64_t n, const int64_t *row_start, const int64_t *row_end,
                            const int64_t *col, const void *val, int sym_upper, int flags,
                            int64_t row_lo, int64_t row_hi);
int qbgpu_destroy(qbgpu_matrix_t A);             /* replaces mkl_sparse_destroy (src/sparse.cc:165,185)        */
int qbgpu_matrix_get_info(qbgpu_matrix_t A, qbgpu_matrix_info *info);
/* csr_mat<T>::to_dense (src/sparse.cc:299-315): column-major n x n, complex interleaved when api_is_complex. */
int qbgpu_to_dense(qbgpu_matrix_t A, void *dense_host);
/* copy the expanded device rows back (tests): rowptr[n_local+1], col[nnz], val[nnz] (complex unless val_is_real) */
int qbgpu_download_expanded(qbgpu_matrix_t A, int64_t *rowptr, int32_t *col, void *val);

/* A second handle on the SAME device arrays that takes fp64 vectors (d entry points).  Only for handles whose stored
 * values are real (val_is_real): a real H applied to a real vector stays real, so a Krylov loop started from
 * vec_randomize (imag = 0, src/miscellaneous.cc:382) can run on half the vector bytes.  Destroy the view before A. */
int qbgpu_real_view(qbgpu_matrix_t A, qbgpu_matrix_t *view);

/* Split a (shard) handle into `nparts` handles by column range: part p keeps the entries with
 * col_bounds[p] <= col < col_bounds[p+1] of the same rows (col_bounds[0] = 0, col_bounds[nparts] = n, nparts <= 16).
 * Used to multiply the block owned by rank p as soon as p's slice of x has arrived.  A is left intact. */
int qbgpu_split_columns(qbgpu_matrix_t A, int nparts, const int64_t *col_bounds, qbgpu_matrix_t *parts, int flags);

/* nnz-balanced contiguous row partition of the EXPANDED matrix over `parts` shards (host only, no GPU needed):
 * bounds[parts+1], bounds[0]=0, bounds[parts]=n. */
int qbgpu_partition_rows(int64_t n, const int64_t *row_start, const int64_t *row_end, const int64_t *col,
                         int sym_upper, int parts, int64_t *bounds);

/* ------------------------------------------------------------------------------------ H*v products
 * Replaces mkl_sparse_{d,z}_mv as csr_mat<T>::MultMv2 calls it (src/sparse.cc:287): y = alpha*H*x + beta*y.
 * MultMv2 is (alpha,beta) = (1,1); MultMv (src/sparse.cc:291-297) is (1,0).  x has n entries; y has the handle's
 * row_hi-row_lo entries.  A `z` handle with real stored values still takes complex x,y. */
int qbgpu_dmv(qbgpu_matrix_t A, double alpha, const double *x, double beta, double *y, int where);
int qbgpu_zmv(qbgpu_matrix_t A, const double alpha[2], const void *x, const double beta[2], void *y, int where);
/* pin a host range so that `where == QBGPU_HOST` products use asynchronous chunked copies (ARPACK's workd) */
int qbgpu_host_register(void *ptr, size_t bytes);
int qbgpu_host_unregister(void *ptr);

/* ------------------------------------------------------------------------------ device vector helpers */
int qbgpu_malloc(void **dptr, size_t bytes);
int qbgpu_free(void *dptr);
int qbgpu_memcpy_h2d(void *dst, const void *src, size_t bytes);
int qbgpu_memcpy_d2h(void *dst, const void *src, size_t bytes);
int qbgpu_memcpy_d2d(void *dst, const void *src, size_t bytes);     /* stream-ordered, asynchronous */
int qbgpu_memset0(void *dptr, size_t bytes);
/* vec_randomize (src/miscellaneous.cc:371-388) generated on the device, bit-identical element values */
int qbgpu_vec_randomize_d(int64_t n, double *x_dev, uint32_t seed);
int qbgpu_vec_randomize_z(int64_t n, void *x_dev, uint32_t seed);
/* BLAS-1 on device vectors, the calls lanczos.cc makes through cblas_* (src/lanczos.cc:10-53). */
int qbgpu_zdotc(int64_t n, const void *x, const void *y, double result[2]);   /* conj(x).y */
int qbgpu_ddot(int64_t n, const double *x, const double *y, double *result);
int qbgpu_dznrm2(int64_t n, const void *x, double *result);
int qbgpu_dnrm2(int64_t n, const double *x, double *result);
int qbgpu_zaxpy(int64_t n, const double a[2], const void *x, void *y);
int qbgpu_daxpy(int64_t n, double a, const double *x, double *y);
int qbgpu_zscal(int64_t n, const double a[2], void *x);
int qbgpu_dscal(int64_t n, double a, double *x);

/* -------------------------------------------------------------------------------- fused Krylov loops
 * Same arguments and meaning as the reference templates; `v` etc. are HOST or DEVICE per `where`.
 *
 * qbgpu_lanczos_*: lanczos<T,MAT>(k, np, maxit, m, dim, mat, v, hessenberg, purpose), src/lanczos.cc:134-266,
 *   for purposes "sr_val0", "sr_val1" (phi0 at v+2n) and "dnmcs".  hessenberg[2*maxit]: b in
 *   [0,maxit), a in [maxit,2maxit).  On return *m = steps performed; v[(m%2)*n] holds v_m and v[((m+1)%2)*n]
 *   holds v_{m-1} like the reference (normalised).  k > 0 resumes (qbasis.h:1044-1061): on entry v holds the
 *   normalised v[k-1], v[k] in those slots and hessenberg a[0..k-1], b[0..k]; the stop rule's counters restart, as in
 *   the reference's lanczos() without checkpoints.
 * qbgpu_lanczos_resume_*: the same with the four quantities the reference's checkpoint carries across an
 *   interruption (src/ckpt.cc, lczs_mlns.dat): stop_state[4] = {cnt_accuE0, accuracy, theta0_prev, theta1_prev}, read
 *   on entry and updated on return, so that a run cut into pieces stops at the step the uninterrupted run stops at.
 *   quantum_basis_b200/ckpt.py writes and reads the reference's out_Qckpt/ files around it.
 * qbgpu_eigenvec_cg_*: eigenvec_CG<T,MAT>(dim, maxit, m, mat, E0, accu, v, r, p, pp), src/lanczos.cc:281-341;
 *   *m == 0 starts from the guess in v, *m > 0 continues from (v, r, p) of step m (what the reference's CG checkpoint
 *   holds: CG_{V,R,P}<m>.dat, src/ckpt.cc:345-480); loops while *m < maxit.
 * qbgpu_energy_scale_*: energy_scale<T,MAT>(dim, mat, v, lo, hi, extend, iters), src/kpm.cc:45-88 (start vector
 *   vec_randomize(seed=1) drawn inside, as the reference does).
 * qbgpu_kpm_moments_*: NEW (the reference has no Chebyshev code): mu_k = <phi|T_k((H-c)/s)|phi>, k < nmom,
 *   c=(hi+lo)/2, s=(hi-lo)/2, with the 2n/2n+1 doubling identities (nmom/2 products).
 * Only single-GPU handles (row_lo == 0, row_hi == n); the sharded loops are driven from
 * quantum_basis_b200/dist.py through the *_step entry points below. */
int qbgpu_lanczos_d(qbgpu_matrix_t A, int64_t k, int64_t np, int64_t maxit, int64_t *m, double *v,
                    double *hessenberg, const char *purpose, int where);
int qbgpu_lanczos_z(qbgpu_matrix_t A, int64_t k, int64_t np, int64_t maxit, int64_t *m, void *v,
                    double *hessenberg, const char *purpose, int where);
int qbgpu_lanczos_resume_d(qbgpu_matrix_t A, int64_t k, int64_t np, int64_t maxit, int64_t *m, double *v,
                           double *hessenberg, const char *purpose, int where, double *stop_state);
int qbgpu_lanczos_resume_z(qbgpu_matrix_t A, int64_t k, int64_t np, int64_t maxit, int64_t *m, void *v,
                           double *hessenberg, const char *purpose, int where, double *stop_state);
int qbgpu_eigenvec_cg_d(qbgpu_matrix_t A, int64_t maxit, int64_t *m, double E0, double *accu,
                        double *v, double *r, double *p, double *pp, int where);
int qbgpu_eigenvec_cg_z(qbgpu_matrix_t A, int64_t maxit, int64_t *m, const double E0[2], double *accu,
                        void *v, void *r, void *p, void *pp, int where);
int qbgpu_energy_scale_z(qbgpu_matrix_t A, void *v, double *lo, double *hi, double extend, int64_t iters, int where);
int qbgpu_energy_scale_d(qbgpu_matrix_t A, double *v, double *lo, double *hi, double extend, int64_t iters, int where);
int qbgpu_kpm_moments_z(qbgpu_matrix_t A, const void *phi, double lo, double hi, int64_t nmom, double *mu, int where);
int qbgpu_kpm_moments_d(qbgpu_matrix_t A, const double *phi, double lo, double hi, int64_t nmom, double *mu, int where);
/* Device-resident thick-restart Lanczos for the `nev` eigenpairs of smallest algebraic value with a basis of `ncv`
 * vectors kept in HBM: the contract of iram<T,MAT>() / model<T>::locate_E0_iram (src/lanczos.cc:497-603,
 * src/model.cc:1320-1366; maxit <= 0 -> nev*100 restarts, tol <= 0 -> machine precision) without the PCIe round trip
 * ARPACK's reverse communication costs per product.  eigenvals[nev] ascending; eigenvecs (may be NULL) nev vectors of
 * length n, HOST or DEVICE per `where`, element type of the handle.  *nconv = converged pairs, *nprod = products used. */
int qbgpu_trlan(qbgpu_matrix_t A, int nev, int ncv, int maxit, double tol, int *nconv, int *nprod, double *eigenvals,
                void *eigenvecs, int where);
/* The same for the algebraically LARGEST eigenvalues (the iram(..., "lr") call of model<T>::locate_Emax_iram,
 * src/model.cc:1370-1422): the iteration runs on -H; eigenvals come back in descending order. */
int qbgpu_trlan_largest(qbgpu_matrix_t A, int nev, int ncv, int maxit, double tol, int *nconv, int *nprod, double *eigenvals,
                        void *eigenvecs, int where);
/* host-side dense Hermitian eigensolver used for the projected matrix (cyclic complex Jacobi): a and s are m x m complex,
 * column-major; w ascending, columns of s are the eigenvectors */
int qbgpu_herm_eigen(int m, const void *a_colmajor, double *w, void *s_colmajor);
/* hess_eigen (src/lanczos.cc:355-390, order "sr"): host-side tridiagonal Ritz solve used by the stop rule.
 * ritz[m]; s[m*m] column-major eigenvectors or NULL. */
int qbgpu_hess_eigen(const double *hessenberg, int64_t maxit, int64_t m, double *ritz, double *s);
/* lowest Ritz value only, by Sturm bisection in O(m): what the per-step part of the stop rule needs (src/lanczos.cc:232) */
int qbgpu_hess_smallest(const double *hessenberg, int64_t maxit, int64_t m, double *theta0);

/* ------------------------------------------------------------------ step-level entry points (DEVICE only)
 * One fused pass each; scalars live in a device array `sc` so that no host synchronisation is needed between
 * them and a collective can be inserted on a slot (multi-GPU: allreduce sc[slot]).  Vector element type follows
 * the handle (complex for z handles, double for d handles).
 *
 *   spmv_fused:  y_i = alpha*(H x)_i + gamma*x_{row_lo+i} + beta*z_i        (z may alias y; z may be NULL if beta==0)
 *                dots[0,1] = sum conj(x_{row_lo+i}) y_i,  dots[2] = sum |y_i|^2 over the local rows (dots may be NULL)
 */
int qbgpu_spmv_fused(qbgpu_matrix_t A, const void *x, const void *z, void *y,
                     const double alpha[2], const double gamma[2], const double beta[2], double *dots_dev);
/* Lanczos step pieces on the local rows (row_lo..row_hi) of a (possibly sharded) handle.
 *   state (8 device doubles): [0]=sx [1]=sz [2]=b_prev [3]=alpha_partial [4],[5]=scratch [6]=norm2_partial [7]=spare
 *   lanczos_step_a : w = sx*H*(ux) - b_prev*sz*uz  -> uz ;  state[3] = sum Re conj(sx*ux_i) w_i   (local rows)
 *   lanczos_step_b : w' = uz - state[3]*sx*ux_local -> uz ; state[6] = sum |w'_i|^2
 *   lanczos_step_c : b = sqrt(state[6]); a_dev[m-1] = state[3]; b_dev[m] = b; rotate (sx,sz,b_prev) <- (1/b,sx,b)
 * ux is the FULL gathered vector (n entries); uz and the local slice of ux have row_hi-row_lo entries. */
int qbgpu_lanczos_step_a(qbgpu_matrix_t A, const void *ux_full, void *uz_local, double *state_dev);
/* the same pass on one column block of a split shard: first != 0 applies the -b*sz*uz term, later blocks accumulate
 * into uz; last != 0 also reduces state[3] (uz then holds the complete w for the local rows) */
int qbgpu_lanczos_step_a_part(qbgpu_matrix_t A_part, const void *ux_full, void *uz_local, double *state_dev, int first, int last);
int qbgpu_lanczos_step_b(qbgpu_matrix_t A, const void *ux_local, void *uz_local, double *state_dev);
int qbgpu_lanczos_step_c(double *state_dev, double *a_dev, double *b_dev, int64_t m);
/* eigenvec_CG, one call per pass of the reference's loop body (src/lanczos.cc:293-332), for a host that keeps the loop and
 * replaces its body; unsharded handles, DEVICE vectors in the handle's element type and order, E0 = {re, im} (im ignored by
 * d handles).  sc (8 device doubles, zeroed by the caller before the first call): [0]=gamma=|r| [1,2]=delta=<p,pp>
 * [3]=|pp|^2 [4]=|r_new|^2 [5]=gamma_next [6]=scratch -- carried from call to call.
 *   cg_restart (:297-314): v /= |v| ; r = (E0 - H) v ; p = r ; *accu = |r| ; *vnorm (may be NULL) = |v| on entry.  The caller
 *                          decides when (m == 0, or accu < 2e-12 with | |v| - 1 | > 2e-12: qbgpu_dznrm2 / qbgpu_dnrm2).
 *   cg_step    (:320-330): pp = (H - E0 + eps) p ; alpha = gamma^2 / delta ; v += alpha p ; r -= alpha pp ;
 *                          beta = |r_new| / gamma ; p = r + beta^2 p ; gamma *= beta ; *accu = gamma
 * qbgpu_eigenvec_cg_* is exactly this sequence (same kernels, same order: bit-identical results). */
int qbgpu_cg_restart(qbgpu_matrix_t A, const double E0[2], double *sc_dev, void *v, void *r, void *p, double *vnorm, double *accu);
int qbgpu_cg_step(qbgpu_matrix_t A, const double E0[2], double *sc_dev, void *v, void *r, void *p, void *pp, double *accu);
/* One step of the Chebyshev recurrence (KPM) as ONE fused product: Ht = (H - c)/s, c = (hi+lo)/2, s = (hi-lo)/2 (the bounds of
 * qbgpu_energy_scale_*).  first != 0: t_next = Ht t_cur ; otherwise t_next = 2 Ht t_cur - t_prev (t_next may alias t_prev: the
 * recurrence written over T_{k-1}).  dots (3 device doubles, may be NULL): <t_cur_local, t_next> (re, im) and |t_next|^2 over the
 * local rows -- the inner products of mu_{2k+1} = 2<T_k,T_{k+1}> - mu_1 and mu_{2k+2} = 2|T_{k+1}|^2 - mu_0.  t_cur: the full
 * vector (n entries); t_prev / t_next: the handle's local rows (shards: all-reduce the dots).  qbgpu_kpm_moments_* is a loop of
 * these. */
int qbgpu_cheb_step(qbgpu_matrix_t A, double lo, double hi, int first, const void *t_cur_full, const void *t_prev_local,
                    void *t_next_local, double *dots_dev);

/* ------------------------------------------------------------- peer-memory exchange over NVLink (multi-GPU)
 * One process per GPU.  A rank exports its vector buffers (CUDA IPC), maps its peers', and pulls the slices it needs
 * with copy-engine transfers, one stream ("lane") per peer, overlapped with the products of the column blocks that
 * have already arrived (quantum_basis_b200/dist.py: PeerExchangeOperator).
 *   ipc_export: 64-byte handle of a qbgpu_malloc'ed buffer;  ipc_open: map a peer's handle -> device pointer
 *   peer_pull_async(lane, slot, dst, src, bytes): enqueue on copy stream `lane` a transfer ordered after the compute
 *       stream's current tail; its completion is event `slot` (0..15)
 *   peer_wait(slot): order the compute stream behind that transfer */
int qbgpu_ipc_export(void *dptr, void *handle64);
int qbgpu_ipc_open(const void *handle64, void **peer_ptr);
int qbgpu_ipc_close(void *peer_ptr);
int qbgpu_peer_pull_async(int lane, int slot, void *dst_local, const void *src_peer, size_t bytes);
/* same, moved by `ctas` thread blocks reading the peer mapping directly (16-byte aligned) instead of a copy engine */
int qbgpu_peer_pull_sm(int lane, int slot, void *dst_local, const void *src_peer, size_t bytes, int ctas);
int qbgpu_peer_wait(int slot);
/* Ring-fused sharded product (EXPERIMENTAL: correct, but measured slower than the column-block scheme -- a row needs every
 * slice, so the kernel serialises behind the last arrival; DESIGN section 6): ONE kernel that multiplies the whole row
 * shard while the peers' vector slices are still arriving.  qbgpu_ring_prepare(A, rank, world, chunk, &view) re-orders every row of the shard A (rows [rank*chunk, ...),
 * chunk a multiple of 4) so that its own rank's columns come first and the others in ring order, and returns a view
 * handle sharing A's arrays (destroy it before A): every product with the VIEW (qbgpu_{d,z}mv, qbgpu_lanczos_step_a)
 * waits, entry by entry, for the arrival flag of the slice it is about to gather from; A itself keeps working with the
 * ordinary kernels.  Per product: qbgpu_peer_ring_reset(), then one qbgpu_peer_pull_flag(lane, slot, dst, src, bytes, d) per
 * peer (d = (owner - rank + world) % world; every d in 1..world-1 must be issued, with bytes = 0 for an empty slice),
 * then the product.  A waiter gives up after ~1 s instead of hanging the device: check qbgpu_peer_ring_status. */
int qbgpu_ring_prepare(qbgpu_matrix_t A, int rank, int world, int64_t chunk, qbgpu_matrix_t *ring_view);
int qbgpu_peer_ring_reset(void);
int qbgpu_peer_pull_flag(int lane, int slot, void *dst_local, const void *src_peer, size_t bytes, int ring_distance);
int qbgpu_peer_ring_status(int *timed_out);

/* --------------------------------------------------------------------- on-device Hamiltonian generators
 * The reference assembles H on the host (model::generate_Ham_sparse_full, src/model.cc:619-716) in Lin-table
 * order (src/basis.cc:1144-1190).  For the BASELINE sizes the reference's own assembler cannot run (SURVEY F6),
 * so these generators build the SAME expanded matrix (same basis order, same values) directly in HBM; they are
 * checked entry-for-entry against matrices assembled by the compiled reference at sizes it can handle.
 *   heisenberg: spin-1/2, H = sum_bonds J (S_i.S_j), fixed number of DOWN spins `ndown` (the reference's digit 1;
 *               Sz_total = nsites/2 - ndown), bonds[2*nbonds] site pairs.
 *   hubbard:    single "electron" orbital, H = -t sum_{<ij>,s} (c+_is c_js + h.c.) + U sum n_up n_dn.
 * row_lo/row_hi select a row shard (0,-1 = all rows). */
int qbgpu_build_heisenberg(qbgpu_matrix_t *A, int nsites, int ndown, int nbonds, const int32_t *bonds, double J,
                           int api_complex, int flags, int64_t row_lo, int64_t row_hi);
int qbgpu_build_hubbard(qbgpu_matrix_t *A, int nsites, int nup, int ndn, int nbonds, const int32_t *bonds,
                        double t, double U, int api_complex, int flags, int64_t row_lo, int64_t row_hi);
/* model::moprXvec_full (src/model.cc:1468-1538) for an operator made of one-site DIAGONAL terms, on a complex device vector
 * in the reference's Lin order of the full basis the generators above use:
 *   kind 0 (heisenberg, n0 = ndown):      A = sum_r coef0[r] S^z_r                          (coef1 ignored)
 *   kind 1 (hubbard, n0 = nup, n1 = ndn): A = sum_r coef0[r] n_up,r + coef1[r] n_dn,r      (S^z_q: coef1 = -coef0)
 * y_j = x_j * <state_j|A|state_j>, rows with |x_j| < 2e-12 skipped like the reference (:1500).  Followed by the norm, the
 * scaling and qbgpu_lanczos_z(..., "dnmcs") this is model::measure_full_dynamic (src/model.cc:1697-1712), the dynamic part of
 * the reference's examples/trans_absent/latt_square/square_Fermi_Hubbard.cc.  The _host variant runs the same row function
 * on host arrays (test hook; no device is touched). */
int qbgpu_full_apply_diag(int kind, int nsites, int n0, int n1, const double *coef0_reim, const double *coef1_reim,
                          const void *x_dev, void *y_dev);
int qbgpu_debug_full_apply_diag_host(int kind, int nsites, int n0, int n1, const double *coef0_reim, const double *coef1_reim,
                                     const void *x_host, void *y_host);
/* Matrix-free handles: the counterpart of the reference's model<T>::MultMv / MultMv2 with matrix_free == true
 * (src/model.cc:942-1121: every row is recomputed on the fly from the Hamiltonian terms and the Lin tables instead of
 * being read from a stored matrix).  Same arguments as the generators; nothing but the basis states (8 bytes per row)
 * and the Lin tables is kept in HBM, so sectors whose stored matrix would not fit (e.g. the Heisenberg chain L = 32,
 * Sz = 0: 601,080,390 states, 238 GB of CSR) still run on one GPU.  The handle works with every entry point above
 * (products, fused Lanczos / CG / KPM loops) and gives the same results as the stored matrix up to summation order.
 * flags: QBGPU_MATFREE_TERMS adds the one-byte-per-entry term codes (replay instead of search; bit-identical results). */
int qbgpu_create_matfree_heisenberg(qbgpu_matrix_t *A, int nsites, int ndown, int nbonds, const int32_t *bonds, double J,
                                    int api_complex, int flags, int64_t row_lo, int64_t row_hi);
int qbgpu_create_matfree_hubbard(qbgpu_matrix_t *A, int nsites, int nup, int ndn, int nbonds, const int32_t *bonds,
                                 double t, double U, int api_complex, int flags, int64_t row_lo, int64_t row_hi);
/* The two parts of a STORED species-order handle or row shard as handles of their own (views sharing the arrays): `local` =
 * diagonal + hops of the down electrons (its gathers never leave the handle's own rows: on a shard it needs no remote data),
 * `cross` = hops of the up electrons.  The multi-GPU product: start the exchange of x, multiply the local part (y = ...),
 * wait for the slices, multiply the cross part (y += ...).  Destroy the views before the handle. */
int qbgpu_species_parts(qbgpu_matrix_t A, qbgpu_matrix_t *local_part, qbgpu_matrix_t *cross_part);

/* --------------------------------------------------------------------- species order (Hubbard, QBGPU_SPECIES_ORDER)
 * In the reference's Lin-table order every hopping term of the Hubbard matrix sends a row far away in the index space,
 * and the gathers of x cost ~19 vector sizes of DRAM traffic per product instead of 1.  With QBGPU_SPECIES_ORDER the
 * handle keeps its vectors INTERNALLY in the order  p = rank(up configuration) * D_dn + rank(down configuration)  and
 * multiplies in two passes: (diagonal + hops of the down electrons), whose gathers stay inside one contiguous block of
 * D_dn entries, then (hops of the up electrons) traversed by tiles of down indices whose gathered columns stay in L2.
 *   qbgpu_build_hubbard          + flag: the two parts are stored (sliced-jagged layout, same entries as the ordinary
 *                                  handle) and multiplied by the production kernels.  A handle built without a row
 *                                  range (row_hi < 0) with real values stores each entry as one 32-bit word,
 *                                  column | code << (bit width of n - 1), with code an index into the part's table of
 *                                  distinct values (info.value_dict: the local part's table): 4 bytes per entry instead
 *                                  of 12, bit-identical products.  Row shards (also one row range covering all rows),
 *                                  complex values (QBGPU_KEEP_COMPLEX) and tables that do not fit keep fp64 or complex
 *                                  values;
 *   qbgpu_create_matfree_hubbard + flag: nothing is stored but per-species hop tables (a few MB).
 * The calling convention does not change: qbgpu_{d,z}mv, qbgpu_lanczos_*, qbgpu_eigenvec_cg_*, qbgpu_energy_scale_*,
 * qbgpu_kpm_moments_* and qbgpu_trlan take and return vectors in the REFERENCE's order (they permute on the way in and
 * out; inside a Krylov loop nothing is permuted).  The fused low-level entry points (qbgpu_spmv_fused,
 * qbgpu_lanczos_step_*) work in the internal order; the three functions below convert.  Not available: to_dense,
 * download_expanded, ring_prepare.  Row shards and qbgpu_split_columns exist for the matrix-free kind only, in units of whole
 * up configurations (row_lo, row_hi and the column bounds multiples of D_dn); shards and parts have no permutation: their
 * vectors are in the internal order.  QBGPU_SPECIES_TILE (environment, default 128) sets the tile width in down indices. */
int qbgpu_native_order(qbgpu_matrix_t A, int *has_internal_order);
int qbgpu_vec_to_native(qbgpu_matrix_t A, const void *x_reference_order_dev, void *x_internal_order_dev);   /* out of place */
int qbgpu_vec_from_native(qbgpu_matrix_t A, const void *x_internal_order_dev, void *x_reference_order_dev); /* out of place */
int qbgpu_native_perm(qbgpu_matrix_t A, int32_t *perm_host);   /* perm[r] = internal index of the reference's row r */
/* Test hook, HOST ONLY (no device is touched): runs the species-order index logic -- the same __host__ __device__ row
 * functions the kernels call -- on host arrays, so that the CPU test-suite can check it against the reference-pinned
 * restatement.  sizes[4] = {D_up, D_dn, up-hop entries, down-hop entries}; every other pointer may be NULL (skipped):
 * perm[n]; the two stored parts as CSR (rowptr[n+1]; nnz_local = D_up*(dn_entries + D_dn), nnz_cross = D_dn*up_entries);
 * slice_order[ceil(n/32)]; y[n] = H x by the two matrix-free passes (x, y real, internal order), touched[p] += 1 for every
 * write of the cross pass (all ones afterwards). */
int qbgpu_debug_species_host(int nsites, int nup, int ndn, int nbonds, const int32_t *bonds, double t, double U, int tile,
                             int64_t *sizes, int32_t *perm, int64_t *rowptr_local, int32_t *col_local, double *val_local,
                             int64_t *rowptr_cross, int32_t *col_cross, double *val_cross, int32_t *slice_order,
                             const double *x, double *y, int32_t *touched);

/* The same for a row shard (up configurations [u_lo, u_hi)) cut into column parts executed in `order` (the multi-GPU
 * exchange pattern): part p keeps the up-hops whose target configuration lies in [part_bounds[p], part_bounds[p+1]). */
int qbgpu_debug_species_parts_host(int nsites, int nup, int ndn, int nbonds, const int32_t *bonds, double t, double U, int tile,
                                   int64_t u_lo, int64_t u_hi, int nparts, const int64_t *part_bounds, const int32_t *order,
                                   const double *x, double *y_local);

/* The packed entry words of the two stored parts, computed on the host with the build's rules (species order, a handle
 * built without a row range, real values).  cbits <= 0: the build's column width (bit width of n - 1).  out[5] = {cbits, local table entries,
 * cross table entries, local part packed (0/1), cross part packed (0/1)}; a part is packed when its table fits in the
 * 32 - cbits bits above the column (and has at most 256 entries).  table_* (256 doubles each, in code order) and
 * words_* (the parts' entries in CSR order, as qbgpu_debug_species_host lists them; written only for a packed part) may
 * be NULL. */
int qbgpu_debug_species_packed_host(int nsites, int nup, int ndn, int nbonds, const int32_t *bonds, double t, double U, int cbits,
                                    int64_t *out, double *table_local, uint32_t *words_local, double *table_cross, uint32_t *words_cross);

/* --------------------------------------------------------------------- translation-symmetric sectors
 * Device counterpart of model::fill_Weisse_table + enumerate_basis_repr + generate_Ham_sparse_repr
 * (src/model.cc:205-249, 275-487, 688-836) for spin-1/2 models on untilted lattices with one site per unit cell and
 * periodic boundaries in every direction (chain, square, triangular; at most 36 sites, at least one even direction):
 * the representatives, their order (Lin order when the reference's Lin tables exist, bisection order otherwise),
 * the norms and every matrix element are those of the reference bit for bit (tests/repr_builders.py restates the
 * convention and is pinned against 39 sectors assembled by the compiled reference).  BASELINE configs 2 and 5.
 *   L[dim]: lattice extents; k[dim]: momentum integers as passed to enumerate_basis_repr; ndown: number of down spins
 *   (digit 1), Sz_total = nsites/2 - ndown.  Sites are numbered like the reference's lattice class: first even
 *   direction fastest (src/lattice.cc:591-615).
 * Up to 32 sites a state is a 32-bit word; 34- and 36-site sectors keep 64-bit states and keys (qbgpu_sector_states64).
 * Device memory of a sector with n representatives: 8 n (norms) + 4 n (keys; 8 n at 34 and 36 sites) + the segment table
 * (256 KB up to 32 sites, at most 4 bytes per representative beyond) + the sublattice tables (2 MB at 32 sites, 19 MB at 36).
 * The (Sz = 0, k) sectors of 36 sites hold about 2.5e8 representatives: 2 GB of keys, 2 GB of norms and 4 GB per complex
 * vector, so they run through qbgpu_sector_matfree_heisenberg. */
typedef struct qbgpu_sector *qbgpu_sector_t;
typedef struct {
    int64_t dim;                 /* number of representatives, including those of zero norm */
    int64_t zero_norm;           /* representatives whose norm vanishes at this momentum (rows fake_pos + i/dim) */
    int     nsites;
    int     lin_order;           /* 1: Lin-table order (odd-site label, even-site label); 0: integer order */
    double  enumerate_seconds, norms_seconds;
    double  lin_check_seconds;   /* host part of enumerate_seconds: the Lin-table existence check over the keys */
    int     state_bits;          /* 32, or 64 for sectors whose states need qbgpu_sector_states64 */
} qbgpu_sector_info;
int qbgpu_sector_create(qbgpu_sector_t *S, int dim, const int32_t *L, int ndown, const int32_t *k);
int qbgpu_sector_destroy(qbgpu_sector_t S);
int qbgpu_sector_get_info(qbgpu_sector_t S, qbgpu_sector_info *info);
int qbgpu_sector_states(qbgpu_sector_t S, uint32_t *states_host);      /* bit s set = site s down, row order; QBGPU_ERR_STATE when state_bits = 64 */
int qbgpu_sector_states64(qbgpu_sector_t S, uint64_t *states_host);    /* the same as 64-bit words, for every sector */
int qbgpu_sector_norms(qbgpu_sector_t S, double *nu_host);
/* H = J sum_bonds S_i.S_j in that sector (bonds[2*nbonds] site pairs, duplicates are separate terms like repeated
 * add_Ham calls); fake_pos is model's constructor argument (default 100, src/qbasis.h:1337). */
int qbgpu_sector_build_heisenberg(qbgpu_sector_t S, qbgpu_matrix_t *A, int nbonds, const int32_t *bonds, double J,
                                  double fake_pos, int flags);
/* The same Hamiltonian WITHOUT stored entries: the handle regenerates every row inside the product -- model<T>::MultMv2 with
 * matrix_free == true, repr branch (src/model.cc:1016-1107): y[i] += x[j] * sqrt(nu_i/nu_j) * conj(c) * exp(2 pi i k.disp_i/L) for
 * every term, fake_pos + i/dim on zero-norm rows.  Works with every entry point that takes a handle (products, Lanczos, CG, KPM).
 * The handle borrows the sector's device tables: destroy it before the sector. */
int qbgpu_sector_matfree_heisenberg(qbgpu_sector_t S, qbgpu_matrix_t *A, int nbonds, const int32_t *bonds, double J,
                                    double fake_pos);
/* A (N_up, N_dn, momentum) sector of single-orbital electrons on an untilted lattice of at most 16 sites -- fill_Weisse_table +
 * enumerate_basis_repr (src/model.cc:205-249, 275-487) for the reference's "electron" orbital (src/basis.cc:49-96: two bits per
 * site, bit 0 up, bit 1 down; qbgpu_sector_states returns these patterns).  Same representatives, row order and norms as the
 * reference, the fermionic translation signs included (src/basis.cc:593-620, 2134-2147). */
int qbgpu_sector_create_electron(qbgpu_sector_t *S, int dim, const int32_t *L, int nup, int ndn, const int32_t *k);
/* generate_Ham_sparse_repr (src/model.cc:688-836) for H = -t sum_hops c+_{to,s} c_{from,s} + U sum_i n_up,i n_dn,i on such a sector.
 * hops[3*nhops] = (to, from, spin) DIRECTED, in the order of the caller's add_Ham calls (they are re-ordered like
 * mopr::operator+= does, src/operators.cc:901-925).  Bit-identical to the reference's csr_mat on 4x2 and 4x3 clusters. */
int qbgpu_sector_build_hubbard(qbgpu_sector_t S, qbgpu_matrix_t *A, int nhops, const int32_t *hops, double t, double U,
                               double fake_pos, int flags);
/* model::moprXvec_repr (src/model.cc:1716-1846) for A = sum_r c_r S^z_r (coef_reim[2*nsites], site order): device
 * vectors x_old (sector S_old) -> y_new (sector S_new, same lattice and Sz, momentum shifted by the operator's q).
 * With measure_repr_dynamic's normalisation and qbgpu_lanczos_z(..., "dnmcs") this is src/model.cc:1897-1912. */
int qbgpu_sector_apply_sz(qbgpu_sector_t S_old, qbgpu_sector_t S_new, const double *coef_reim, const void *x_old_dev,
                          void *y_new_dev);
/* The off-diagonal branch of the same routine (src/model.cc:1762-1834) for the spin-1/2 ladder operators:
 * A = sum_r coef[r] S^-_r (lower = 1; S_new has one more down spin) or sum_r coef[r] S^+_r (lower = 0; one fewer).
 * y_new (S_new's dimension) is overwritten.  Contributions are added with fp64 atomics -- the reference adds them from
 * several threads in no fixed order either -- so results agree with it to rounding, not to the bit. */
int qbgpu_sector_apply_ladder(qbgpu_sector_t S_old, qbgpu_sector_t S_new, int lower, const double *coef_reim,
                              const void *x_old_dev, void *y_new_dev);
/* The same routine for one-site ELECTRON operators A = sum_r c_r O_r between electron sectors of one lattice (coefficients
 * *_reim[2*nsites] in site order; device vectors x_old_dev (S_old) -> y_new_dev (S_new), which is overwritten).  The target
 * momentum is the caller's choice, as for the spin entries:
 *   - coefficients e^{+i q.r} move a vector from momentum K to K + q (S^z_q, n_q, S^-_q of the reference's examples);
 *   - c_k = N^{-1/2} sum_r e^{-i k.r} c_r moves it from K to K - k, c+_k = N^{-1/2} sum_r e^{+i k.r} c+_r from K to K + k.
 * Source rows with |x| < 2e-12 and rows of zero norm in either sector contribute nothing (src/model.cc:1752,1760,1810).
 * Single-electron operators carry oprXphi's sign (src/basis.cc:2717-2731) and the translation sign of the representative
 * in the sector they land in.  Every output row is computed once, in a fixed term order (the adjoint of A applied to the
 * target representative), so repeated calls are bit-identical; for coefficients e^{+i q.r} between K and K + q this is the
 * reference's scatter to rounding.  QBGPU_ERR_STATE on a spin sector, QBGPU_ERR_ARG on another lattice or particle numbers
 * that do not match the operator. */
/* A = sum_r cu[r] n_up,r + cd[r] n_dn,r.  S_old, S_new: same lattice, same N_up and N_dn.
 * S^z_q: cd = -cu.  Charge n_q: cd = cu. */
int qbgpu_sector_apply_density(qbgpu_sector_t S_old, qbgpu_sector_t S_new, const double *cu_reim,
                               const double *cd_reim, const void *x_old_dev, void *y_new_dev);
/* lower = 1: A = sum_r c[r] c+_{r,dn} c_{r,up}  (S^-; S_new has N_up-1, N_dn+1)
 * lower = 0: the S^+ counterpart                 (S_new has N_up+1, N_dn-1) */
int qbgpu_sector_apply_spin_flip(qbgpu_sector_t S_old, qbgpu_sector_t S_new, int lower,
                                 const double *c_reim, const void *x_old_dev, void *y_new_dev);
/* create = 0: A = sum_r c[r] c_{r,spin}   (S_new has one electron fewer of that spin; spin 0 up, 1 down)
 * create = 1: A = sum_r c[r] c+_{r,spin}  (S_new has one more) */
int qbgpu_sector_apply_fermion(qbgpu_sector_t S_old, qbgpu_sector_t S_new, int create, int spin,
                               const double *c_reim, const void *x_old_dev, void *y_new_dev);
/* Momentum sector for an ARBITRARY abelian symmetry group given as site permutations (BASELINE config 4: the tilted
 * 31-site triangular cluster, which the reference itself cannot build -- SURVEY F5 -- so there is no reference convention
 * to reproduce; representative = smallest bit pattern of the orbit, orbits on whose stabiliser the character is not
 * trivial are dropped, rows ascending by representative).  perms[t*nsites + s] = image of site s under group element t
 * (element 0 = identity), chi_reim[2t], chi_reim[2t+1] = character of element t in the wanted one-dimensional irrep.
 * states_out (host, may be NULL) receives the representatives if states_capacity >= dimension. */
int qbgpu_build_heisenberg_orbit(qbgpu_matrix_t *A, int nsites, int ndown, int ntrans, const int32_t *perms,
                                 const double *chi_reim, int nbonds, const int32_t *bonds, double J, int flags,
                                 uint32_t *states_out, int64_t states_capacity);
/* dimension of those sectors (host only) */
int64_t qbgpu_dim_heisenberg(int nsites, int nup);
int64_t qbgpu_dim_hubbard(int nsites, int nup, int ndn);

/* ---------------------------------------------------------------------------- multi-GPU drivers (csrc/dist.cu)
 * One process per GPU; everything a rank needs from its peers travels through peer memory (CUDA IPC over NVLink): copy-engine
 * pulls of the vector slices and a push-based, deterministic all-reduce kernel for the scalars -- no MPI / NCCL inside, so a
 * C or C++ host (the reference is one: model<T>::locate_E0_lanczos, src/model.cc:1124-1316) can drive the GPUs of a box with
 * this library alone.  The host hands the 64-byte handles around by any means it has (INTEGRATION.md).
 *   create   every rank: rows [bounds[r], bounds[r+1]) belong to rank r; vectors are complex128 or fp64
 *   export   64 bytes to give to every other rank;  connect: all ranks' handles, rank-major (world * 64 bytes)
 * A shard is (local_part, rest): for a species-order shard the two views of qbgpu_species_parts (the local part needs no
 * remote data and runs while the slices travel); for any other row shard local_part = NULL and rest = the shard.
 * All entry points are collective: every rank calls them in the same order. */
typedef struct qbgpu_dist *qbgpu_dist_t;
int qbgpu_dist_create(qbgpu_dist_t *D, int rank, int world, int64_t n, const int64_t *bounds, int vec_complex);
int qbgpu_dist_export(qbgpu_dist_t D, void *handle64);
int qbgpu_dist_connect(qbgpu_dist_t D, const void *handles_world_x_64);
int qbgpu_dist_destroy(qbgpu_dist_t D);
/* refinement of a shard: parts that need no remote data (they run while the slices travel) / parts that follow the arrival;
 * and the row ranges of the peers' slices that are fetched at all (default: every slice, whole) */
int qbgpu_dist_set_parts(qbgpu_dist_t D, int n_early, const qbgpu_matrix_t *early, int n_late, const qbgpu_matrix_t *late);
int qbgpu_dist_set_pull_plan(qbgpu_dist_t D, int nseg, const int32_t *owner, const int64_t *first_row, const int64_t *nrows, int lanes);
/* the cross part of a stored species-order handle or shard cut by column ranges (owning handles, same rows and traversal) */
int qbgpu_species_split_cross(qbgpu_matrix_t A, int nparts, const int64_t *col_bounds, qbgpu_matrix_t *parts);
/* a view of a sliced-jagged handle (a part of a species shard) restricted to its local rows [r0, r1): whole 32-row slices, and
 * for a tile-ordered cross part multiples of tile_period = D_dn; products through it address y / z at the view's rows */
int qbgpu_row_view(qbgpu_matrix_t A, int64_t r0, int64_t r1, int64_t tile_period, int tile, qbgpu_matrix_t *view);
/* late part j may start as soon as the first wait_after[j] segments of the pull plan have arrived (default: all of them) */
int qbgpu_dist_set_wait_points(qbgpu_dist_t D, int n_late, const int32_t *wait_after);
int qbgpu_dist_own(qbgpu_dist_t D, int b, void **own_slice_dev, int64_t *nloc);   /* this rank's rows of vector buffer b (0 | 1) */
int qbgpu_dist_full(qbgpu_dist_t D, int b, void **full_vector_dev);
int qbgpu_dist_barrier(qbgpu_dist_t D);                                            /* stream-ordered, device-side */
int qbgpu_dist_allreduce(qbgpu_dist_t D, double *dev, int count);                  /* in-place sum of <= 8 device doubles, rank order */
/* own slice of X[b] <- this rank's rows of vec_randomize(n, seed) (src/miscellaneous.cc:371-388), normalised over all ranks;
 * opens and closes with a barrier (no peer is still reading the slice; every slice is final before anybody pulls) */
int qbgpu_dist_randomize(qbgpu_dist_t D, int b, uint32_t seed, const int32_t *ref_row_dev);
int qbgpu_species_ref_rows(int nsites, int nup, int ndn, int64_t row_lo, int64_t row_hi, int32_t *ref_rows_dev);
/* y_local = (H x)_local with x = X[b].  Who may touch a slice when: a rank's own product is finished once ITS pulls are, while
 * its peers may still be reading its slice of X[b].  barrier bit 0 (1): barrier BEFORE the pulls (the slices the caller just
 * wrote are final everywhere); bit 1 (2): barrier AFTER the product (every rank's pulls are done: the own slice of X[b] may be
 * rewritten).  Without bit 1 write the next x into the other buffer (the loops below ping-pong) or call qbgpu_dist_barrier. */
int qbgpu_dist_mv(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, int b, void *y_local_dev, int barrier);
/* lanczos(0, np, maxit, ...) of src/lanczos.cc:134-266 on the shards: "sr_val0" with the stop rule of :228-248, or "dnmcs"
 * ("sr_val1" needs phi0: qbgpu_dist_lanczos_val1) */
int qbgpu_dist_lanczos(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, int64_t np, int64_t maxit, int64_t *m,
                       double *hess, const char *purpose, int stop_on_breakdown);
/* lanczos(0, np, maxit, ..., "sr_val1") of src/lanczos.cc:134-266 on the shards: the loop of qbgpu_dist_lanczos (stop rule of
 * sr_val0) with the re-orthogonalisation against phi0 of :218-226 in every step after the first.  Start: the normalised start
 * vector, orthogonal to phi0, in the own slice of X[0] and visible to the peers.  phi0_local: this rank's rows of phi0 (device,
 * element type of D, in the shard's order), not NULL.  The projection is decided on the device from the all-reduced
 * <phi0, v_m> (|<phi0, v_m>| > 2e-12, as the reference) and is in the stream before the next step's transfers: no host round
 * trip.  On return the normalised v_m is the own slice of X[m % 2], v_{m-1} of X[(m-1) % 2], as for qbgpu_dist_lanczos.  On a
 * breakdown (|b_m| < 2e-12 with stop_on_breakdown) the reference stops before it projects; here v_m handed back is the one
 * after the projection of step m (when the projection ran), normalised.  hess is the same either way. */
int qbgpu_dist_lanczos_val1(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, const void *phi0_local, int64_t np, int64_t maxit,
                            int64_t *m, double *hess, int stop_on_breakdown);
/* model<T>::locate_E0_lanczos(nev, ncv, maxit) of src/model.cc:1124-1316 on the shards; collective.  0 < nev <= 2,
 * nev-1 <= ncv <= nev (else QBGPU_ERR_ARG).  eigenvals[nev] on every rank (E0, E1); phi_local: ncv vectors of this rank's rows
 * one after the other (device, element type of D, in the shard's order: the internal order for species-order shards; may be
 * NULL if ncv == 0); steps[4] / accuracies[4]: Lanczos E0, CG phi0, Lanczos E1, CG phi1 (0 for stages not run).  ref_row_dev
 * as for qbgpu_dist_randomize (NULL for ordinary shards).  Overwrites X[0] and X[1]. */
int qbgpu_dist_locate_e0_lanczos(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, const int32_t *ref_row_dev,
                                 int nev, int ncv, int64_t maxit, double *eigenvals, void *phi_local, int64_t *steps, double *accuracies);
/* energy_scale of src/kpm.cc:45-88; Chebyshev moments of the own slices of X[0]; eigenvec_CG of src/lanczos.cc:281-341 */
int qbgpu_dist_energy_scale(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, const int32_t *ref_row_dev, double *lo, double *hi,
                            double extend, int64_t iters);
int qbgpu_dist_kpm_moments(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, double lo, double hi, int64_t nmom, double *mu);
int qbgpu_dist_eigenvec_cg(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, int64_t maxit, int64_t *m, const double E0[2],
                           double *accu, void *v_dev, void *r_dev, void *p_dev, void *pp_dev);

/* pass 1 of the matrix-free species-order product: id = 1000 + v, v = 0 grid-stride rows (default), 1 contiguous row ranges
 * with one 1024-thread CTA per SM, 2 block x[iu, :] staged in shared memory.  Any other id: QBGPU_ERR_ARG. */
int qbgpu_debug_set_variant(int id);
/* word width of the spin sectors created afterwards: 0 by size (32-bit states up to 32 sites, the default), 64 the 64-bit
 * path for every spin sector (to compare both widths on one sector).  Any other value: QBGPU_ERR_ARG. */
int qbgpu_debug_sector_words(int bits);
/* Rows of a full-basis Heisenberg (kind 0, n0 = down spins) or Hubbard (kind 1, n0/n1 = N_up/N_dn) operator recomputed on the
 * HOST in long double from the Lin tables (reference src/basis.cc:1144-1190) and the generators' own row function: the
 * size-independent parity check of bench.py on the BASELINE-size matrices.  rows: indices in the reference's order; x_host: the
 * full vector (x_complex: re,im pairs); y_out: 2 doubles per listed row.  No device involved. */
int qbgpu_debug_rows_host(int kind, int nsites, int n0, int n1, int nbonds, const int32_t *bonds, double J, double t, double U,
                          int64_t nrows, const int64_t *rows, const void *x_host, int x_complex, double *y_out);

/* counters for bench.py's `gpu_launches` (kernels launched by this library since the last reset) */
int64_t qbgpu_kernel_launches(int reset);

#ifdef __cplusplus
}
#endif
#endif /* QBGPU_H */
