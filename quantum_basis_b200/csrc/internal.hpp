// quantum_basis_b200/csrc/internal.hpp -- types shared by the translation units of libqbgpu.
#pragma once
#include "common.cuh"
#include "../../include/qbgpu.h"
#include <cmath>

// Device-resident matrix behind qbgpu_matrix_t.
//
// HBM layout ("expanded CSR"): the full Hermitian matrix, i.e. the reference's upper triangle plus its
// materialised conjugate transpose, so that every row is complete and a product needs no atomics:
//   rowptr[n_local+1]  int64   offsets into col/val (local to this handle: rowptr[0] == 0)
//   col[nnz]           int32   global column indices, ascending within a row
//   val[nnz]           fp64 or (re,im) fp64 pairs (fp64 when the input was real or had all imag == 0)
// n_local = row_hi - row_lo rows of the global n x n matrix (a row shard for multi-GPU runs).
struct qbgpu_matrix {
    int64_t n = 0, row_lo = 0, row_hi = 0;
    int64_t nnz = 0, nnz_input = 0;
    bool    val_real = false, api_complex = false;
    bool    borrowed = false;      // a view sharing another handle's arrays (qbgpu_real_view): destroy frees nothing
    int     format = QBGPU_FORMAT_CSR;
    int     lanes = 8;
    int64_t *rowptr = nullptr;
    int32_t *col = nullptr;
    void    *val = nullptr;
    // QBGPU_FORMAT_SELL ("sliced jagged"): same arrays, but inside every slice of 32 consecutive rows the entries
    // are stored jagged-diagonal-wise: rows ranked by length (descending), then for k = 0,1,.. the k-th entry of
    // every row that has one, in rank order.  Slice s still occupies [rowptr[32 s], rowptr[32 s + 32]) -- no padding.
    // rowinfo[32 s + rank] = (row-in-slice << 24) | length.
    uint32_t *rowinfo = nullptr;
    // optional value dictionary (QBGPU_VALUE_DICT, fp64 values with <= 256 distinct bit patterns): val is then an array
    // of 1-byte codes into vdict[ndict]; products decode through shared memory and are bit-identical.
    double  *vdict = nullptr;
    int      ndict = 0;
    // > 0: packed layout (the stored parts of a species handle built without a row range, real values; species.cu): col[]
    // holds one 32-bit word per entry, column | code << cbits, where cbits is the bit width of n - 1 and code indexes
    // vdict[ndict]; there is no val array.  4 bytes per entry instead of 12; products decode the identical doubles and are bit-identical.
    int      cbits = 0;
    // QBGPU_FORMAT_MATFREE: no stored entries at all; `mf` owns the sector tables, the bond list and the per-row
    // basis states from which every row is regenerated inside the product (builders.cu).
    void    *mf = nullptr;
    void    *mf_sec = nullptr;     // matrix-free product over a translation-symmetric sector (sectors.cu); borrows the sector's tables
    // ring-fused row shard (qbgpu_ring_prepare): every row's entries are rotated so that the columns owned by this rank
    // come first, then those of rank+1, ... (ring order); the product then consumes the vector slices in the order the
    // peer pulls deliver them and waits, entry by entry, on the arrival flags of peer.cu.
    int      ring_world = 0, ring_rank = 0;
    int64_t  ring_chunk = 0;
    // QBGPU_SPECIES_ORDER handles (species.cu; single-orbital Hubbard): vectors live INTERNALLY in the order
    // p = rank(up configuration) * D_dn + rank(down configuration).  `perm[r]` = internal index of the reference's row r;
    // the reference-shaped entry points (mv, lanczos, CG, energy_scale, KPM) permute through it, the fused low-level ones
    // (spmv_fused, lanczos_step_*) work in the internal order.  `sp` owns the species tables.  A stored handle holds the
    // "local" part (diagonal + hops of the down electrons: inside the block of one up configuration) and `second` the
    // "cross" part (hops of the up electrons), whose 32-row slices are traversed in `slice_order` (tiles of down indices).
    int32_t *perm = nullptr;
    int32_t *perm_inv = nullptr;     // perm_inv[p] = the reference's row of internal index p (the way in gathers, so both ways write coalesced)
    void    *sp = nullptr;
    qbgpu_matrix *second = nullptr;
    int32_t *slice_order = nullptr;
    // > 0: rows [u*block_D, (u+1)*block_D) reference only columns of the same block (the local part of a species handle):
    // the product may stage the block of x in shared memory (sjds_bulk.cu: sjds_block_smem_kernel)
    int64_t  block_D = 0;
    // > 0: the row metadata repeats -- rowinfo of slice s equals that of slice s % period_slices, and rowptr[32 s] =
    // rowptr[32 (s % P)] + (s / P) * period_entries -- for all FULL slices (the local part of a species handle: its row lengths depend
    // on the down configuration only).  The block-local kernel then reads 0.8 MB of metadata from L2 instead of 0.8 GB from HBM.
    int64_t  period_slices = 0, period_entries = 0;
    bool     owns_order = false;       // a row view (qbgpu_row_view) shares every array but owns its slice_order
    // column part of a matrix-free species shard (qbgpu_split_columns): only the up-hops whose target configuration lies in
    // [sp_col_lo, sp_col_hi) (units: up configurations), plus the whole local pass when sp_has_local; -1 = no filter
    int64_t  sp_col_lo = -1, sp_col_hi = -1;
    bool     sp_has_local = true;
    void    *perm_x = nullptr, *perm_y = nullptr;      // staging vectors of the reference-order product of a species handle, or of
                                                       // the opt-in fp64 product of an ordinary one (lazily allocated; freed by destroy)
    // the device whose context first multiplied with this handle (the creating thread's): a product issued from a thread
    // bound to ANOTHER device (the context is thread-local) is refused instead of running on the wrong device or stream
    mutable int device = -1;
    mutable bool last_x_had_imag = false;      // mv_species: the previous vector had non-zero imaginary parts -> look at the flag BEFORE the fp64 passes
    double  upload_s = 0, convert_s = 0, autotune_s = 0;
    int64_t nrows() const { return row_hi - row_lo; }
    size_t  val_bytes() const { return cbits ? 0 : ndict ? 1 : (val_real ? 8 : 16); }
    size_t  vec_bytes() const { return api_complex ? 16 : 8; }
};

namespace qb {

// Arguments of the fused product  y_i = alpha*(H x)_i + gamma*x_{row_lo+i} + beta*z_i  (+ running dots).
// scal_mode 0: alpha/gamma/beta are the immediates below.
// scal_mode 1 (Lanczos step a): alpha = sc[0], gamma = 0, beta = -sc[2]*sc[1]; dot[0..1] scaled by sc[0].
struct FusedArgs {
    const void *x = nullptr;       // full vector, n entries
    const void *z = nullptr;       // local rows (may alias y), or null
    void       *y = nullptr;       // local rows
    double2     alpha = {1.0, 0.0}, gamma = {0.0, 0.0}, beta = {0.0, 0.0};
    int         scal_mode = 0;
    const double *sc = nullptr;    // device scalars for scal_mode != 0
    double     *dots = nullptr;    // device: out[0]=Re sum conj(x)y, out[1]=Im, out[2]=sum|y|^2 ; null = no dots
    // species handles, real-content route of MultMv (species.cu: mv_species): the way OUT fused into the closing pass (fp64
    // vectors, y += H_cross x): instead of y[row] the bulk-streamed kernel writes y_ref[perm_inv[row]] = out_alpha * (y, 0)
    // -- complex, in the reference's order -- and the separate permutation is skipped
    const int32_t *perm_inv = nullptr;
    void       *y_ref = nullptr;
    double2     out_alpha = {1.0, 0.0};
};

// spmv.cu
int launch_spmv(const qbgpu_matrix *A, const FusedArgs &args, int lanes_override = 0);
int autotune(qbgpu_matrix *A, int flags = 0);
int sjds_convert(qbgpu_matrix *A, bool forward);
int sjds_rows_fit(const qbgpu_matrix *A, bool *fits);   // every row shorter than 2^24 entries (the sliced-jagged length field)
int value_dict_encode(qbgpu_matrix *A, int max_entries = 256);   // matrix.cu: try to replace fp64 values by 1-byte codes
// order of a value table: by value, -0.0 before +0.0 (distinct bit patterns), so that a layout does not depend on thread timing
inline bool value_table_less(double a, double b) { return a != b ? a < b : std::signbit(a) > std::signbit(b); }
// Packed entry words (qbgpu_matrix::cbits): the column takes the bit width of n - 1, the value code the bits above it.  A
// table fits when its codes do (and the 256 entries the product kernels stage in shared memory).
constexpr uint32_t kPackedMaxTable = 256;
__host__ __device__ inline int packed_col_bits(int64_t n)
{ int b = 1; while (b < 31 && ((n - 1) >> b) != 0) b++; return b; }
__host__ __device__ inline bool packed_table_fits(int64_t ntable, int cbits)
{ return ntable > 0 && ntable <= (int64_t)kPackedMaxTable && ntable <= (int64_t)1 << (32 - cbits); }
__host__ __device__ inline uint32_t packed_word(int32_t col, uint32_t code, int cbits) { return (uint32_t)col | code << cbits; }
int launch_spmv_sjds(const qbgpu_matrix *A, const FusedArgs &args);
// sjds_bulk.cu: the same product with the matrix stream moved by cp.async.bulk into per-warp shared-memory rings, and the
// block-local product (rows of block u reference only columns of block u) with the block of x staged in shared memory
int launch_spmv_sjds_bulk(const qbgpu_matrix *A, const FusedArgs &args);        // tile-ordered handles (slice_order set)
bool sjds_bulk_out_fusable(const qbgpu_matrix *cross_part);      // the closing pass of this part can write the reference-order result itself
bool block_smem_applicable(const qbgpu_matrix *A, int64_t D);
int launch_spmv_block_smem(const qbgpu_matrix *A, const FusedArgs &args, int64_t D);
int launch_spmv_matfree(const qbgpu_matrix *A, const FusedArgs &args);     // builders.cu
void matfree_destroy(qbgpu_matrix *A);
int launch_spmv_sector_matfree(const qbgpu_matrix *A, const FusedArgs &a);      // sectors.cu
void sector_matfree_destroy(qbgpu_matrix *A);
int64_t matfree_bytes(const qbgpu_matrix *A);
int ring_prepare(qbgpu_matrix *A, int rank, int world, int64_t chunk, qbgpu_matrix **view);     // sjds.cu
int peer_ring_flags(const int **flags, int **timeout_flag);                 // peer.cu: arrival flags by ring distance
int peer_mark_fence();                                                      // peer.cu: pulls enqueued later are ordered after THIS point of the compute stream
int peer_pull_fenced(int lane, int slot, void *dst_local, const void *src_peer, size_t bytes);
int peer_record_on_lane(int lane, cudaEvent_t ev);                          // peer.cu: an event behind everything enqueued on that copy lane so far
// species.cu
int launch_spmv_species(const qbgpu_matrix *A, const FusedArgs &args);      // the two-pass products of species-order handles
void species_destroy(qbgpu_matrix *A);
void set_kron_local_variant(int v);       // tuning hook (qbgpu_debug_set_variant(1000 + v)); default 0
int64_t species_bytes(const qbgpu_matrix *A);
// dst[perm[r]] = src[r]  (reference order -> internal order); complex -> real takes the real part, real -> complex sets imag = 0
int vec_to_native(const qbgpu_matrix *A, bool src_cplx, bool dst_cplx, const void *src, void *dst);
// dst[r] = a * src[perm[r]] + b * dst[r]  (internal order -> reference order; b == 0: dst is not read)
int vec_from_native(const qbgpu_matrix *A, bool src_cplx, bool dst_cplx, const void *src, void *dst, double2 a, double2 b);
int mv_species(qbgpu_matrix *A, double2 alpha, const void *x, double2 beta, void *y, int where);   // y = alpha*H*x + beta*y, reference order
int species_split_columns(qbgpu_matrix *A, int nparts, const int64_t *col_bounds, qbgpu_matrix_t *parts);   // views on a matrix-free shard
inline int no_species(const qbgpu_matrix *A, const char *what)
{ return (A && A->sp) ? fail(QBGPU_ERR_STATE, std::string(what) + ": not available for species-order handles") : QBGPU_OK; }
// matrix.cu
int alloc_matrix_arrays(qbgpu_matrix *A);
int split_columns(qbgpu_matrix *A, int nparts, const int64_t *bounds, qbgpu_matrix_t *out, int flags);   // owning part handles by column range
// expand a device-resident reference-format CSR (int64 row_start/row_end/col, offsets from 0) into a new handle
int create_from_device_csr(qbgpu_matrix_t *out, int64_t n, const int64_t *d_rs, const int64_t *d_re, const int64_t *d_col,
                           const void *d_val, bool val_complex, int64_t nnz_input, int sym, int flags, bool api_complex);
// vecops.cu
int vec_dotc(int64_t n, bool cplx, const void *x, const void *y, double *out_dev3);   // out: re, im, (unused)
int vec_dotc_scaled(int64_t n, bool cplx, const void *x, const void *y, double *out_dev3, const double *scale_dev);
int vec_nrm2sq(int64_t n, bool cplx, const void *x, double *out_dev);
// Lanczos step a on one (block of a) handle: w = sx*H*ux - b*sz*uz (first) or w += sx*H_p*ux (later blocks) written to uz;
// when `last`, state[3] = sum Re conj(sx*ux_i) w_i over the local rows.
int lanczos_step_a(const qbgpu_matrix *A, const void *ux_full, void *uz_local, double *state, bool first, bool last, void *w_out = nullptr);   // w_out: the product goes there instead of over uz (dist.cu: speculative early parts)
int vec_axpy(int64_t n, bool cplx, double2 a, const void *x, void *y);
int vec_scal(int64_t n, bool cplx, double2 a, void *x);
int vec_randomize(int64_t n, bool cplx, void *x, uint32_t seed);
int read_scalars(const double *dev, double *host, int count);   // stream-ordered D2H + sync
int vec_imag_norm2(int64_t n, const void *x, double *out_dev);
int vec_take_real(int64_t n, const void *cplx_in, double *real_out);
int vec_put_real(int64_t n, const double *real_in, void *cplx_out);
int lanczos_step_b(int64_t nloc, bool cplx, const void *ux_local, void *uz_local, double *state, const void *w_in = nullptr);                    // w_in: uz = w_in - a*sx*ux (out of place)
int lanczos_step_c(double *state, double *a_dev, double *b_dev, int64_t m);
int cg_update_vr(int64_t n, bool cplx, const double *sc, void *v, void *r, const void *p, const void *pp);
int cg_update_p(int64_t n, bool cplx, double *sc, const void *r, void *p);
int scale_copy(int64_t n, bool cplx, const double *scale_dev, double scale_imm, const void *src, void *dst);

// Scope guards for the device buffers and events of a function that leaves early through QB_TRY / QB_CUDA (an error after an
// allocation -- e.g. out of memory at BASELINE config 3 -- must not leave the earlier ones behind: a retry would fail too).
struct DevBufGuard {
    void *p = nullptr;
    DevBufGuard() = default;
    DevBufGuard(const DevBufGuard &) = delete;
    DevBufGuard &operator=(const DevBufGuard &) = delete;
    ~DevBufGuard() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
};
template <int N> struct EventGuard {
    cudaEvent_t e[N] = {};
    int n = 0;
    EventGuard() = default;
    EventGuard(const EventGuard &) = delete;
    EventGuard &operator=(const EventGuard &) = delete;
    ~EventGuard() { for (int i = 0; i < n; i++) cudaEventDestroy(e[i]); }
    cudaError_t create(unsigned flags = cudaEventDefault) { cudaError_t r = cudaEventCreateWithFlags(&e[n], flags); if (r == cudaSuccess) n++; return r; }
};

}  // namespace qb
