// quantum_basis_b200/csrc/spmv.cu -- the H*v kernels (sm_100a, FP64 CUDA cores, HBM-bound).
//
// Replaces mkl_sparse_{d,z}_mv as called from csr_mat<T>::MultMv2 (reference src/sparse.cc:262-289).  The matrix
// is the expanded Hermitian CSR described in internal.hpp, so each row is a private dot product: no atomics, no
// transposed scatter.  The epilogue fuses what the reference does in separate BLAS-1 sweeps around the product
// (src/lanczos.cc:195-200: the -b*v_{m-2} term and the alpha dot; src/lanczos.cc:320-323: the (eps-E0)*p shift and
// <p,pp>; the Chebyshev recurrence), so that a Krylov step reads H once and each vector once.
//
// Kernel: CSR-vector.  LANES threads cooperate on a row (LANES in {2,4,8,16,32}, chosen per matrix by autotune):
// consecutive lanes read consecutive (col,val) entries -> fully coalesced 4-byte column and 8/16-byte value
// streams issued through the streaming (evict-first) path; the x gathers use the read-only path and own L1/L2;
// the row sum is finished with warp shuffles.  Two independent accumulators per lane keep >= 4 loads in flight.
// Grid = resident blocks per SM x number of SMs (persistent, grid-stride over row groups).
#include "internal.hpp"
#include <cstdlib>
#include <cstring>

namespace qb {

constexpr int kBlock = 256;

template <typename ValT, typename VecT, int LANES, bool DOTS>
__global__ void __launch_bounds__(kBlock, 3)     // min 3 blocks/SM: lets ptxas keep ~8 column/value/gather loads in flight per lane
spmv_csr_vector_kernel(int64_t nrows, int64_t row_lo, const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                       const ValT *__restrict__ val, const VecT *__restrict__ x, const VecT *z, VecT *y,
                       double2 alpha, double2 gamma, double2 beta, int scal_mode, const double *__restrict__ sc,
                       double *dots_out, double *partials, unsigned *ticket)
{
    using VT = VecTraits<VecT>;
    constexpr int RPB = kBlock / LANES;                    // rows per block per sweep
    const int lane = threadIdx.x & (LANES - 1);
    const int grp = threadIdx.x / LANES;
    // shuffle mask = the LANES threads of this row group only: groups of one warp leave the row loop at different
    // trips, and a full-warp mask would wait for lanes that already left
    const unsigned gmask = LANES == 32 ? 0xffffffffu : (((1u << LANES) - 1u) << ((threadIdx.x & 31) & ~(LANES - 1)));
    double dot_scale = 1.0;
    if (scal_mode != 0) {                                  // Lanczos step a (scalars produced by earlier kernels):
        const double sx = sc[0], sz = sc[1], bprev = sc[2]; // 1 = first column block (w = sx*H*ux - b*sz*uz),
        alpha = make_double2(sx, 0.0);                      // 2 = a later column block (w += sx*H_p*ux)
        gamma = make_double2(0.0, 0.0);
        beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
        dot_scale = sx;
    }
    const bool use_gamma = (gamma.x != 0.0 || gamma.y != 0.0);
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    double d[3] = {0.0, 0.0, 0.0};

    for (int64_t row = (int64_t)blockIdx.x * RPB + grp; row < nrows; row += (int64_t)gridDim.x * RPB) {
        const int64_t s = rowptr[row], e = rowptr[row + 1];
        VecT acc0 = VT::zero(), acc1 = VT::zero();
        int64_t k = s + lane;
        for (; k + LANES < e; k += 2 * LANES) {
            const int c0 = ld_stream(col + k), c1 = ld_stream(col + k + LANES);
            const ValT v0 = ld_stream(val + k), v1 = ld_stream(val + k + LANES);
            const VecT x0 = ld_vec(x + c0), x1 = ld_vec(x + c1);
            mac(acc0, v0, x0);
            mac(acc1, v1, x1);
        }
        if (k < e) {
            const int c0 = ld_stream(col + k);
            const ValT v0 = ld_stream(val + k);
            mac(acc0, v0, ld_vec(x + c0));
        }
        VecT acc = VT::add(acc0, acc1);
#pragma unroll
        for (int o = LANES / 2; o > 0; o >>= 1) acc = VT::add(acc, VT::shfl_xor(acc, o, LANES, gmask));
        if (lane == 0) {
            VecT out = VT::scale(alpha, acc);
            VecT xi = VT::zero();
            if (use_gamma || DOTS) xi = x[row_lo + row];
            if (use_gamma) out = VT::add(out, VT::scale(gamma, xi));
            if (use_beta) out = VT::add(out, VT::scale(beta, z[row]));
            y[row] = out;
            if (DOTS) {
                const double2 p = VT::conj_mul(xi, out);
                d[0] += p.x; d[1] += p.y; d[2] += VT::abs2(out);
            }
        }
    }
    if (DOTS) {
        d[0] *= dot_scale; d[1] *= dot_scale;
        block_reduce_finalize<3, kBlock>(d, partials, ticket, dots_out);
    }
}

template <typename ValT, typename VecT, int LANES, bool DOTS>
static int launch_variant(const qbgpu_matrix *A, const FusedArgs &a)
{
    Context &c = ctx();
    auto kern = spmv_csr_vector_kernel<ValT, VecT, LANES, DOTS>;
    static int blocks_per_sm = 0;                          // per template instance
    if (blocks_per_sm == 0) {
        QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, kBlock, 0));
        if (blocks_per_sm < 1) blocks_per_sm = 1;
    }
    const int64_t nrows = A->nrows();
    if (nrows == 0) return QBGPU_OK;
    constexpr int RPB = kBlock / LANES;
    int64_t want = (nrows + RPB - 1) / RPB;
    int64_t cap = (int64_t)c.num_sms * blocks_per_sm;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    const int grid = (int)(want < cap ? want : cap);
    kern<<<grid, kBlock, 0, c.stream>>>(nrows, A->row_lo, A->rowptr, A->col, (const ValT *)A->val, (const VecT *)a.x,
                                        (const VecT *)a.z, (VecT *)a.y, a.alpha, a.gamma, a.beta, a.scal_mode, a.sc,
                                        a.dots, c.partials, c.ticket);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

template <typename ValT, typename VecT, bool DOTS>
static int launch_lanes(const qbgpu_matrix *A, const FusedArgs &a, int lanes)
{
    switch (lanes) {
    case 2:  return launch_variant<ValT, VecT, 2, DOTS>(A, a);
    case 4:  return launch_variant<ValT, VecT, 4, DOTS>(A, a);
    case 8:  return launch_variant<ValT, VecT, 8, DOTS>(A, a);
    case 16: return launch_variant<ValT, VecT, 16, DOTS>(A, a);
    case 32: return launch_variant<ValT, VecT, 32, DOTS>(A, a);
    default: return fail(QBGPU_ERR_ARG, "lanes must be 2,4,8,16 or 32");
    }
}

int launch_spmv(const qbgpu_matrix *A, const FusedArgs &a, int lanes_override)
{
    {   // handles are bound to the device of the thread that uses them first; the context is thread-local
        const int dev = ctx().device;
        if (A->device < 0) A->device = dev;
        else if (A->device != dev) return fail(QBGPU_ERR_STATE, "this handle lives on device " + std::to_string(A->device) + " but the calling thread's context is bound to device " + std::to_string(dev) + " (qbgpu_init(device) in this thread)");
    }
    if (A->sp) return launch_spmv_species(A, a);             // two passes in the handle's internal order (species.cu)
    if (A->mf_sec) return launch_spmv_sector_matfree(A, a);
    if (A->format == QBGPU_FORMAT_MATFREE) return launch_spmv_matfree(A, a);
    if (A->format == QBGPU_FORMAT_SELL) return launch_spmv_sjds(A, a);
    if (A->ndict) return fail(QBGPU_ERR_STATE, "dictionary-coded values need the sliced-jagged layout");
    const int lanes = lanes_override ? lanes_override : A->lanes;
    const bool dots = a.dots != nullptr;
    if (!A->api_complex) {
        return dots ? launch_lanes<double, double, true>(A, a, lanes) : launch_lanes<double, double, false>(A, a, lanes);
    } else if (A->val_real) {
        return dots ? launch_lanes<double, double2, true>(A, a, lanes) : launch_lanes<double, double2, false>(A, a, lanes);
    } else {
        return dots ? launch_lanes<double2, double2, true>(A, a, lanes) : launch_lanes<double2, double2, false>(A, a, lanes);
    }
}

// Pick the lane count per matrix by timing the plain product (the analogue of mkl_sparse_optimize; the reference
// never calls it, src/sparse.cc:258).  Cheap: 5 variants x 3 products.
int autotune(qbgpu_matrix *A, int flags)
{
    Context &c = ctx();
    const int64_t nrows = A->nrows();
    const double mean = nrows ? (double)A->nnz / (double)nrows : 0.0;
    // heuristic default: about 4 entries per lane
    int lanes = 2;
    while (lanes < 32 && mean > 4.0 * lanes) lanes *= 2;
    A->lanes = lanes;
    if (flags & QBGPU_VALUE_DICT) {
        QB_TRY(value_dict_encode(A));                       // opt-in 1-byte value codes; only the sliced-jagged kernel decodes them
        if (A->ndict) return sjds_convert(A, true);
    }
    if (flags & QBGPU_FORMAT_SELL) return sjds_convert(A, true);
    if ((flags & QBGPU_NO_AUTOTUNE) || nrows < 4096) return QBGPU_OK;
    const bool verbose = getenv("QBGPU_VERBOSE") != nullptr;
    const size_t vb = A->vec_bytes();
    DevBufGuard gx, gy;                                     // (freed on every way out of this function)
    EventGuard<3> ge;
    QB_CUDA(gx.alloc(vb * (size_t)A->n));
    QB_CUDA(gy.alloc(vb * (size_t)nrows));
    void *x = gx.p, *y = gy.p;
    QB_TRY(vec_randomize(A->n, A->api_complex, x, 1));
    QB_CUDA(ge.create());
    QB_CUDA(ge.create());
    QB_CUDA(ge.create());
    const cudaEvent_t e0 = ge.e[0], e1 = ge.e[1], t0 = ge.e[2];
    FusedArgs a;
    a.x = x; a.y = y;
    auto time3 = [&](int l, float &ms) -> int {
        QB_TRY(launch_spmv(A, a, l));                       // warm-up
        QB_CUDA(cudaEventRecord(e0, c.stream));
        for (int r = 0; r < 3; r++) QB_TRY(launch_spmv(A, a, l));
        QB_CUDA(cudaEventRecord(e1, c.stream));
        QB_CUDA(cudaEventSynchronize(e1));
        QB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        ms /= 3.0f;
        return QBGPU_OK;
    };
    float best = 1e30f;
    int best_lanes = lanes;
    QB_CUDA(cudaEventRecord(t0, c.stream));
    for (int l = 2; l <= 32; l *= 2) {
        float ms = 0;
        QB_TRY(time3(l, ms));
        if (verbose) fprintf(stderr, "[qbgpu autotune] csr-vector lanes=%2d  %.4f ms/product  (n=%lld nnz=%lld)\n", l, ms, (long long)A->n, (long long)A->nnz);
        if (ms < best) { best = ms; best_lanes = l; }
    }
    A->lanes = best_lanes;
    bool sell_fits = !(flags & QBGPU_FORMAT_CSR);
    if (sell_fits) QB_TRY(sjds_rows_fit(A, &sell_fits));   // a row of 2^24 entries or more: CSR-vector serves it alone
    if (sell_fits) {                                        // try the sliced-jagged layout; keep it only if faster
        QB_TRY(sjds_convert(A, true));
        float ms = 0;
        QB_TRY(time3(0, ms));
        if (verbose) fprintf(stderr, "[qbgpu autotune] sliced-jagged      %.4f ms/product\n", ms);
        if (ms >= best) QB_TRY(sjds_convert(A, false));
    }
    float tot = 0;
    QB_CUDA(cudaEventRecord(e1, c.stream));
    QB_CUDA(cudaEventSynchronize(e1));
    QB_CUDA(cudaEventElapsedTime(&tot, t0, e1));
    A->autotune_s = tot * 1e-3;
    return QBGPU_OK;
}

// ------------------------------------------------------------------ products through the C ABI
static int check_handle(const qbgpu_matrix *A, bool want_complex)
{
    if (!A) return fail(QBGPU_ERR_ARG, "null matrix handle");
    if (A->api_complex != want_complex) return fail(QBGPU_ERR_ARG, "handle scalar type does not match this entry point");
    return QBGPU_OK;
}

static int ensure_stage(void **buf, size_t *have, size_t need)
{
    if (*have >= need) return QBGPU_OK;
    if (*buf) QB_CUDA(cudaFree(*buf));
    *buf = nullptr; *have = 0;
    cudaError_t e = cudaMalloc(buf, need);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(QBGPU_ERR_ALLOC, "cudaMalloc of the staging vector failed"); }
    *have = need;
    return QBGPU_OK;
}

// y = alpha*H*x + beta*y with HOST vectors: H2D(x) [+ H2D(y) when beta != 0], then the product in row chunks whose
// D2H copies run on the copy stream while the next chunk computes (the ARPACK callback path, src/lanczos.cc:426,476).
static int mv_host(const qbgpu_matrix *A, double2 alpha, const void *x, double2 beta, void *y)
{
    Context &c = ctx();
    const size_t vb = A->vec_bytes();
    const int64_t nloc = A->nrows();
    QB_TRY(ensure_stage(&c.stage_x, &c.stage_x_bytes, vb * (size_t)A->n));
    QB_TRY(ensure_stage(&c.stage_y, &c.stage_y_bytes, vb * (size_t)nloc));
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    QB_CUDA(cudaMemcpyAsync(c.stage_x, x, vb * (size_t)A->n, cudaMemcpyHostToDevice, c.stream));
    if (use_beta) QB_CUDA(cudaMemcpyAsync(c.stage_y, y, vb * (size_t)nloc, cudaMemcpyHostToDevice, c.stream));
    const int chunks = nloc >= (1 << 20) ? 8 : 1;
    EventGuard<8> ge;                                       // (destroyed on every way out)
    for (int k = 0; k < chunks; k++) QB_CUDA(ge.create(cudaEventDisableTiming));
    cudaEvent_t *ev = ge.e;
    for (int k = 0; k < chunks; k++) {
        // chunk boundaries on multiples of 32 rows so that a chunk is a whole number of slices in either layout
        const int64_t r0 = (nloc * k / chunks) & ~31LL, r1 = (k + 1 == chunks) ? nloc : ((nloc * (k + 1) / chunks) & ~31LL);
        if (r1 <= r0) { QB_CUDA(cudaEventRecord(ev[k], c.stream)); continue; }
        qbgpu_matrix sub = *A;                              // a view on rows [r0, r1) of this handle
        sub.row_lo = A->row_lo + r0; sub.row_hi = A->row_lo + r1;
        sub.rowptr = A->rowptr + r0;
        if (A->rowinfo) sub.rowinfo = A->rowinfo + r0;
        FusedArgs a;
        a.x = c.stage_x;
        a.y = (char *)c.stage_y + vb * (size_t)r0;
        a.z = use_beta ? a.y : nullptr;
        a.alpha = alpha; a.beta = beta;
        QB_TRY(launch_spmv(&sub, a));
        QB_CUDA(cudaEventRecord(ev[k], c.stream));
        QB_CUDA(cudaStreamWaitEvent(c.copy_stream, ev[k], 0));
        QB_CUDA(cudaMemcpyAsync((char *)y + vb * (size_t)r0, (char *)c.stage_y + vb * (size_t)r0, vb * (size_t)(r1 - r0),
                                cudaMemcpyDeviceToHost, c.copy_stream));
    }
    QB_CUDA(cudaStreamSynchronize(c.copy_stream));
    QB_CUDA(cudaStreamSynchronize(c.stream));
    return QBGPU_OK;
}

// Opt-in (QBGPU_MV_REAL_MODE=1; measured by bench.py's probe before it may become the default): through the reference's
// public API every vector is complex<double>, but with real couplings H is real and so is every vector the reference's
// flows produce (SURVEY F3) -- the fused Krylov loops already run on fp64 vectors then (krylov.cu, real-mode dispatch).
// The same for the plain product with device vectors: when the stored values are real and x (and y, if it is read) has
// no imaginary part at all, multiply on fp64 copies -- half the vector bytes, half the gather sectors -- and widen the
// result.  Exact: the real parts go through the identical fma sequence, the imaginary parts are exact zeros either way.
static int mv_real_mode(qbgpu_matrix *A, double2 alpha, const void *x, double2 beta, void *y, bool *done)
{
    *done = false;
    const bool enabled = getenv("QBGPU_MV_REAL_MODE") != nullptr;          // read per call: a test can switch it around a product
    if (!enabled || !A->api_complex || !A->val_real || A->borrowed || A->row_lo != 0 || A->row_hi != A->n) return QBGPU_OK;
    if (alpha.y != 0.0 || beta.y != 0.0) return QBGPU_OK;
    Context &c = ctx();
    const int64_t n = A->n;
    const bool use_beta = beta.x != 0.0;
    double *t = c.scal_dev + 58;
    double h[2] = {0.0, 0.0};
    QB_TRY(vec_imag_norm2(n, x, t));
    if (use_beta) QB_TRY(vec_imag_norm2(n, y, t + 1));
    QB_TRY(read_scalars(t, h, use_beta ? 2 : 1));
    if (h[0] != 0.0 || h[1] != 0.0) return QBGPU_OK;
    // (an allocation failure here is not an error of the product: fall back to the complex kernels)
    if (!A->perm_x && cudaMalloc(&A->perm_x, sizeof(double) * (size_t)n) != cudaSuccess) { (void)cudaGetLastError(); A->perm_x = nullptr; return QBGPU_OK; }
    if (!A->perm_y && cudaMalloc(&A->perm_y, sizeof(double) * (size_t)n) != cudaSuccess) { (void)cudaGetLastError(); A->perm_y = nullptr; return QBGPU_OK; }
    QB_TRY(vec_take_real(n, x, (double *)A->perm_x));
    if (use_beta) QB_TRY(vec_take_real(n, y, (double *)A->perm_y));
    qbgpu_matrix R = *A;                                    // same arrays, fp64 vectors
    R.api_complex = false;
    FusedArgs a;
    a.x = A->perm_x; a.y = A->perm_y; a.z = A->perm_y; a.alpha = alpha; a.beta = beta;
    QB_TRY(launch_spmv(&R, a));
    QB_TRY(vec_put_real(n, (const double *)A->perm_y, y));
    *done = true;
    return QBGPU_OK;
}

static int mv_any(qbgpu_matrix *A, double2 alpha, const void *x, double2 beta, void *y, int where)
{
    QB_TRY(ensure_init());
    if (!x || !y) return fail(QBGPU_ERR_ARG, "null vector pointer");
    if (A->sp && A->perm) return mv_species(A, alpha, x, beta, y, where);   // reference order at the boundary, internal order inside
    if (A->sp && where == QBGPU_HOST) return fail(QBGPU_ERR_STATE, "host-vector products on a shard or column part of a species-order handle are not available");
    if (where == QBGPU_DEVICE) {
        bool done = false;
        QB_TRY(mv_real_mode(A, alpha, x, beta, y, &done));
        if (done) return QBGPU_OK;
    }
    if (where == QBGPU_HOST) return mv_host(A, alpha, x, beta, y);
    if (where != QBGPU_DEVICE) return fail(QBGPU_ERR_ARG, "where must be QBGPU_HOST or QBGPU_DEVICE");
    FusedArgs a;
    a.x = x; a.y = y; a.z = y; a.alpha = alpha; a.beta = beta;
    return launch_spmv(A, a);
}

int lanczos_step_a(const qbgpu_matrix *A, const void *ux_full, void *uz_local, double *state, bool first, bool last, void *w_out)
{
    FusedArgs a;
    a.x = ux_full; a.z = uz_local; a.y = uz_local;
    if (w_out) { a.y = w_out; if (!first) a.z = w_out; }   // the opening part reads uz and writes w; the others accumulate into w
    a.scal_mode = first ? 1 : 2; a.sc = state;
    a.beta = make_double2(1.0, 0.0);                       // placeholder: the kernel derives beta from the state
    // complex vectors: the dot rides in the product's epilogue (+0.5 ms on BASELINE config 3).  fp64 vectors: the
    // epilogue variant of the kernel costs 2-4 ms there (profiles/r01_kbench_fused_*.txt) while a separate pass over
    // the two local vectors costs 0.45 ms, so the dot is a second kernel.
    const bool fuse_dot = A->api_complex;
    a.dots = (last && fuse_dot) ? state + 3 : nullptr;     // state[3]=alpha partial, [4]=Im (unused), [5]=|w|^2 (unused)
    QB_TRY(launch_spmv(A, a));
    if (last && !fuse_dot)
        QB_TRY(vec_dotc_scaled(A->nrows(), false, (const double *)ux_full + A->row_lo, w_out ? w_out : uz_local, state + 3, state + 0));
    return QBGPU_OK;
}

}  // namespace qb

using namespace qb;

extern "C" {

int qbgpu_dmv(qbgpu_matrix_t A, double alpha, const double *x, double beta, double *y, int where)
{
    QB_TRY(check_handle(A, false));
    return mv_any(A, make_double2(alpha, 0.0), x, make_double2(beta, 0.0), y, where);
}

int qbgpu_zmv(qbgpu_matrix_t A, const double alpha[2], const void *x, const double beta[2], void *y, int where)
{
    QB_TRY(check_handle(A, true));
    if (!alpha || !beta) return fail(QBGPU_ERR_ARG, "null scalar pointer");
    return mv_any(A, make_double2(alpha[0], alpha[1]), x, make_double2(beta[0], beta[1]), y, where);
}

int qbgpu_spmv_fused(qbgpu_matrix_t A, const void *x, const void *z, void *y, const double alpha[2],
                     const double gamma[2], const double beta[2], double *dots_dev)
{
    QB_TRY(ensure_init());
    if (!A || !x || !y || !alpha || !gamma || !beta) return fail(QBGPU_ERR_ARG, "null argument");
    FusedArgs a;
    a.x = x; a.z = z; a.y = y;
    a.alpha = make_double2(alpha[0], alpha[1]); a.gamma = make_double2(gamma[0], gamma[1]); a.beta = make_double2(beta[0], beta[1]);
    if ((a.beta.x != 0.0 || a.beta.y != 0.0) && !z) return fail(QBGPU_ERR_ARG, "beta != 0 needs z");
    a.dots = dots_dev;
    return launch_spmv(A, a);
}

int qbgpu_lanczos_step_a_part(qbgpu_matrix_t A, const void *ux_full, void *uz_local, double *state_dev, int first, int last)
{
    QB_TRY(ensure_init());
    if (!A || !ux_full || !uz_local || !state_dev) return fail(QBGPU_ERR_ARG, "null argument");
    return lanczos_step_a(A, ux_full, uz_local, state_dev, first != 0, last != 0);
}

int qbgpu_lanczos_step_a(qbgpu_matrix_t A, const void *ux_full, void *uz_local, double *state_dev)
{
    return qbgpu_lanczos_step_a_part(A, ux_full, uz_local, state_dev, 1, 1);
}

}  // extern "C"
