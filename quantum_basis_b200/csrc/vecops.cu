// quantum_basis_b200/csrc/vecops.cu -- fused vector passes around the H*v kernel (HBM-bound, one read per operand).
//
// These replace the BLAS-1 sweeps of the reference's Krylov loops (cblas_{d,z}{dot,axpy,nrm2,scal,copy},
// src/lanczos.cc:10-53 and their call sites :195-214, :296-330; src/kpm.cc:57-76).  All reductions are
// deterministic (fixed grid, per-block partials, fixed-shape final tree) and leave their result in device memory,
// so consecutive passes chain without a host round trip.
#include "internal.hpp"

namespace qb {

constexpr int kVBlock = 256;

static int vec_grid(int64_t n)
{
    Context &c = ctx();
    int64_t want = (n + kVBlock - 1) / kVBlock;
    int64_t cap = (int64_t)c.num_sms * 8;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

// grid-stride loop, unrolled by 4 so that each thread keeps 4 independent element loads per operand in flight
#define GRID_STRIDE(i, n) _Pragma("unroll 4") for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (int64_t)gridDim.x * blockDim.x)

// ------------------------------------------------------------------------------------- dot / nrm2 / axpy / scal
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) dotc_kernel(int64_t n, const VecT *__restrict__ x, const VecT *__restrict__ y,
                                                       double *out, double *partials, unsigned *ticket, const double *scale_dev)
{
    using VT = VecTraits<VecT>;
    double d[3] = {0.0, 0.0, 0.0};
    GRID_STRIDE(i, n) { const VecT xi = x[i], yi = y[i]; const double2 p = VT::conj_mul(xi, yi); d[0] += p.x; d[1] += p.y; d[2] += VT::abs2(yi); }
    if (scale_dev) { const double s = *scale_dev; d[0] *= s; d[1] *= s; }      // <s*x, y> for an unnormalised x
    block_reduce_finalize<3, kVBlock>(d, partials, ticket, out);
}
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) nrm2sq_kernel(int64_t n, const VecT *__restrict__ x, double *out, double *partials, unsigned *ticket)
{
    using VT = VecTraits<VecT>;
    double d[1] = {0.0};
    GRID_STRIDE(i, n) d[0] += VT::abs2(x[i]);
    block_reduce_finalize<1, kVBlock>(d, partials, ticket, out);
}
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) axpy_kernel(int64_t n, double2 a, const VecT *__restrict__ x, VecT *y)
{
    using VT = VecTraits<VecT>;
    GRID_STRIDE(i, n) y[i] = VT::add(y[i], VT::scale(a, x[i]));
}
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) scal_kernel(int64_t n, double2 a, VecT *x)
{
    using VT = VecTraits<VecT>;
    GRID_STRIDE(i, n) x[i] = VT::scale(a, x[i]);
}
// dst = s * src with s = (scale_dev ? *scale_dev : 1) * scale_imm
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) scale_copy_kernel(int64_t n, const double *scale_dev, double scale_imm,
                                                             const VecT *src, VecT *dst)      // src may alias dst
{
    using VT = VecTraits<VecT>;
    const double s = (scale_dev ? *scale_dev : 1.0) * scale_imm;
    GRID_STRIDE(i, n) dst[i] = VT::rscale(s, src[i]);
}

#define LAUNCH_V(kern, n, ...)                                                    \
    do {                                                                          \
        kern<<<vec_grid(n), kVBlock, 0, ctx().stream>>>(__VA_ARGS__);             \
        QB_LAUNCH_COUNT();                                                        \
        QB_CUDA(cudaGetLastError());                                              \
    } while (0)

int vec_dotc_scaled(int64_t n, bool cplx, const void *x, const void *y, double *out3, const double *scale_dev)
{
    Context &c = ctx();
    if (cplx) LAUNCH_V(dotc_kernel<double2>, n, n, (const double2 *)x, (const double2 *)y, out3, c.partials, c.ticket, scale_dev);
    else      LAUNCH_V(dotc_kernel<double>, n, n, (const double *)x, (const double *)y, out3, c.partials, c.ticket, scale_dev);
    return QBGPU_OK;
}
int vec_dotc(int64_t n, bool cplx, const void *x, const void *y, double *out3) { return vec_dotc_scaled(n, cplx, x, y, out3, nullptr); }
int vec_nrm2sq(int64_t n, bool cplx, const void *x, double *out)
{
    Context &c = ctx();
    if (cplx) LAUNCH_V(nrm2sq_kernel<double2>, n, n, (const double2 *)x, out, c.partials, c.ticket);
    else      LAUNCH_V(nrm2sq_kernel<double>, n, n, (const double *)x, out, c.partials, c.ticket);
    return QBGPU_OK;
}
int vec_axpy(int64_t n, bool cplx, double2 a, const void *x, void *y)
{
    if (cplx) LAUNCH_V(axpy_kernel<double2>, n, n, a, (const double2 *)x, (double2 *)y);
    else      LAUNCH_V(axpy_kernel<double>, n, n, a, (const double *)x, (double *)y);
    return QBGPU_OK;
}
int vec_scal(int64_t n, bool cplx, double2 a, void *x)
{
    if (cplx) LAUNCH_V(scal_kernel<double2>, n, n, a, (double2 *)x);
    else      LAUNCH_V(scal_kernel<double>, n, n, a, (double *)x);
    return QBGPU_OK;
}
int scale_copy(int64_t n, bool cplx, const double *scale_dev, double scale_imm, const void *src, void *dst)
{
    if (cplx) LAUNCH_V(scale_copy_kernel<double2>, n, n, scale_dev, scale_imm, (const double2 *)src, (double2 *)dst);
    else      LAUNCH_V(scale_copy_kernel<double>, n, n, scale_dev, scale_imm, (const double *)src, (double *)dst);
    return QBGPU_OK;
}

// ----------------------------------------------------------------- real <-> complex views of an all-real vector
__global__ void __launch_bounds__(kVBlock, 4) imag_abs2_kernel(int64_t n, const double2 *__restrict__ x, double *out, double *partials, unsigned *ticket)
{
    double d[1] = {0.0};
    GRID_STRIDE(i, n) { const double im = x[i].y; d[0] += im * im; }
    block_reduce_finalize<1, kVBlock>(d, partials, ticket, out);
}
__global__ void __launch_bounds__(kVBlock, 4) take_real_kernel(int64_t n, const double2 *__restrict__ in, double *out) { GRID_STRIDE(i, n) out[i] = in[i].x; }
__global__ void __launch_bounds__(kVBlock, 4) put_real_kernel(int64_t n, const double *__restrict__ in, double2 *out) { GRID_STRIDE(i, n) out[i] = make_double2(in[i], 0.0); }

int vec_imag_norm2(int64_t n, const void *x, double *out_dev)
{
    Context &c = ctx();
    LAUNCH_V(imag_abs2_kernel, n, n, (const double2 *)x, out_dev, c.partials, c.ticket);
    return QBGPU_OK;
}
int vec_take_real(int64_t n, const void *cplx_in, double *real_out) { LAUNCH_V(take_real_kernel, n, n, (const double2 *)cplx_in, real_out); return QBGPU_OK; }
int vec_put_real(int64_t n, const double *real_in, void *cplx_out) { LAUNCH_V(put_real_kernel, n, n, real_in, (double2 *)cplx_out); return QBGPU_OK; }

int read_scalars(const double *dev, double *host, int count)
{
    Context &c = ctx();
    if (count > 64) return fail(QBGPU_ERR_ARG, "read_scalars: too many");
    QB_CUDA(cudaMemcpyAsync(c.scal_host, dev, sizeof(double) * count, cudaMemcpyDeviceToHost, c.stream));
    QB_CUDA(cudaStreamSynchronize(c.stream));
    for (int i = 0; i < count; i++) host[i] = c.scal_host[i];
    return QBGPU_OK;
}

// -------------------------------------------------------------------------------------------- vec_randomize
// std::minstd_rand0 is the Lehmer generator s <- 16807*s mod (2^31-1) (reference src/miscellaneous.cc:380-382).
// Element j needs s_j = seed * 16807^(j+1) mod p: each thread jumps to its first element by modular
// exponentiation and then steps sequentially, so the element values are bit-identical to the host sequence.
__device__ __forceinline__ uint64_t lehmer_pow(uint64_t base, uint64_t e)
{
    const uint64_t p = 2147483647ull;
    uint64_t r = 1;
    base %= p;
    while (e) { if (e & 1) r = (r * base) % p; base = (base * base) % p; e >>= 1; }
    return r;
}
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) randomize_kernel(int64_t n, VecT *x, uint32_t seed, int64_t per_thread)
{
    const uint64_t p = 2147483647ull;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t j0 = t * per_thread;
    if (j0 >= n) return;
    uint64_t s0 = seed % p;
    if (s0 == 0) s0 = 1;
    uint64_t s = (s0 * lehmer_pow(16807ull, (uint64_t)j0)) % p;
    const double pref = 1.0 / 2147483647.0;
    const int64_t j1 = (j0 + per_thread < n) ? j0 + per_thread : n;
    for (int64_t j = j0; j < j1; j++) {
        s = (s * 16807ull) % p;
        const double v = (double)s * pref - 0.5;
        if constexpr (sizeof(VecT) == 16) x[j] = make_double2(v, 0.0); else x[j] = v;
    }
}
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) fill_kernel(int64_t n, VecT *x, double v)
{
    GRID_STRIDE(i, n) { if constexpr (sizeof(VecT) == 16) x[i] = make_double2(v, 0.0); else x[i] = v; }
}

int vec_randomize(int64_t n, bool cplx, void *x, uint32_t seed)
{
    Context &c = ctx();
    if (n <= 0) return QBGPU_OK;
    if (seed == 0) {                                       // constant vector 1/sqrt(n), src/miscellaneous.cc:374-377
        const double v = sqrt(1.0 / (double)n);
        if (cplx) LAUNCH_V(fill_kernel<double2>, n, n, (double2 *)x, v);
        else      LAUNCH_V(fill_kernel<double>, n, n, (double *)x, v);
        return QBGPU_OK;
    }
    const int64_t per_thread = 64;
    const int64_t threads = (n + per_thread - 1) / per_thread;
    const int grid = (int)((threads + kVBlock - 1) / kVBlock);
    if (cplx) randomize_kernel<double2><<<grid, kVBlock, 0, c.stream>>>(n, (double2 *)x, seed, per_thread);
    else      randomize_kernel<double><<<grid, kVBlock, 0, c.stream>>>(n, (double *)x, seed, per_thread);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    // normalise: x /= nrm2(x)  (src/miscellaneous.cc:383-384)
    double *nn = c.scal_dev + 40;
    QB_TRY(vec_nrm2sq(n, cplx, x, nn));
    double h;
    QB_TRY(read_scalars(nn, &h, 1));
    QB_TRY(vec_scal(n, cplx, make_double2(1.0 / sqrt(h), 0.0), x));
    return QBGPU_OK;
}

// ---------------------------------------------------------------------------------------- Lanczos step b, c
// state: [0]=sx [1]=sz [2]=b_prev [3]=alpha [4],[5] scratch [6]=norm2 [7] spare  (see include/qbgpu.h)
// step b: w' = uz - alpha*sx*ux -> uz ; state[6] = sum |w'|^2   (reference: axpy + nrm2, src/lanczos.cc:206-208)
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) lanczos_b_kernel(int64_t n, const VecT *__restrict__ ux, const VecT *win, VecT *uz, double *state,
                                                               double *partials, unsigned *ticket)
{
    using VT = VecTraits<VecT>;
    const double f = -state[3] * state[0];
    double d[1] = {0.0};
    // 4 elements per thread per trip, all loads first: uz is read and written, so without the explicit batching the
    // compiler keeps each load behind the previous store
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += 4 * stride) {
        VecT w[4], v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) { const int64_t j = i + k * stride; if (j < n) { w[k] = win[j]; v[k] = ux[j]; } }      // (win == uz: in place)
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int64_t j = i + k * stride;
            if (j < n) { const VecT r = VT::add(w[k], VT::rscale(f, v[k])); uz[j] = r; d[0] += VT::abs2(r); }
        }
    }
    block_reduce_finalize<1, kVBlock>(d, partials, ticket, state + 6);
}
// step c: b_m = sqrt(norm2); record a_{m-1}, b_m; the freshly written buffer becomes x with scale 1/b_m
// (the reference's scal by 1/b, src/lanczos.cc:214, is deferred into the next product's alpha).
__global__ void lanczos_c_kernel(double *state, double *a_dev, double *b_dev, int64_t m)
{
    const double b = sqrt(state[6]);
    a_dev[m - 1] = state[3];
    b_dev[m] = b;
    const double sx_old = state[0];
    state[0] = 1.0 / b;
    state[1] = sx_old;
    state[2] = b;
}

int lanczos_step_b(int64_t nloc, bool cplx, const void *ux_local, void *uz_local, double *state, const void *w_in)
{
    Context &c = ctx();
    if (!w_in) w_in = uz_local;
    if (cplx) LAUNCH_V(lanczos_b_kernel<double2>, nloc, nloc, (const double2 *)ux_local, (const double2 *)w_in, (double2 *)uz_local, state, c.partials, c.ticket);
    else      LAUNCH_V(lanczos_b_kernel<double>, nloc, nloc, (const double *)ux_local, (const double *)w_in, (double *)uz_local, state, c.partials, c.ticket);
    return QBGPU_OK;
}
int lanczos_step_c(double *state, double *a_dev, double *b_dev, int64_t m)
{
    lanczos_c_kernel<<<1, 1, 0, ctx().stream>>>(state, a_dev, b_dev, m);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

// ------------------------------------------------------------------ Lanczos step re-orthogonalised against phi0 (sr_val1)
// The reference's re-orthogonalisation (src/lanczos.cc:218-226: tmp = <phi0, v_m>; if |tmp| > 2e-12 { v_m -= tmp phi0;
// v_m /= |v_m| }) on the unnormalised vector v_m = sx*U: U -= h phi0 with h = <phi0, U>, then sx = 1/|U|.  The decision is
// taken on the device from the reduced sums, so a multi-GPU loop can order the projection before the next step's pulls
// without a host round trip.  p1 (device, 8 doubles): [0] = |U|^2, [1], [2] = Re, Im <phi0, U> (partials, then reduced),
// [3] = projection flag, [4], [5] = -h, [6] = |U - h phi0|^2, [7] spare.
// step b with the phi0 dot: as lanczos_b_kernel, plus the partial <phi0, U> of the freshly written U, in the same pass
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) lanczos_b_phi_kernel(int64_t n, const VecT *__restrict__ ux, const VecT *win, VecT *uz,
                                                                   const VecT *__restrict__ phi, const double *state, double *p1,
                                                                   double *partials, unsigned *ticket)
{
    using VT = VecTraits<VecT>;
    const double f = -state[3] * state[0];
    double d[3] = {0.0, 0.0, 0.0};
    // loads batched as in lanczos_b_kernel: 96 bytes per thread in flight (4 real or 2 complex elements of three operands;
    // 4 complex ones spill at the 64 registers of 4 blocks per SM)
    constexpr int B = sizeof(VecT) == 16 ? 2 : 4;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += B * stride) {
        VecT w[B], v[B], q[B];
#pragma unroll
        for (int k = 0; k < B; k++) { const int64_t j = i + k * stride; if (j < n) { w[k] = win[j]; v[k] = ux[j]; q[k] = phi[j]; } }
#pragma unroll
        for (int k = 0; k < B; k++) {
            const int64_t j = i + k * stride;
            if (j < n) {
                const VecT r = VT::add(w[k], VT::rscale(f, v[k]));
                uz[j] = r;
                d[0] += VT::abs2(r);
                const double2 h = VT::conj_mul(q[k], r);
                d[1] += h.x; d[2] += h.y;
            }
        }
    }
    block_reduce_finalize<3, kVBlock>(d, partials, ticket, p1);
}
// step c for sr_val1: lanczos_c_kernel on the reduced |U|^2 (b_m is recorded before the projection, as the reference records
// it), then the decision |h sx| > 2e-12 with the new sx = 1/b_m.  No projection in the start-up step (m == 1): the reference's
// first step has no checks (:167-191).
__global__ void lanczos_c_phi_kernel(double *state, double *p1, double *a_dev, double *b_dev, int64_t m)
{
    const double b = sqrt(p1[0]);
    a_dev[m - 1] = state[3];
    b_dev[m] = b;
    const double sx_old = state[0];
    const double sx = 1.0 / b;
    state[0] = sx;
    state[1] = sx_old;
    state[2] = b;
    const double tr = p1[1] * sx, ti = p1[2] * sx;
    p1[3] = (m > 1 && sqrt(tr * tr + ti * ti) > 2e-12) ? 1.0 : 0.0;
    p1[4] = -p1[1];
    p1[5] = -p1[2];
}
// projection pass: when the flag is set U += (-h) phi0 and p1[6] = partial |U|^2 (else 0; the vector is not touched)
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) lanczos_project_kernel(int64_t n, const VecT *__restrict__ phi, VecT *uz, double *p1,
                                                                     double *partials, unsigned *ticket)
{
    using VT = VecTraits<VecT>;
    double d[1] = {0.0};
    if (p1[3] != 0.0) {
        const double2 c = make_double2(p1[4], p1[5]);
        GRID_STRIDE(i, n) { const VecT r = VT::add(uz[i], VT::scale(c, phi[i])); uz[i] = r; d[0] += VT::abs2(r); }
    }
    block_reduce_finalize<1, kVBlock>(d, partials, ticket, p1 + 6);
}
// after the all-reduce of p1[6]: the projected vector's scale
__global__ void lanczos_project_finalize_kernel(double *state, const double *p1)
{
    if (p1[3] != 0.0) state[0] = 1.0 / sqrt(p1[6]);
}

int lanczos_step_b_phi(int64_t nloc, bool cplx, const void *ux_local, void *uz_local, const void *phi_local, const double *state, double *p1,
                       const void *w_in)
{
    Context &c = ctx();
    if (!w_in) w_in = uz_local;
    if (cplx) LAUNCH_V(lanczos_b_phi_kernel<double2>, nloc, nloc, (const double2 *)ux_local, (const double2 *)w_in, (double2 *)uz_local, (const double2 *)phi_local, state, p1, c.partials, c.ticket);
    else      LAUNCH_V(lanczos_b_phi_kernel<double>, nloc, nloc, (const double *)ux_local, (const double *)w_in, (double *)uz_local, (const double *)phi_local, state, p1, c.partials, c.ticket);
    return QBGPU_OK;
}
int lanczos_step_c_phi(double *state, double *p1, double *a_dev, double *b_dev, int64_t m)
{
    lanczos_c_phi_kernel<<<1, 1, 0, ctx().stream>>>(state, p1, a_dev, b_dev, m);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}
int lanczos_project(int64_t nloc, bool cplx, const void *phi_local, void *uz_local, double *p1)
{
    Context &c = ctx();
    if (cplx) LAUNCH_V(lanczos_project_kernel<double2>, nloc, nloc, (const double2 *)phi_local, (double2 *)uz_local, p1, c.partials, c.ticket);
    else      LAUNCH_V(lanczos_project_kernel<double>, nloc, nloc, (const double *)phi_local, (double *)uz_local, p1, c.partials, c.ticket);
    return QBGPU_OK;
}
int lanczos_project_finalize(double *state, const double *p1)
{
    lanczos_project_finalize_kernel<<<1, 1, 0, ctx().stream>>>(state, p1);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

// ------------------------------------------------------------------------------------------------ CG passes
// sc (device): [0]=gamma (residual norm, `accu`) [1],[2]=delta=<p,pp> (re,im) [3]=|pp|^2 scratch [4]=|r|^2
// pass 1 (src/lanczos.cc:324-327): alpha = gamma^2/delta ; v += alpha p ; r -= alpha pp ; sc[4] = |r|^2
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) cg_vr_kernel(int64_t n, const double *__restrict__ sc, VecT *v, VecT *r,
                                                        const VecT *__restrict__ p, const VecT *__restrict__ pp,
                                                        double *out, double *partials, unsigned *ticket)
{
    using VT = VecTraits<VecT>;
    const double g2 = sc[0] * sc[0];
    double2 alpha;
    if (VT::ncomp == 1) alpha = make_double2(g2 / sc[1], 0.0);
    else { const double den = sc[1] * sc[1] + sc[2] * sc[2]; alpha = make_double2(g2 * sc[1] / den, -g2 * sc[2] / den); }
    const double2 nalpha = make_double2(-alpha.x, -alpha.y);
    double d[1] = {0.0};
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += 2 * stride) {     // loads batched, see lanczos_b_kernel
        VecT vv[2], rr[2], pv[2], qv[2];
#pragma unroll
        for (int k = 0; k < 2; k++) { const int64_t j = i + k * stride; if (j < n) { vv[k] = v[j]; rr[k] = r[j]; pv[k] = p[j]; qv[k] = pp[j]; } }
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const int64_t j = i + k * stride;
            if (j < n) {
                v[j] = VT::add(vv[k], VT::scale(alpha, pv[k]));
                const VecT ri = VT::add(rr[k], VT::scale(nalpha, qv[k]));
                r[j] = ri;
                d[0] += VT::abs2(ri);
            }
        }
    }
    block_reduce_finalize<1, kVBlock>(d, partials, ticket, out);
}
// pass 2 (src/lanczos.cc:327-330): beta = |r|/gamma ; p = r + beta^2 p ; gamma *= beta (written to sc[5])
template <typename VecT>
__global__ void __launch_bounds__(kVBlock, 4) cg_p_kernel(int64_t n, double *sc, const VecT *__restrict__ r, VecT *p)
{
    using VT = VecTraits<VecT>;
    const double beta = sqrt(sc[4]) / sc[0];
    const double b2 = beta * beta;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += 4 * stride) {
        VecT rv[4], pv[4];
#pragma unroll
        for (int k = 0; k < 4; k++) { const int64_t j = i + k * stride; if (j < n) { rv[k] = r[j]; pv[k] = p[j]; } }
#pragma unroll
        for (int k = 0; k < 4; k++) { const int64_t j = i + k * stride; if (j < n) p[j] = VT::add(rv[k], VT::rscale(b2, pv[k])); }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) sc[5] = sc[0] * beta;
}

int cg_update_vr(int64_t n, bool cplx, const double *sc, void *v, void *r, const void *p, const void *pp)
{
    Context &c = ctx();
    double *out = const_cast<double *>(sc) + 4;
    if (cplx) LAUNCH_V(cg_vr_kernel<double2>, n, n, sc, (double2 *)v, (double2 *)r, (const double2 *)p, (const double2 *)pp, out, c.partials, c.ticket);
    else      LAUNCH_V(cg_vr_kernel<double>, n, n, sc, (double *)v, (double *)r, (const double *)p, (const double *)pp, out, c.partials, c.ticket);
    return QBGPU_OK;
}
int cg_update_p(int64_t n, bool cplx, double *sc, const void *r, void *p)
{
    if (cplx) LAUNCH_V(cg_p_kernel<double2>, n, n, sc, (const double2 *)r, (double2 *)p);
    else      LAUNCH_V(cg_p_kernel<double>, n, n, sc, (const double *)r, (double *)p);
    return QBGPU_OK;
}

}  // namespace qb

using namespace qb;

// --------------------------------------------------------------------------------------------- C ABI: BLAS-1
extern "C" {

int qbgpu_vec_randomize_d(int64_t n, double *x, uint32_t seed) { QB_TRY(ensure_init()); return vec_randomize(n, false, x, seed); }
int qbgpu_vec_randomize_z(int64_t n, void *x, uint32_t seed) { QB_TRY(ensure_init()); return vec_randomize(n, true, x, seed); }

int qbgpu_zdotc(int64_t n, const void *x, const void *y, double result[2])
{
    QB_TRY(ensure_init());
    double *o = ctx().scal_dev + 44;
    QB_TRY(vec_dotc(n, true, x, y, o));
    return read_scalars(o, result, 2);
}
int qbgpu_ddot(int64_t n, const double *x, const double *y, double *result)
{
    QB_TRY(ensure_init());
    double *o = ctx().scal_dev + 44;
    QB_TRY(vec_dotc(n, false, x, y, o));
    return read_scalars(o, result, 1);
}
int qbgpu_dznrm2(int64_t n, const void *x, double *result)
{
    QB_TRY(ensure_init());
    double *o = ctx().scal_dev + 48;
    QB_TRY(vec_nrm2sq(n, true, x, o));
    QB_TRY(read_scalars(o, result, 1));
    *result = sqrt(*result);
    return QBGPU_OK;
}
int qbgpu_dnrm2(int64_t n, const double *x, double *result)
{
    QB_TRY(ensure_init());
    double *o = ctx().scal_dev + 48;
    QB_TRY(vec_nrm2sq(n, false, x, o));
    QB_TRY(read_scalars(o, result, 1));
    *result = sqrt(*result);
    return QBGPU_OK;
}
int qbgpu_zaxpy(int64_t n, const double a[2], const void *x, void *y) { QB_TRY(ensure_init()); return vec_axpy(n, true, make_double2(a[0], a[1]), x, y); }
int qbgpu_daxpy(int64_t n, double a, const double *x, double *y) { QB_TRY(ensure_init()); return vec_axpy(n, false, make_double2(a, 0.0), x, y); }
int qbgpu_zscal(int64_t n, const double a[2], void *x) { QB_TRY(ensure_init()); return vec_scal(n, true, make_double2(a[0], a[1]), x); }
int qbgpu_dscal(int64_t n, double a, double *x) { QB_TRY(ensure_init()); return vec_scal(n, false, make_double2(a, 0.0), x); }

int qbgpu_lanczos_step_b(qbgpu_matrix_t A, const void *ux_local, void *uz_local, double *state_dev)
{
    QB_TRY(ensure_init());
    if (!A || !ux_local || !uz_local || !state_dev) return fail(QBGPU_ERR_ARG, "null argument");
    return lanczos_step_b(A->nrows(), A->api_complex, ux_local, uz_local, state_dev);
}
int qbgpu_lanczos_step_c(double *state_dev, double *a_dev, double *b_dev, int64_t m)
{
    QB_TRY(ensure_init());
    if (!state_dev || !a_dev || !b_dev || m < 1) return fail(QBGPU_ERR_ARG, "bad argument");
    return lanczos_step_c(state_dev, a_dev, b_dev, m);
}

}  // extern "C"
