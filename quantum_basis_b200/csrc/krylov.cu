// quantum_basis_b200/csrc/krylov.cu -- device-resident Krylov loops behind the reference's lanczos(), eigenvec_CG()
// and energy_scale() signatures, plus Chebyshev/KPM moments (new functionality).
//
// Reference loops: src/lanczos.cc:134-266 (lanczos), :281-341 (eigenvec_CG), :355-390 (hess_eigen),
// src/kpm.cc:45-88 (energy_scale).  What changes is the data flow, not the mathematics: vectors stay in HBM, each
// step is 2-3 fused kernels (one pass over H, one over each vector), scalars chain through device memory, and the
// host only sees (a_m, b_m) to evaluate the reference's stop rule.  The checkpoint hooks and the per-step log
// files of the reference (ckpt_lanczos_update, log_Lanczos_srval, log_CG.txt) are host I/O outside the path.
#include "internal.hpp"
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace qb {

constexpr double kLanczosPrecision = 2e-12;   // reference src/miscellaneous.cc:47

// ---------------------------------------------------------------------------------------------- hess_eigen
// Implicit QL with Wilkinson shifts for the symmetric tridiagonal (diag d, off-diag e).  The reference calls
// LAPACKE_dstedc('I') (src/lanczos.cc:367).  z: full eigenvector matrix (m x m column-major, identity on entry),
// or null; zlast: only the last row of the eigenvector matrix (e_m^T Q), or null -- the stop rule needs
// s[m-1] of the lowest Ritz vector only (src/lanczos.cc:231), which keeps the per-step cost O(m^2).
static int tridiag_ql(int64_t m, double *d, double *e, double *z, double *zlast)
{
    for (int64_t l = 0; l < m; l++) {
        int iter = 0;
        int64_t mm;
        do {
            for (mm = l; mm < m - 1; mm++) {
                const double dd = fabs(d[mm]) + fabs(d[mm + 1]);
                if (fabs(e[mm]) <= DBL_EPSILON * dd) break;
            }
            if (mm != l) {
                if (iter++ == 300) return 1;
                double g = (d[l + 1] - d[l]) / (2.0 * e[l]);
                double r = hypot(g, 1.0);
                g = d[mm] - d[l] + e[l] / (g + copysign(r, g));
                double s = 1.0, c = 1.0, p = 0.0;
                int64_t i;
                bool underflow = false;
                for (i = mm - 1; i >= l; i--) {
                    double f = s * e[i];
                    const double b = c * e[i];
                    r = hypot(f, g);
                    e[i + 1] = r;
                    if (r == 0.0) { d[i + 1] -= p; e[mm] = 0.0; underflow = true; break; }
                    s = f / r; c = g / r;
                    g = d[i + 1] - p;
                    r = (d[i] - g) * s + 2.0 * c * b;
                    p = s * r;
                    d[i + 1] = g + p;
                    g = c * r - b;
                    if (z) for (int64_t k = 0; k < m; k++) {
                        f = z[k + (i + 1) * m];
                        z[k + (i + 1) * m] = s * z[k + i * m] + c * f;
                        z[k + i * m] = c * z[k + i * m] - s * f;
                    }
                    if (zlast) { f = zlast[i + 1]; zlast[i + 1] = s * zlast[i] + c * f; zlast[i] = c * zlast[i] - s * f; }
                }
                if (underflow) continue;
                d[l] -= p; e[l] = g; e[mm] = 0.0;
            }
        } while (mm != l);
    }
    return 0;
}

// Smallest eigenvalue of the m x m tridiagonal (diag hess[maxit+j], off-diag hess[j+1]) by bisection on the Sturm
// count, to machine precision.  O(m) per evaluation: the per-step part of the stop rule (the relative change of the
// lowest Ritz value, src/lanczos.cc:232-239) needs nothing else; the O(m^2) QL solve for the residual estimate
// |b_m s_{m-1}| (:231) is only run once that change has stayed below the threshold for more than 15 steps.
double tridiag_smallest(const double *hess, int64_t maxit, int64_t m)
{
    const double *a = hess + maxit, *b = hess;             // b[j] couples j-1 and j (j = 1..m-1)
    double lo = a[0], hi = a[0];
    for (int64_t j = 0; j < m; j++) {
        const double r = (j > 0 ? fabs(b[j]) : 0.0) + (j + 1 < m ? fabs(b[j + 1]) : 0.0);
        lo = fmin(lo, a[j] - r); hi = fmax(hi, a[j] + r);
    }
    auto count_below = [&](double x) {                     // number of eigenvalues < x
        int64_t cnt = 0;
        double q = 1.0;
        for (int64_t j = 0; j < m; j++) {
            const double off2 = j > 0 ? b[j] * b[j] : 0.0;
            q = a[j] - x - (j > 0 ? off2 / q : 0.0);
            if (q == 0.0) q = -DBL_MIN;
            if (q < 0.0) cnt++;
        }
        return cnt;
    };
    hi = fmin(hi, a[0]);                                   // the smallest eigenvalue is <= any diagonal entry
    for (int it = 0; it < 200; it++) {
        const double mid = 0.5 * (lo + hi);
        if (mid <= lo || mid >= hi) break;
        if (count_below(mid) >= 1) hi = mid; else lo = mid;
    }
    return 0.5 * (lo + hi);
}

// ritz ascending ("sr"); s (optional) full vectors; s_last0 (optional) = last component of the lowest vector
int hess_eigen_host(const double *hess, int64_t maxit, int64_t m, double *ritz, double *s, double *s_last0)
{
    std::vector<double> d(m), e(m), z, zl;
    std::vector<int64_t> ord(m);
    for (int64_t j = 0; j < m; j++) { d[j] = hess[maxit + j]; e[j] = (j + 1 < m) ? hess[j + 1] : 0.0; ord[j] = j; }
    if (s) { z.assign((size_t)m * m, 0.0); for (int64_t j = 0; j < m; j++) z[j + j * m] = 1.0; }
    if (s_last0) { zl.assign(m, 0.0); zl[m - 1] = 1.0; }
    if (tridiag_ql(m, d.data(), e.data(), s ? z.data() : nullptr, s_last0 ? zl.data() : nullptr)) return 1;
    for (int64_t i = 1; i < m; i++) { const int64_t k = ord[i]; int64_t j = i - 1; while (j >= 0 && d[ord[j]] > d[k]) { ord[j + 1] = ord[j]; j--; } ord[j + 1] = k; }
    for (int64_t j = 0; j < m; j++) {
        ritz[j] = d[ord[j]];
        if (s) memcpy(s + m * j, z.data() + m * ord[j], sizeof(double) * (size_t)m);
    }
    if (s_last0) *s_last0 = zl[ord[0]];
    return 0;
}

// ------------------------------------------------------------------------------------------------- helpers
struct DevBuf {             // RAII-ish device scratch
    void *p = nullptr;
    int alloc(size_t bytes) { cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1); if (e != cudaSuccess) { (void)cudaGetLastError(); p = nullptr; return fail(QBGPU_ERR_ALLOC, "cudaMalloc failed in a Krylov driver"); } return 0; }
    void release() { if (p) cudaFree(p); p = nullptr; }
    ~DevBuf() { release(); }
};

static int check_single(const qbgpu_matrix *A, bool cplx)
{
    if (!A) return fail(QBGPU_ERR_ARG, "null matrix handle");
    if (A->api_complex != cplx) return fail(QBGPU_ERR_ARG, "handle scalar type does not match this entry point");
    if (A->row_lo != 0 || A->row_hi != A->n) return fail(QBGPU_ERR_STATE, "this loop needs an unsharded handle (use quantum_basis_b200.dist for shards)");
    return QBGPU_OK;
}

// ------------------------------------------------------------------------------------------------ the drivers' boundary
// The loops below run on device vectors in one scalar type and one order; the public drivers reach them through begin() and
// end(), which own every decision about the caller's vectors:
// - host vectors are staged on the device;
// - real mode: through the reference's public API every vector is complex<double> (only model<complex> is instantiated,
//   SURVEY F3), but when the stored values are real (all imaginary parts exactly 0) and the input vectors are real -- which
//   vec_randomize always is (src/miscellaneous.cc:382: imag = 0) -- the whole Krylov recurrence stays real.  The loop then
//   runs on fp64 vectors (half the vector bytes, half the gather sectors) and the results are widened at the end.  Row sums
//   go through the identical fma sequence; (a_m, b_m) agree with the complex run to round-off (only the grouping of the
//   block-level reductions differs).  QBGPU_NO_REAL_MODE forces the complex loop;
// - a handle with an internal order (A->perm, species.cu) multiplies in that order: the caller's vectors are permuted into
//   the loop's on the way in (narrowed in the same pass in real mode) and back on the way out.  (a_m, b_m), E0, the KPM
//   moments and the spectral bounds do not depend on the order; vectors come back in the reference's order.
// Otherwise the loop runs on the caller's (or the staged) vectors themselves, without a copy.
struct Boundary {
    qbgpu_matrix view;          // the handle as the loop sees it when the vectors are converted
    qbgpu_matrix *H = nullptr;  // the loop's handle: the caller's, or `view`
    bool cplx = false;          // scalar type of the loop's vectors
    bool convert = false;       // the loop's vectors are permuted and/or narrowed copies
    char *v[4] = {};            // the loop's vectors, slot by slot
    DevBuf stage[4], work;      // device copies of host vectors (API type, reference order); the converted vectors
};

static int check_where(int where)
{
    return (where == QBGPU_HOST || where == QBGPU_DEVICE) ? QBGPU_OK : fail(QBGPU_ERR_ARG, "where must be QBGPU_HOST or QBGPU_DEVICE");
}

// user[j]: the caller's vector of slot j (nslots <= 4); bit j of `in`: slot j is read by the loop; allow_real: the driver's
// own condition for real mode (every input slot must be real as well)
static int begin(Boundary &B, qbgpu_matrix *A, bool cplx, void *const *user, int nslots, unsigned in, int where, bool allow_real)
{
    Context &c = ctx();
    const int64_t n = A->n;
    const size_t vb = cplx ? 16 : 8;
    const char *src[4] = {};
    for (int j = 0; j < nslots; j++) {
        if (!(in >> j & 1)) continue;
        src[j] = (const char *)user[j];
        if (where == QBGPU_HOST) {
            QB_TRY(B.stage[j].alloc(vb * n));
            QB_CUDA(cudaMemcpyAsync(B.stage[j].p, user[j], vb * n, cudaMemcpyHostToDevice, c.stream));
            src[j] = (const char *)B.stage[j].p;
        }
    }
    bool real = cplx && A->val_real && allow_real && !getenv("QBGPU_NO_REAL_MODE");
    for (int j = 0; real && j < nslots; j++) {
        if (!(in >> j & 1)) continue;
        double h;
        QB_TRY(vec_imag_norm2(n, src[j], c.scal_dev + 56));
        QB_TRY(read_scalars(c.scal_dev + 56, &h, 1));
        real = h == 0.0;
    }
    B.cplx = cplx && !real;
    B.convert = A->perm || real;
    if (!B.convert) {
        B.H = A;
        for (int j = 0; j < nslots; j++) {
            if (where == QBGPU_HOST && !B.stage[j].p) QB_TRY(B.stage[j].alloc(vb * n));
            B.v[j] = where == QBGPU_HOST ? (char *)B.stage[j].p : (char *)user[j];
        }
        return QBGPU_OK;
    }
    B.view = *A;
    B.view.api_complex = B.cplx;
    B.H = &B.view;
    const size_t vl = B.cplx ? 16 : 8;
    QB_TRY(B.work.alloc(vl * n * nslots));
    QB_CUDA(cudaMemsetAsync(B.work.p, 0, vl * n * nslots, c.stream));
    for (int j = 0; j < nslots; j++) {
        B.v[j] = (char *)B.work.p + vl * n * j;
        if (!(in >> j & 1)) continue;
        if (A->perm) QB_TRY(vec_to_native(A, cplx, B.cplx, src[j], B.v[j]));
        else QB_TRY(vec_take_real(n, src[j], (double *)B.v[j]));
    }
    return QBGPU_OK;
}

// bit j of `out`: the loop's vector of slot j goes back to the caller's
static int end(Boundary &B, const qbgpu_matrix *A, bool cplx, void *const *user, int nslots, unsigned out, int where)
{
    Context &c = ctx();
    const int64_t n = A->n;
    const size_t vb = cplx ? 16 : 8;
    DevBuf scratch;
    char *tmp = nullptr;                                    // host callers of converted vectors: one device vector for every output
    if (B.convert && where == QBGPU_HOST) {
        for (DevBuf &s : B.stage) if (s.p) tmp = (char *)s.p;    // (the staged inputs are spent)
        if (!tmp) { QB_TRY(scratch.alloc(vb * n)); tmp = (char *)scratch.p; }
    }
    for (int j = 0; j < nslots; j++) {
        if (!(out >> j & 1)) continue;
        char *dst = B.v[j];
        if (B.convert) {
            dst = where == QBGPU_HOST ? tmp : (char *)user[j];
            if (A->perm) QB_TRY(vec_from_native(A, B.cplx, cplx, B.v[j], dst, make_double2(1.0, 0.0), make_double2(0.0, 0.0)));
            else QB_TRY(vec_put_real(n, (const double *)B.v[j], dst));
        }
        if (where == QBGPU_HOST) QB_CUDA(cudaMemcpyAsync(user[j], dst, vb * n, cudaMemcpyDeviceToHost, c.stream));
    }
    QB_CUDA(cudaStreamSynchronize(c.stream));
    return QBGPU_OK;
}

// ------------------------------------------------------------------------------------------------- lanczos
// state layout: see include/qbgpu.h (lanczos_step_*).
// k > 0 resumes (src/lanczos.cc:144-148, qbasis.h:1044-1061): u[0], u[1] hold the normalised v[k-1], v[k] in their slots, hess
// holds a[0..k-1] and b[0..k].  u[2] = phi0 for val1.  stop_state (optional, in/out) = {cnt_accuE0, accuracy, theta0_prev,
// theta1_prev}: what the reference's checkpoint carries across an interruption (ckpt.cc: lczs_mlns.dat); without it a resumed
// run restarts the stop rule's counters, like the reference's lanczos() called with k > 0 and checkpoints disabled.
static int lanczos_impl(qbgpu_matrix *A, bool cplx, int64_t k, int64_t np, int64_t maxit, int64_t *m_out, char *const *u,
                        double *hess, bool is_val, bool is_val1, bool stop_on_breakdown, double *stop_state)
{
    Context &c = ctx();
    const int64_t n = A->n;
    const int64_t mm = k + np;
    DevBuf dstate, dhess;
    char *Ubuf[2] = {u[0], u[1]};
    char *phi = u[2];
    QB_TRY(dstate.alloc(sizeof(double) * 8));
    QB_TRY(dhess.alloc(sizeof(double) * 2 * maxit));
    double *state = (double *)dstate.p;
    double *b_dev = (double *)dhess.p, *a_dev = b_dev + maxit;
    // state = {scale of ux, scale of uz, b_prev, ...}: both live vectors of a resumed run are normalised and b_prev = b[k]
    const double init[8] = {1.0, k > 0 ? 1.0 : 0.0, k > 0 ? hess[k] : 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    QB_CUDA(cudaMemcpyAsync(state, init, sizeof init, cudaMemcpyHostToDevice, c.stream));
    QB_CUDA(cudaMemsetAsync(dhess.p, 0, sizeof(double) * 2 * maxit, c.stream));
    QB_CUDA(cudaStreamSynchronize(c.stream));              // `init` is on the host stack
    // the caller's array as the reference leaves it: zeros beyond what is known (b[0..k], a[0..k-1] are kept on a resume)
    for (int64_t j = (k > 0 ? k + 1 : 0); j < maxit; j++) hess[j] = 0.0;
    for (int64_t j = maxit + k; j < 2 * maxit; j++) hess[j] = 0.0;

    std::vector<double> ritz(mm + 1);
    int cnt_accuE0 = stop_state ? (int)stop_state[0] : 0;
    double accuracy = stop_state ? stop_state[1] : 0.0;
    double theta0_prev = stop_state ? stop_state[2] : (k > 0 && is_val ? tridiag_smallest(hess, maxit, k) : 0.0);
    bool converged = false;
    int64_t m = k;
    // QBGPU_VERBOSE: per-phase device time of the loop (events around the three passes) and host time of the stop rule
    const bool prof = getenv("QBGPU_VERBOSE") != nullptr;
    EventGuard<4> pg;                                       // (destroyed on every way out of the loop, error returns included)
    double t_a = 0, t_b = 0, t_c = 0, t_host = 0;
    if (prof) for (int i = 0; i < 4; i++) QB_CUDA(pg.create());
    cudaEvent_t *pe = pg.e;
    while (m < mm) {
        m++;
        // one fused Lanczos step (src/lanczos.cc:167-187 for m == 1, :194-214 otherwise)
        const void *ux = Ubuf[(m - 1) % 2];
        void *uz = Ubuf[m % 2];
        if (prof) QB_CUDA(cudaEventRecord(pe[0], c.stream));
        QB_TRY(lanczos_step_a(A, ux, uz, state, true, true));
        if (prof) QB_CUDA(cudaEventRecord(pe[1], c.stream));
        QB_TRY(lanczos_step_b(n, cplx, ux, uz, state));
        if (prof) QB_CUDA(cudaEventRecord(pe[2], c.stream));
        QB_TRY(lanczos_step_c(state, a_dev, b_dev, m));
        if (prof) QB_CUDA(cudaEventRecord(pe[3], c.stream));
        double ab[2];
        QB_CUDA(cudaMemcpyAsync(c.scal_host, a_dev + (m - 1), sizeof(double), cudaMemcpyDeviceToHost, c.stream));
        QB_CUDA(cudaMemcpyAsync(c.scal_host + 1, b_dev + m, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
        QB_CUDA(cudaStreamSynchronize(c.stream));
        ab[0] = c.scal_host[0]; ab[1] = c.scal_host[1];
        hess[maxit + m - 1] = ab[0];
        hess[m] = ab[1];
        if (prof) {
            float f;
            cudaEventElapsedTime(&f, pe[0], pe[1]); t_a += f;
            cudaEventElapsedTime(&f, pe[1], pe[2]); t_b += f;
            cudaEventElapsedTime(&f, pe[2], pe[3]); t_c += f;
        }
        const auto th0 = std::chrono::steady_clock::now();
        struct HostTimer { const std::chrono::steady_clock::time_point t0; double &acc; ~HostTimer() { acc += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); } } host_timer{th0, t_host};
        if (m == 1) continue;                               // the start-up step has no checks in the reference (:167-191)
        if (stop_on_breakdown && fabs(hess[m]) < kLanczosPrecision) break;                         // :216
        if (is_val1) {                                      // re-orthogonalise against phi0, :218-226
            double *dd = c.scal_dev + 52;
            QB_TRY(vec_dotc(n, cplx, phi, uz, dd));
            double h[3];
            QB_TRY(read_scalars(dd, h, 2));
            double sx;
            QB_TRY(read_scalars(state, &sx, 1));
            const double tr = h[0] * sx, ti = cplx ? h[1] * sx : 0.0;
            if (sqrt(tr * tr + ti * ti) > kLanczosPrecision) {
                // v_m = sx*U ;  v_m -= tmp*phi  <=>  U -= (tmp/sx)*phi ;  then renormalise: sx <- 1/||U||
                QB_TRY(vec_axpy(n, cplx, make_double2(-h[0], cplx ? -h[1] : 0.0), phi, uz));
                QB_TRY(vec_nrm2sq(n, cplx, uz, dd));
                double nn;
                QB_TRY(read_scalars(dd, &nn, 1));
                const double nsx = 1.0 / sqrt(nn);
                QB_CUDA(cudaMemcpyAsync(state, &nsx, sizeof(double), cudaMemcpyHostToDevice, c.stream));
                QB_CUDA(cudaStreamSynchronize(c.stream));
            }
        }
        if (is_val) {                                       // stop rule, :228-248
            const double theta0 = tridiag_smallest(hess, maxit, m);
            if (m > 3) {
                const double accu_E0 = fabs((theta0 - theta0_prev) / theta0);
                if (accu_E0 < kLanczosPrecision) cnt_accuE0++; else cnt_accuE0 = 0;
                if (cnt_accuE0 > 15) {                      // only now is the residual estimate |b_m s_{m-1}| needed
                    double s_last = 0.0;
                    if (hess_eigen_host(hess, maxit, m, ritz.data(), nullptr, &s_last)) return fail(QBGPU_ERR_NUMERIC, "hess_eigen: QL did not converge");
                    accuracy = fabs(hess[m] * s_last);
                    if (accuracy < kLanczosPrecision) { converged = true; break; }
                }
            }
            theta0_prev = theta0;
        }
    }
    if (prof) {
        fprintf(stderr, "[qbgpu lanczos] %lld steps, per step: product+epilogue %.3f ms, update pass %.3f ms, scalar kernel %.4f ms, host stop rule %.3f ms (n=%lld, %s vectors)\n",
                (long long)m, t_a / m, t_b / m, t_c / m, t_host / m, (long long)n, cplx ? "complex" : "fp64");
    }
    *m_out = m;
    if (stop_state && is_val && m > k) {
        // what ckpt_lanczos_update would save at this step (src/lanczos.cc:231-248): the residual estimate of step m and,
        // unless the run stopped on the rule (the reference breaks before updating them), this step's Ritz values
        double s_last = 0.0;
        std::vector<double> rz(m + 1);
        if (hess_eigen_host(hess, maxit, m, rz.data(), nullptr, &s_last)) return fail(QBGPU_ERR_NUMERIC, "hess_eigen: QL did not converge");
        stop_state[0] = (double)cnt_accuE0;
        if (m > 3) stop_state[1] = fabs(hess[m] * s_last);
        if (!converged) { stop_state[2] = rz[0]; stop_state[3] = m > 1 ? rz[1] : 0.0; }
        (void)accuracy;
    }
    // hand the two live vectors back normalised, in the reference's slots: v_m at (m%2), v_{m-1} at ((m-1)%2)
    QB_TRY(scale_copy(n, cplx, state + 0, 1.0, Ubuf[m % 2], Ubuf[m % 2]));
    QB_TRY(scale_copy(n, cplx, state + 1, 1.0, Ubuf[(m - 1) % 2], Ubuf[(m - 1) % 2]));
    QB_CUDA(cudaStreamSynchronize(c.stream));
    return QBGPU_OK;
}

static int lanczos(qbgpu_matrix *A, bool cplx, int64_t k, int64_t np, int64_t maxit, int64_t *m_out, void *v,
                   double *hess, const char *purpose, int where, double *stop_state = nullptr)
{
    QB_TRY(ensure_init());
    QB_TRY(check_single(A, cplx));
    if (!m_out || !v || !hess || !purpose) return fail(QBGPU_ERR_ARG, "lanczos: null argument");
    QB_TRY(check_where(where));
    const bool is_val = strstr(purpose, "val") != nullptr;
    const bool is_val1 = strstr(purpose, "val1") != nullptr;
    const bool is_dn = strcmp(purpose, "dnmcs") == 0;
    if (!is_val && !is_dn) return fail(QBGPU_ERR_ARG, "lanczos: purpose must be sr_val0, sr_val1 or dnmcs");
    if (!(k + np < maxit && k >= 0 && np >= 0)) return fail(QBGPU_ERR_ARG, "lanczos: need k >= 0, np >= 0 and k + np < maxit");   // src/lanczos.cc:147
    *m_out = k;
    if (stop_state && is_val && (int)stop_state[0] > 15 && stop_state[1] < kLanczosPrecision) return QBGPU_OK;   // :149 (already converged)
    if (np == 0) return QBGPU_OK;                                                                  // :150
    const size_t vb = cplx ? 16 : 8;
    void *slots[3] = {v, (char *)v + vb * A->n, (char *)v + 2 * vb * A->n};
    const int nvec = is_val1 ? 3 : 2;
    Boundary B;                                             // inputs: v[0]; v[1] of a resumed run; phi0 of val1
    QB_TRY(begin(B, A, cplx, slots, nvec, 0x1u | (k > 0 ? 0x2u : 0u) | (is_val1 ? 0x4u : 0u), where, true));
    QB_TRY(lanczos_impl(B.H, B.cplx, k, np, maxit, m_out, B.v, hess, is_val, is_val1, true, stop_state));
    return end(B, A, cplx, slots, nvec, 0x3u, where);      // the two live vectors, like the reference's slots
}

// --------------------------------------------------------------------------------------------- eigenvec_CG
// The two branches of the reference's loop body (src/lanczos.cc:295-331) on device vectors; sc: 8 device doubles
// [0]=gamma=|r| [1,2]=delta [3]=|pp|^2 [4]=|r_new|^2 [5]=gamma_next [6]=scratch.  Shared by the whole loop (cg_impl) and by the
// step-level entry points qbgpu_cg_restart_* / qbgpu_cg_step_*.
// :297-314  v <- v / rnorm ; r = (E0 - H) v in one pass, |r|^2 from the epilogue ; p = r ; accu = |r| (left in sc[0] as gamma)
static int cg_restart_piece(qbgpu_matrix *A, bool cplx, double2 E0, double rnorm, double *sc, char *dv, char *dr, char *dp, double *accu)
{
    Context &c = ctx();
    const int64_t n = A->n;
    const size_t vb = cplx ? 16 : 8;
    QB_TRY(vec_scal(n, cplx, make_double2(1.0 / rnorm, 0.0), dv));
    FusedArgs fa;
    fa.x = dv; fa.y = dr; fa.alpha = make_double2(-1.0, 0.0); fa.gamma = E0; fa.dots = sc + 1;
    QB_TRY(launch_spmv(A, fa));
    QB_CUDA(cudaMemcpyAsync(dp, dr, vb * n, cudaMemcpyDeviceToDevice, c.stream));   // p = r
    double h[3];
    QB_TRY(read_scalars(sc + 1, h, 3));
    *accu = sqrt(h[2]);
    QB_CUDA(cudaMemcpyAsync(sc, accu, sizeof(double), cudaMemcpyHostToDevice, c.stream));
    QB_CUDA(cudaStreamSynchronize(c.stream));
    return QBGPU_OK;
}
// :320-330  pp = (H - E0 + eps) p ; delta = <p,pp> ; v += alpha p ; r -= alpha pp ; p = r + beta p ; accu = |r_new|
static int cg_iterate_piece(qbgpu_matrix *A, bool cplx, double2 E0, double *sc, char *dv, char *dr, char *dp, char *dpp, double *accu)
{
    Context &c = ctx();
    const int64_t n = A->n;
    FusedArgs fa;
    fa.x = dp; fa.y = dpp; fa.alpha = make_double2(1.0, 0.0);
    fa.gamma = make_double2(DBL_EPSILON - E0.x, -E0.y); fa.dots = sc + 1;
    QB_TRY(launch_spmv(A, fa));
    QB_TRY(cg_update_vr(n, cplx, sc, dv, dr, dp, dpp));          // :324-327
    QB_TRY(cg_update_p(n, cplx, sc, dr, dp));                    // :327-330
    QB_CUDA(cudaMemcpyAsync(sc, sc + 5, sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
    return read_scalars(sc, accu, 1);
}

static int cg_impl(qbgpu_matrix *A, bool cplx, int64_t maxit, int64_t *m_io, double2 E0, double *accu_out,
                   char *dv, char *dr, char *dp, char *dpp)
{
    Context &c = ctx();
    const int64_t n = A->n;
    DevBuf dsc;
    QB_TRY(dsc.alloc(sizeof(double) * 8));
    double *sc = (double *)dsc.p;                           // [0]=gamma [1,2]=delta [3]=|pp|^2 [4]=|r|^2 [5]=gamma_next
    QB_CUDA(cudaMemsetAsync(sc, 0, sizeof(double) * 8, c.stream));

    int64_t m = *m_io;
    double accu = 0.0;                                      // src/lanczos.cc:288-292: 0 at m == 0, |r| on a resume
    if (m > 0) {
        double nn;
        QB_TRY(vec_nrm2sq(n, cplx, dr, sc + 6));
        QB_TRY(read_scalars(sc + 6, &nn, 1));
        accu = sqrt(nn);
        QB_CUDA(cudaMemcpyAsync(sc, &accu, sizeof(double), cudaMemcpyHostToDevice, c.stream));
        QB_CUDA(cudaStreamSynchronize(c.stream));
    }
    while (m < maxit) {
        if (accu < kLanczosPrecision) {                     // :295
            double nn;
            QB_TRY(vec_nrm2sq(n, cplx, dv, sc + 6));
            QB_TRY(read_scalars(sc + 6, &nn, 1));
            const double rnorm = sqrt(nn);
            if (m == 0 || fabs(rnorm - 1.0) > kLanczosPrecision) {       // :297 re-normalise and restart
                QB_TRY(cg_restart_piece(A, cplx, E0, rnorm, sc, dv, dr, dp, &accu));
                m++;
                if (accu < kLanczosPrecision) break;        // :315
            } else {
                break;                                      // :317
            }
        } else {
            QB_TRY(cg_iterate_piece(A, cplx, E0, sc, dv, dr, dp, dpp, &accu));     // :320-330
            m++;
        }
    }
    *m_io = m;
    *accu_out = accu;
    QB_CUDA(cudaStreamSynchronize(c.stream));
    return QBGPU_OK;
}

static int eigenvec_cg(qbgpu_matrix *A, bool cplx, int64_t maxit, int64_t *m_io, double2 E0, double *accu_out,
                       void *v, void *r, void *p, void *pp, int where)
{
    QB_TRY(ensure_init());
    QB_TRY(check_single(A, cplx));
    if (!m_io || !accu_out || !v || !r || !p || !pp) return fail(QBGPU_ERR_ARG, "eigenvec_CG: null argument");
    QB_TRY(check_where(where));
    if (maxit <= 0 || *m_io < 0 || *m_io >= maxit) return fail(QBGPU_ERR_ARG, "eigenvec_CG: need 0 <= m < maxit");        // src/lanczos.cc:287
    const bool resumed = *m_io > 0;                         // a resumed run continues from (v, r, p) of step m
    void *slots[4] = {v, r, p, pp};
    Boundary B;                                             // (a resumed run keeps the API's scalar type)
    QB_TRY(begin(B, A, cplx, slots, 4, resumed ? 0x7u : 0x1u, where, E0.y == 0.0 && !resumed));
    QB_TRY(cg_impl(B.H, B.cplx, maxit, m_io, E0, accu_out, B.v[0], B.v[1], B.v[2], B.v[3]));
    return end(B, A, cplx, slots, 4, 0xfu, where);
}

// -------------------------------------------------------------------------------------------- energy_scale
static int energy_scale(qbgpu_matrix *A, bool cplx, void *v, double *lo, double *hi, double extend, int64_t iters, int where)
{
    QB_TRY(ensure_init());
    QB_TRY(check_single(A, cplx));
    if (!v || !lo || !hi || iters < 3) return fail(QBGPU_ERR_ARG, "energy_scale: bad argument");
    QB_TRY(check_where(where));
    const int64_t n = A->n;
    const size_t vb = cplx ? 16 : 8;
    const int64_t mm = iters - 1;                          // src/kpm.cc:53
    // The reference draws its start vector itself: vec_randomize(dim, seed 1), src/kpm.cc:60.  The draw normalises with a sum
    // in the vector's scalar type, and fp64 and complex sums may round differently.  So on a handle without an internal order
    // it is drawn straight into the loop's vector (fp64 in real mode); on one with, it is drawn in the API's type and the
    // reference's order and then enters the loop's order like any input vector.
    void *slots[2] = {v, (char *)v + vb * n};
    Boundary B;
    DevBuf draw;
    if (A->perm) {
        QB_TRY(draw.alloc(vb * n));
        QB_TRY(vec_randomize(n, cplx, draw.p, 1));
        void *in[2] = {draw.p, nullptr};
        QB_TRY(begin(B, A, cplx, in, 2, 0x1u, QBGPU_DEVICE, true));
    } else {
        QB_TRY(begin(B, A, cplx, slots, 2, 0x0u, where, true));
        QB_TRY(vec_randomize(n, B.cplx, B.v[0], 1));
    }
    std::vector<double> hess(2 * iters, 0.0), ritz(mm);
    int64_t m = 0;
    QB_TRY(lanczos_impl(B.H, B.cplx, 0, mm, iters, &m, B.v, hess.data(), false, false, /*stop_on_breakdown=*/false, nullptr));
    if (hess_eigen_host(hess.data(), iters, mm, ritz.data(), nullptr, nullptr)) return fail(QBGPU_ERR_NUMERIC, "hess_eigen: QL did not converge");
    const double l = ritz[0], h = ritz[mm - 1], slack = extend * (h - l);                          // :83-87
    *lo = l - slack; *hi = h + slack;
    return end(B, A, cplx, slots, 2, 0x3u, where);
}

// --------------------------------------------------------------------------------------------- KPM moments
// mu_k = <phi| T_k(Ht) |phi>, Ht = (H - c)/s.  One fused product per TWO moments:
//   T_{k+1} = 2 Ht T_k - T_{k-1}   (alpha = 2/s, gamma = -2c/s, beta = -1, written over T_{k-1})
//   mu_{2k+1} = 2 <T_k, T_{k+1}> - mu_1 ,  mu_{2k+2} = 2 <T_{k+1}, T_{k+1}> - mu_0
// both inner products come out of the product's epilogue into a device array; the host reads them once at the end.
static int kpm_impl(qbgpu_matrix *A, bool cplx, const void *phi, double lo, double hi, int64_t nmom, double *mu)
{
    Context &c = ctx();
    const int64_t n = A->n;
    const size_t vb = cplx ? 16 : 8;
    const double cc = 0.5 * (hi + lo), ss = 0.5 * (hi - lo);
    DevBuf t, ddots;
    QB_TRY(t.alloc(vb * n * 2));
    char *T[2] = {(char *)t.p, (char *)t.p + vb * n};
    const int64_t nprod = nmom / 2 + 1;                    // products needed to reach index nmom-1
    QB_TRY(ddots.alloc(sizeof(double) * 4 * (nprod + 1)));
    double *dots = (double *)ddots.p;
    QB_CUDA(cudaMemcpyAsync(T[0], phi, vb * n, cudaMemcpyDeviceToDevice, c.stream));
    QB_TRY(vec_nrm2sq(n, cplx, T[0], dots));               // mu_0 = <phi,phi>
    for (int64_t k = 0; k < nprod; k++) {
        FusedArgs fa;
        fa.x = T[k % 2]; fa.y = T[(k + 1) % 2]; fa.dots = dots + 4 * (k + 1);
        if (k == 0) { fa.alpha = make_double2(1.0 / ss, 0.0); fa.gamma = make_double2(-cc / ss, 0.0); }
        else { fa.alpha = make_double2(2.0 / ss, 0.0); fa.gamma = make_double2(-2.0 * cc / ss, 0.0); fa.beta = make_double2(-1.0, 0.0); fa.z = fa.y; }
        QB_TRY(launch_spmv(A, fa));
    }
    std::vector<double> h(4 * (nprod + 1));
    QB_CUDA(cudaMemcpyAsync(h.data(), dots, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, c.stream));
    QB_CUDA(cudaStreamSynchronize(c.stream));
    const double mu0 = h[0];
    const double mu1 = h[4 + 0];                           // <T0,T1>
    for (int64_t j = 0; j < nmom; j++) {
        if (j == 0) mu[j] = mu0;
        else if (j == 1) mu[j] = mu1;
        else if (j % 2 == 0) { const int64_t k = j / 2 - 1; mu[j] = 2.0 * h[4 * (k + 1) + 2] - mu0; }      // 2<T_{k+1},T_{k+1}> - mu0
        else { const int64_t k = (j - 1) / 2; mu[j] = 2.0 * h[4 * (k + 1) + 0] - mu1; }                    // 2<T_k,T_{k+1}> - mu1
    }
    return QBGPU_OK;
}

static int kpm_moments(qbgpu_matrix *A, bool cplx, const void *phi, double lo, double hi, int64_t nmom, double *mu, int where)
{
    QB_TRY(ensure_init());
    QB_TRY(check_single(A, cplx));
    if (!phi || !mu || nmom < 1 || !(hi > lo)) return fail(QBGPU_ERR_ARG, "kpm_moments: bad argument");
    QB_TRY(check_where(where));
    void *slots[1] = {const_cast<void *>(phi)};
    Boundary B;
    QB_TRY(begin(B, A, cplx, slots, 1, 0x1u, where, true));
    return kpm_impl(B.H, B.cplx, B.v[0], lo, hi, nmom, mu);    // (phi is only read)
}

}  // namespace qb

using namespace qb;

extern "C" {

int qbgpu_hess_eigen(const double *hess, int64_t maxit, int64_t m, double *ritz, double *s)
{
    if (!hess || !ritz || m < 1 || m >= maxit) return fail(QBGPU_ERR_ARG, "hess_eigen: need 0 < m < maxit");   // src/lanczos.cc:358
    if (hess_eigen_host(hess, maxit, m, ritz, s, nullptr)) return fail(QBGPU_ERR_NUMERIC, "hess_eigen: QL did not converge");
    return QBGPU_OK;
}

int qbgpu_hess_smallest(const double *hess, int64_t maxit, int64_t m, double *theta0)
{
    if (!hess || !theta0 || m < 1 || m >= maxit) return fail(QBGPU_ERR_ARG, "hess_smallest: need 0 < m < maxit");
    *theta0 = tridiag_smallest(hess, maxit, m);
    return QBGPU_OK;
}

int qbgpu_lanczos_d(qbgpu_matrix_t A, int64_t k, int64_t np, int64_t maxit, int64_t *m, double *v, double *hess, const char *purpose, int where)
{ return lanczos(A, false, k, np, maxit, m, v, hess, purpose, where); }
int qbgpu_lanczos_z(qbgpu_matrix_t A, int64_t k, int64_t np, int64_t maxit, int64_t *m, void *v, double *hess, const char *purpose, int where)
{ return lanczos(A, true, k, np, maxit, m, v, hess, purpose, where); }

int qbgpu_lanczos_resume_d(qbgpu_matrix_t A, int64_t k, int64_t np, int64_t maxit, int64_t *m, double *v, double *hess, const char *purpose, int where, double *stop_state)
{ return lanczos(A, false, k, np, maxit, m, v, hess, purpose, where, stop_state); }
int qbgpu_lanczos_resume_z(qbgpu_matrix_t A, int64_t k, int64_t np, int64_t maxit, int64_t *m, void *v, double *hess, const char *purpose, int where, double *stop_state)
{ return lanczos(A, true, k, np, maxit, m, v, hess, purpose, where, stop_state); }

int qbgpu_eigenvec_cg_d(qbgpu_matrix_t A, int64_t maxit, int64_t *m, double E0, double *accu, double *v, double *r, double *p, double *pp, int where)
{ return eigenvec_cg(A, false, maxit, m, make_double2(E0, 0.0), accu, v, r, p, pp, where); }
int qbgpu_eigenvec_cg_z(qbgpu_matrix_t A, int64_t maxit, int64_t *m, const double E0[2], double *accu, void *v, void *r, void *p, void *pp, int where)
{ if (!E0) return fail(QBGPU_ERR_ARG, "null E0"); return eigenvec_cg(A, true, maxit, m, make_double2(E0[0], E0[1]), accu, v, r, p, pp, where); }

int qbgpu_energy_scale_d(qbgpu_matrix_t A, double *v, double *lo, double *hi, double extend, int64_t iters, int where)
{ return energy_scale(A, false, v, lo, hi, extend, iters, where); }
int qbgpu_energy_scale_z(qbgpu_matrix_t A, void *v, double *lo, double *hi, double extend, int64_t iters, int where)
{ return energy_scale(A, true, v, lo, hi, extend, iters, where); }

int qbgpu_kpm_moments_d(qbgpu_matrix_t A, const double *phi, double lo, double hi, int64_t nmom, double *mu, int where)
{ return kpm_moments(A, false, phi, lo, hi, nmom, mu, where); }
int qbgpu_kpm_moments_z(qbgpu_matrix_t A, const void *phi, double lo, double hi, int64_t nmom, double *mu, int where)
{ return kpm_moments(A, true, phi, lo, hi, nmom, mu, where); }

// ---------------------------------------------------------------- step-level entry points (SURVEY section 8b), DEVICE vectors
// The bodies the loops above are made of, one call per step, for a host that keeps the reference's loop and replaces its body
// (eigenvec_CG: src/lanczos.cc:293-332).  Element type and order of the vectors follow the handle (qbgpu_native_order); no
// real mode, no permutation.
int qbgpu_cg_restart(qbgpu_matrix_t A, const double E0[2], double *sc_dev, void *v, void *r, void *p, double *vnorm, double *accu)
{
    QB_TRY(ensure_init());
    if (!A || !E0 || !sc_dev || !v || !r || !p || !accu) return fail(QBGPU_ERR_ARG, "cg_restart: null argument");
    QB_TRY(check_single(A, A->api_complex));
    double nn = 0.0;
    QB_TRY(vec_nrm2sq(A->n, A->api_complex, v, sc_dev + 6));
    QB_TRY(read_scalars(sc_dev + 6, &nn, 1));
    const double rnorm = sqrt(nn);
    if (vnorm) *vnorm = rnorm;
    if (!(rnorm > 0.0)) return fail(QBGPU_ERR_NUMERIC, "cg_restart: the vector is zero");
    return cg_restart_piece(A, A->api_complex, make_double2(E0[0], A->api_complex ? E0[1] : 0.0), rnorm, sc_dev, (char *)v, (char *)r, (char *)p, accu);
}

int qbgpu_cg_step(qbgpu_matrix_t A, const double E0[2], double *sc_dev, void *v, void *r, void *p, void *pp, double *accu)
{
    QB_TRY(ensure_init());
    if (!A || !E0 || !sc_dev || !v || !r || !p || !pp || !accu) return fail(QBGPU_ERR_ARG, "cg_step: null argument");
    QB_TRY(check_single(A, A->api_complex));
    return cg_iterate_piece(A, A->api_complex, make_double2(E0[0], A->api_complex ? E0[1] : 0.0), sc_dev, (char *)v, (char *)r, (char *)p, (char *)pp, accu);
}

// One step of the Chebyshev recurrence as ONE fused product (the body of kpm_impl): Ht = (H - c)/s, c = (hi+lo)/2, s = (hi-lo)/2;
// first: t_next = Ht t_cur; otherwise t_next = 2 Ht t_cur - t_prev (t_next may alias t_prev).  dots (may be NULL): the local
// rows' <t_cur, t_next> (2 doubles) and |t_next|^2 -- what the 2k / 2k+1 doubling identities need.  Works on shards too
// (t_cur: the full vector; t_prev / t_next: the local rows), like qbgpu_spmv_fused.
int qbgpu_cheb_step(qbgpu_matrix_t A, double lo, double hi, int first, const void *t_cur_full, const void *t_prev_local, void *t_next_local, double *dots_dev)
{
    QB_TRY(ensure_init());
    if (!A || !t_cur_full || !t_next_local || !(hi > lo)) return fail(QBGPU_ERR_ARG, "cheb_step: bad argument");
    if (!first && !t_prev_local) return fail(QBGPU_ERR_ARG, "cheb_step: t_prev is needed after the first step");
    const double cc = 0.5 * (hi + lo), ss = 0.5 * (hi - lo);
    FusedArgs fa;
    fa.x = t_cur_full; fa.y = t_next_local; fa.dots = dots_dev;
    if (first) { fa.alpha = make_double2(1.0 / ss, 0.0); fa.gamma = make_double2(-cc / ss, 0.0); }
    else { fa.alpha = make_double2(2.0 / ss, 0.0); fa.gamma = make_double2(-2.0 * cc / ss, 0.0); fa.beta = make_double2(-1.0, 0.0); fa.z = t_prev_local; }
    return launch_spmv(A, fa);
}

}  // extern "C"
