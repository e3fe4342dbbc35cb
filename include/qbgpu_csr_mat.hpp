// include/qbgpu_csr_mat.hpp -- C++ adaptor over the C ABI with the shape of the reference's csr_mat<T>.
//
// The reference's Krylov routines are templates over a duck-typed matrix `MAT` that only needs
//     void MultMv2(const T *x, T *y) const;   // y = H*x + y      (src/sparse.cc:262-289)
//     void MultMv (const T *x, T *y) const;   // y = H*x          (src/sparse.cc:291-297)
//     std::vector<T> to_dense() const;        //                  (src/sparse.cc:299-315)
// (qbasis.h:1065-1093,1654: lanczos, eigenvec_CG, iram, energy_scale).  qbgpu::csr_mat<T> provides exactly those
// members on top of libqbgpu, so `lanczos<T, qbgpu::csr_mat<T>>` etc. instantiate unchanged, and adds the fused
// device-resident loops as members with the reference's argument lists.  Errors become std::runtime_error like the
// reference's (src/sparse.cc:130,259,288).  Header-only; link with -lqbgpu.
#pragma once
#include <complex>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>
#include "qbgpu.h"

namespace qbgpu {

inline void check(int rc, const char *what)
{
    if (rc != QBGPU_OK) throw std::runtime_error(std::string(what) + " failed: " + qbgpu_last_error());
}

template <typename T> class csr_mat {
    static_assert(std::is_same<T, double>::value || std::is_same<T, std::complex<double>>::value, "T must be double or complex<double>");
    static constexpr bool is_complex = !std::is_same<T, double>::value;
public:
    int64_t dim = 0;
    int64_t nnz = 0;
    bool sym = false;
    qbgpu_matrix_t handle = nullptr;       // replaces `sparse_matrix_t handle` (qbasis.h:985)

    csr_mat() = default;
    // from the reference's arrays (csr_mat<T>::dim, nnz, sym, val, ja, ia; MKL_INT == int64 under -DMKL_ILP64).
    // Upload + conversion happen here, where the reference creates its MKL handle (src/sparse.cc:129,258).
    csr_mat(int64_t dim_, int64_t nnz_, bool sym_, const T *val, const long long *ja, const long long *ia, int flags = 0)
        : dim(dim_), nnz(nnz_), sym(sym_)
    {
        const int64_t *ia64 = reinterpret_cast<const int64_t *>(ia), *ja64 = reinterpret_cast<const int64_t *>(ja);
        if (is_complex) check(qbgpu_create_zcsr(&handle, dim, ia64, ia64 + 1, ja64, val, sym ? 1 : 0, flags), "qbgpu_create_zcsr");
        else check(qbgpu_create_dcsr(&handle, dim, ia64, ia64 + 1, ja64, reinterpret_cast<const double *>(val), sym ? 1 : 0, flags), "qbgpu_create_dcsr");
    }
    // from any object with the reference csr_mat's public members (qbasis.h:976-985)
    template <typename RefCsr> explicit csr_mat(const RefCsr &ref, int flags = 0) : csr_mat(ref.dim, ref.nnz, ref.sym, ref.val, ref.ja, ref.ia, flags) {}
    // adopt a handle produced by one of the on-device assemblers (qbgpu_build_*, qbgpu_sector_build_heisenberg, ...)
    static csr_mat adopt(qbgpu_matrix_t h)
    {
        csr_mat m;
        qbgpu_matrix_info inf;
        check(qbgpu_matrix_get_info(h, &inf), "qbgpu_matrix_get_info");
        m.dim = inf.n; m.nnz = inf.nnz_input; m.sym = true; m.handle = h;
        return m;
    }
    csr_mat(const csr_mat &) = delete;
    csr_mat &operator=(const csr_mat &) = delete;
    csr_mat(csr_mat &&o) noexcept : dim(o.dim), nnz(o.nnz), sym(o.sym), handle(o.handle) { o.handle = nullptr; }
    csr_mat &operator=(csr_mat &&o) noexcept { if (this != &o) { destroy(); dim = o.dim; nnz = o.nnz; sym = o.sym; handle = o.handle; o.handle = nullptr; } return *this; }
    ~csr_mat() { if (handle) qbgpu_destroy(handle); }
    void destroy() { if (handle) { check(qbgpu_destroy(handle), "qbgpu_destroy"); handle = nullptr; } }   // src/sparse.cc:150-169
    int64_t dimension() const { return dim; }

    void MultMv2(const T *x, T *y) const { mv(1.0, x, 1.0, y); }
    void MultMv(const T *x, T *y) const { mv(1.0, x, 0.0, y); }
    std::vector<T> to_dense() const
    {
        std::vector<T> res(static_cast<size_t>(dim) * dim);
        check(qbgpu_to_dense(handle, res.data()), "qbgpu_to_dense");
        return res;
    }

    // fused device-resident loops with the reference's argument lists (host pointers)
    void lanczos(int64_t k, int64_t np, int64_t maxit, int64_t &m, T *v, double *hessenberg, const std::string &purpose) const
    {
        if (is_complex) check(qbgpu_lanczos_z(handle, k, np, maxit, &m, v, hessenberg, purpose.c_str(), QBGPU_HOST), "qbgpu_lanczos_z");
        else check(qbgpu_lanczos_d(handle, k, np, maxit, &m, reinterpret_cast<double *>(v), hessenberg, purpose.c_str(), QBGPU_HOST), "qbgpu_lanczos_d");
    }
    void eigenvec_CG(int64_t maxit, int64_t &m, const T &E0, double &accu, T *v, T *r, T *p, T *pp) const
    {
        if (is_complex) {
            const double e[2] = {std::real(E0), std::imag(E0)};
            check(qbgpu_eigenvec_cg_z(handle, maxit, &m, e, &accu, v, r, p, pp, QBGPU_HOST), "qbgpu_eigenvec_cg_z");
        } else {
            check(qbgpu_eigenvec_cg_d(handle, maxit, &m, std::real(E0), &accu, reinterpret_cast<double *>(v), reinterpret_cast<double *>(r),
                                      reinterpret_cast<double *>(p), reinterpret_cast<double *>(pp), QBGPU_HOST), "qbgpu_eigenvec_cg_d");
        }
    }
    void energy_scale(T *v, double &lo, double &hi, double extend, int64_t iters) const
    {
        if (is_complex) check(qbgpu_energy_scale_z(handle, v, &lo, &hi, extend, iters, QBGPU_HOST), "qbgpu_energy_scale_z");
        else check(qbgpu_energy_scale_d(handle, reinterpret_cast<double *>(v), &lo, &hi, extend, iters, QBGPU_HOST), "qbgpu_energy_scale_d");
    }
    // Chebyshev moments mu_k = <phi|T_k((H - c)/s)|phi>, k < nmom, c = (hi+lo)/2, s = (hi-lo)/2 with (lo, hi) from energy_scale():
    // the recurrence the north star places in kpm.cc (the reference's src/kpm.cc stops at energy_scale); host phi, one fused
    // product per two moments on the device
    std::vector<double> kpm_moments(const T *phi, double lo, double hi, int64_t nmom) const
    {
        std::vector<double> mu(static_cast<size_t>(nmom > 0 ? nmom : 0));
        if (is_complex) check(qbgpu_kpm_moments_z(handle, phi, lo, hi, nmom, mu.data(), QBGPU_HOST), "qbgpu_kpm_moments_z");
        else check(qbgpu_kpm_moments_d(handle, reinterpret_cast<const double *>(phi), lo, hi, nmom, mu.data(), QBGPU_HOST), "qbgpu_kpm_moments_d");
        return mu;
    }
    // iram<T,MAT>(dim, mat, v0, nev, ncv, maxit, "sr" | "lr", nconv, eigenvals, eigenvecs) (src/lanczos.cc:497-603) without the
    // PCIe round trip per product: thick-restart Lanczos with the basis in HBM.  eigenvecs (host, nev * dim entries) may be null.
    void iram_device(int nev, int ncv, int maxit, const std::string &order, int &nconv, double *eigenvals, T *eigenvecs = nullptr) const
    {
        int nprod = 0;
        if (order == "sr") check(qbgpu_trlan(handle, nev, ncv, maxit, 0.0, &nconv, &nprod, eigenvals, eigenvecs, QBGPU_HOST), "qbgpu_trlan");
        else if (order == "lr") check(qbgpu_trlan_largest(handle, nev, ncv, maxit, 0.0, &nconv, &nprod, eigenvals, eigenvecs, QBGPU_HOST), "qbgpu_trlan_largest");
        else throw std::runtime_error("qbgpu::csr_mat::iram_device: order must be \"sr\" or \"lr\"");
    }
    // Step-level members for a host that keeps the reference's loops and replaces their bodies (DEVICE pointers: qbgpu_malloc /
    // qbgpu_memcpy_h2d; sc = 8 device doubles, zeroed before the first call).  cg_restart / cg_step are the two branches of
    // eigenvec_CG's loop body (src/lanczos.cc:297-314 / :320-330); cheb_step is one fused product of T_{k+1} = 2 Ht T_k - T_{k-1}.
    double cg_restart(const T &E0, double *sc_dev, T *v_dev, T *r_dev, T *p_dev, double *vnorm = nullptr) const
    {
        const double e[2] = {std::real(E0), std::imag(E0)};
        double accu = 0.0;
        check(qbgpu_cg_restart(handle, e, sc_dev, v_dev, r_dev, p_dev, vnorm, &accu), "qbgpu_cg_restart");
        return accu;
    }
    double cg_step(const T &E0, double *sc_dev, T *v_dev, T *r_dev, T *p_dev, T *pp_dev) const
    {
        const double e[2] = {std::real(E0), std::imag(E0)};
        double accu = 0.0;
        check(qbgpu_cg_step(handle, e, sc_dev, v_dev, r_dev, p_dev, pp_dev, &accu), "qbgpu_cg_step");
        return accu;
    }
    void cheb_step(double lo, double hi, bool first, const T *t_cur_dev, const T *t_prev_dev, T *t_next_dev, double *dots_dev = nullptr) const
    {
        check(qbgpu_cheb_step(handle, lo, hi, first ? 1 : 0, t_cur_dev, t_prev_dev, t_next_dev, dots_dev), "qbgpu_cheb_step");
    }

private:
    void mv(double alpha, const T *x, double beta, T *y) const
    {
        if (!handle) throw std::runtime_error("qbgpu::csr_mat: matrix-vector product on an empty matrix");
        if (is_complex) {
            const double a[2] = {alpha, 0.0}, b[2] = {beta, 0.0};
            check(qbgpu_zmv(handle, a, x, b, y, QBGPU_HOST), "matrix-vector product");
        } else {
            check(qbgpu_dmv(handle, alpha, reinterpret_cast<const double *>(x), beta, reinterpret_cast<double *>(y), QBGPU_HOST), "matrix-vector product");
        }
    }
};

// One (Sz, momentum) sector of a spin-1/2 model: the device counterpart of model::fill_Weisse_table +
// enumerate_basis_repr + generate_Ham_sparse_repr (src/model.cc:205-249, 275-487, 688-836) with the reference's
// representatives, row order, norms and matrix elements.  A maintainer fills basis_repr / norm_repr from states() /
// norms() and HamMat_csr_repr from heisenberg().
class sector {
public:
    qbgpu_sector_t handle = nullptr;
    qbgpu_sector_info info{};
    sector(const std::vector<int> &L, int ndown, const std::vector<int> &momentum)
    {
        if (L.size() != momentum.size()) throw std::runtime_error("qbgpu::sector: one momentum integer per lattice direction");
        std::vector<int32_t> l(L.begin(), L.end()), k(momentum.begin(), momentum.end());
        check(qbgpu_sector_create(&handle, static_cast<int>(l.size()), l.data(), ndown, k.data()), "qbgpu_sector_create");
        check(qbgpu_sector_get_info(handle, &info), "qbgpu_sector_get_info");
    }
    sector(const sector &) = delete;
    sector &operator=(const sector &) = delete;
    ~sector() { if (handle) qbgpu_sector_destroy(handle); }
    int64_t dim() const { return info.dim; }
    // 32-bit bit patterns (QBGPU_ERR_STATE for the 34- and 36-site sectors, info.state_bits == 64: use states64())
    std::vector<uint32_t> states() const { std::vector<uint32_t> s(info.dim); check(qbgpu_sector_states(handle, s.data()), "qbgpu_sector_states"); return s; }
    std::vector<uint64_t> states64() const { std::vector<uint64_t> s(info.dim); check(qbgpu_sector_states64(handle, s.data()), "qbgpu_sector_states64"); return s; }
    std::vector<double> norms() const { std::vector<double> s(info.dim); check(qbgpu_sector_norms(handle, s.data()), "qbgpu_sector_norms"); return s; }
    // H = J sum_bonds S_i.S_j (bonds = {i0, j0, i1, j1, ...}); fake_pos as in model's constructor (qbasis.h:1337)
    csr_mat<std::complex<double>> heisenberg(const std::vector<int32_t> &bonds, double J = 1.0, double fake_pos = 100.0, int flags = 0) const
    {
        qbgpu_matrix_t h = nullptr;
        check(qbgpu_sector_build_heisenberg(handle, &h, static_cast<int>(bonds.size() / 2), bonds.data(), J, fake_pos, flags), "qbgpu_sector_build_heisenberg");
        return csr_mat<std::complex<double>>::adopt(h);
    }
    // the same operator without stored entries: model<T>::MultMv2 with matrix_free == true, repr branch (src/model.cc:1016-1107).
    // The handle borrows this sector's tables: let it go out of scope before the sector does.
    csr_mat<std::complex<double>> heisenberg_matrix_free(const std::vector<int32_t> &bonds, double J = 1.0, double fake_pos = 100.0) const
    {
        qbgpu_matrix_t h = nullptr;
        check(qbgpu_sector_matfree_heisenberg(handle, &h, static_cast<int>(bonds.size() / 2), bonds.data(), J, fake_pos), "qbgpu_sector_matfree_heisenberg");
        return csr_mat<std::complex<double>>::adopt(h);
    }
};

// One (N_up, N_dn, momentum) sector of single-orbital electrons (the reference's "electron" orbital: two bits per site, bit 0 up,
// bit 1 down; at most 16 sites): fill_Weisse_table + enumerate_basis_repr + generate_Ham_sparse_repr of
// examples/trans_symmetric/latt_square/square_Fermi_Hubbard.cc on the device, fermionic translation signs included.
class electron_sector {
public:
    qbgpu_sector_t handle = nullptr;
    qbgpu_sector_info info{};
    electron_sector(const std::vector<int> &L, int nup, int ndn, const std::vector<int> &momentum)
    {
        if (L.size() != momentum.size()) throw std::runtime_error("qbgpu::electron_sector: one momentum integer per lattice direction");
        std::vector<int32_t> l(L.begin(), L.end()), k(momentum.begin(), momentum.end());
        check(qbgpu_sector_create_electron(&handle, static_cast<int>(l.size()), l.data(), nup, ndn, k.data()), "qbgpu_sector_create_electron");
        check(qbgpu_sector_get_info(handle, &info), "qbgpu_sector_get_info");
    }
    electron_sector(const electron_sector &) = delete;
    electron_sector &operator=(const electron_sector &) = delete;
    ~electron_sector() { if (handle) qbgpu_sector_destroy(handle); }
    int64_t dim() const { return info.dim; }
    std::vector<uint32_t> states() const { std::vector<uint32_t> s(info.dim); check(qbgpu_sector_states(handle, s.data()), "qbgpu_sector_states"); return s; }
    std::vector<double> norms() const { std::vector<double> s(info.dim); check(qbgpu_sector_norms(handle, s.data()), "qbgpu_sector_norms"); return s; }
    // H = -t sum_hops c+_{to,s} c_{from,s} + U sum_i n_up,i n_dn,i ; hops = {to0, from0, spin0, to1, ...} DIRECTED, in add_Ham order
    csr_mat<std::complex<double>> hubbard(const std::vector<int32_t> &hops, double t = 1.0, double U = 1.1, double fake_pos = 100.0, int flags = 0) const
    {
        qbgpu_matrix_t h = nullptr;
        check(qbgpu_sector_build_hubbard(handle, &h, static_cast<int>(hops.size() / 3), hops.data(), t, U, fake_pos, flags), "qbgpu_sector_build_hubbard");
        return csr_mat<std::complex<double>>::adopt(h);
    }
    // model::moprXvec_repr (src/model.cc:1716-1846) for one-site electron operators on device vectors: x_dev (this sector) ->
    // y_dev (target, overwritten), one coefficient per site.  Coefficients e^{+i q.r} move a vector from K to K + q.
    // A = sum_r cu[r] n_up,r + cd[r] n_dn,r (target: same particle numbers)
    void apply_density(const electron_sector &target, const std::vector<std::complex<double>> &cu, const std::vector<std::complex<double>> &cd,
                       const std::complex<double> *x_dev, std::complex<double> *y_dev) const
    {
        coef_size(cu); coef_size(cd);
        check(qbgpu_sector_apply_density(handle, target.handle, reinterpret_cast<const double *>(cu.data()), reinterpret_cast<const double *>(cd.data()),
                                         x_dev, y_dev), "qbgpu_sector_apply_density");
    }
    // A = sum_r c[r] c+_{r,dn} c_{r,up} (lower, S^-) or c+_{r,up} c_{r,dn} (S^+)
    void apply_spin_flip(const electron_sector &target, bool lower, const std::vector<std::complex<double>> &c,
                         const std::complex<double> *x_dev, std::complex<double> *y_dev) const
    {
        coef_size(c);
        check(qbgpu_sector_apply_spin_flip(handle, target.handle, lower ? 1 : 0, reinterpret_cast<const double *>(c.data()), x_dev, y_dev),
              "qbgpu_sector_apply_spin_flip");
    }
    // A = sum_r c[r] c_{r,spin} (create false) or c+_{r,spin}; spin 0 up, 1 down
    void apply_fermion(const electron_sector &target, bool create, int spin, const std::vector<std::complex<double>> &c,
                       const std::complex<double> *x_dev, std::complex<double> *y_dev) const
    {
        coef_size(c);
        check(qbgpu_sector_apply_fermion(handle, target.handle, create ? 1 : 0, spin, reinterpret_cast<const double *>(c.data()), x_dev, y_dev),
              "qbgpu_sector_apply_fermion");
    }

private:
    void coef_size(const std::vector<std::complex<double>> &c) const
    {
        if (static_cast<int>(c.size()) != info.nsites) throw std::runtime_error("qbgpu::electron_sector: one coefficient per site");
    }
};

}  // namespace qbgpu
