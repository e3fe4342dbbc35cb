// quantum_basis_b200/csrc/sectors.cu -- translation-symmetric ("repr") sectors assembled on the device.
//
// SURVEY section 8f rank 1 for BASELINE configs 2 and 5: the reference builds momentum sectors on the host with
// Weisse's sublattice-coding tables (model::fill_Weisse_table src/model.cc:205-249, enumerate_basis_repr :275-487,
// generate_Ham_sparse_repr :688-836; tables from classify_Weisse_tables src/basis.cc:1670-2101) at about two thousand
// rows per second -- hours for the chain L=32.  This file produces the SAME csr_mat (same representatives, same row
// order, same norms, same matrix elements bit for bit) directly in HBM and hands it to the expansion of matrix.cu.
//
// What the reference's tables encode, stated without them (tests/repr_builders.py pins this statement against 39
// sectors assembled by the compiled reference):
//   * sites are numbered with the first even direction fastest (lattice::site2coor_old, src/lattice.cc:591-615), so a
//     parent state is the zip of two half states a (even sites) and b (odd sites) living on the divided lattice
//     (divide_lattice, src/lattice.cc:1076-1115; zipper_basis, src/basis.cc:946-969);
//   * rep[x] / dist[x] of a half state: first state of its sublattice orbit in integer order and the first displacement
//     (lexicographic, last index fastest) that reaches x (classify_trans_full2rep, src/basis.cc:1351-1421);
//   * the representative of a parent orbit: among the orbit's elements whose even half IS the smaller of the two
//     half-representatives, the one whose odd half has the smallest dist; for equal dist the smallest parent
//     displacement i gives the phase exp(2 pi i k.i/L) (the lt/eq/gt tables and the (disp_j, disp_i) minimisation at
//     src/basis.cc:1836-1840, 1897-1901, 1949-1953);
//   * basis order: Lin order (odd label, even label) if J = Ja[ia] + Jb[ib] is solvable, else integer order
//     (src/model.cc:435-443; ALGraph::BSF_set_JaJb, src/miscellaneous.cc:660-708);
//   * nu = orbit size when every stabiliser t has k.t integer, else 0 (norm_trans_repr, src/basis.cc:2104-2202);
//   * rows with nu = 0 hold fake_pos + i/dim on the diagonal only; other elements are
//     sqrt(nu_i/nu_j) * conj(c) * exp(2 pi i k.disp_i/L), accumulated with lil_mat::add's erase rule
//     (src/sparse.cc:57-81) in the term order of mopr::operator+= (src/operators.cc:901-925: sorted by site pair).
//
// Every parent translation acts on the two halves through sublattice translations (possibly exchanging them), so a
// translated state costs two lookups in a [sublattice translations] x [2^(N/2)] table that lives in L2.
#include "internal.hpp"
#include <cub/device/device_scan.cuh>
#include <cub/device/device_reduce.cuh>
#include <thrust/iterator/transform_iterator.h>
#include <thrust/iterator/counting_iterator.h>
#include <chrono>
#include <cub/device/device_select.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <algorithm>
#include <complex>
#include <cstring>
#include <map>
#include <vector>

namespace qb {

constexpr int kSBlock = 128;
constexpr int kMaxTrans = 32;          // one site per cell, at most 32 sites
constexpr int kMaxTerms = 128;         // bond terms per Hamiltonian

struct SecDev {                        // passed to kernels by value
    int nsites, nsub, ntrans, shift, lin_order;
    int64_t n;
    const uint16_t *subT;              // [nsubtrans << nsub]  subT[(j << nsub) + x] = S_j x
    const uint16_t *rep;               // [1 << nsub]
    const uint8_t  *dist;              // [1 << nsub]
    const uint32_t *keys;              // [n] ascending; Lin key (b << nsub | a) or the zipped bit pattern
    const uint32_t *seg;               // [(1 << (2 nsub - shift)) + 1] first index with key >> shift >= h
    const double   *nu;                // [n]
    uint8_t fwd_swap[kMaxTrans], fwd_ja[kMaxTrans], fwd_jb[kMaxTrans];   // T_i (a,b)
    uint8_t inv_swap[kMaxTrans], inv_ja[kMaxTrans], inv_jb[kMaxTrans];   // T_i^{-1} (a,b)
    uint8_t bad[kMaxTrans];            // k.t not an integer: a stabiliser t kills the norm
    // single-orbital electrons (two bits per site: bit 0 up, bit 1 down; nsub then counts the BITS of a half state):
    int electron;
    int16_t kt[kMaxTrans];             // k.t in units of 1/N
    const uint16_t *invmask;           // [ntrans][16]  invmask[i*16 + s1] = sites s2 > s1 that translation i moves in front of s1
};

__host__ __device__ __forceinline__ uint32_t spread_bits(uint32_t x)
{
    x &= 0xFFFFu;
    x = (x | (x << 8)) & 0x00FF00FFu;
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x;
}
__host__ __device__ __forceinline__ uint32_t squeeze_bits(uint32_t x)
{
    x &= 0x55555555u;
    x = (x | (x >> 1)) & 0x33333333u;
    x = (x | (x >> 2)) & 0x0F0F0F0Fu;
    x = (x | (x >> 4)) & 0x00FF00FFu;
    x = (x | (x >> 8)) & 0x0000FFFFu;
    return x;
}

// two-bit digits: half digit t -> parent digit 2t (even half) / 2t+1 (odd half)
__host__ __device__ __forceinline__ uint32_t spread_digits(uint32_t x)
{
    x &= 0xFFFFu;
    x = (x | (x << 8)) & 0x00FF00FFu;
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    return x;
}
__host__ __device__ __forceinline__ uint32_t squeeze_digits(uint32_t x)
{
    x &= 0x33333333u;
    x = (x | (x >> 2)) & 0x0F0F0F0Fu;
    x = (x | (x >> 4)) & 0x00FF00FFu;
    x = (x | (x >> 8)) & 0x0000FFFFu;
    return x;
}
template <class SD> __device__ __forceinline__ uint32_t sec_zip(const SD &S, uint32_t a, uint32_t b)
{ return S.electron ? (spread_digits(a) | (spread_digits(b) << 2)) : (spread_bits(a) | (spread_bits(b) << 1)); }
template <class SD> __device__ __forceinline__ void sec_unzip(const SD &S, uint32_t st, uint32_t &a, uint32_t &b)
{
    if (S.electron) { a = squeeze_digits(st); b = squeeze_digits(st >> 2); }
    else { a = squeeze_bits(st); b = squeeze_bits(st >> 1); }
}

__device__ __forceinline__ void sec_move(const SecDev &S, int swap, int ja, int jb, uint32_t a, uint32_t b, uint32_t &ao, uint32_t &bo)
{
    const uint16_t *Ta = S.subT + ((size_t)ja << S.nsub), *Tb = S.subT + ((size_t)jb << S.nsub);
    if (swap) { ao = Ta[b]; bo = Tb[a]; } else { ao = Ta[a]; bo = Tb[b]; }
}

// (a, b) -> representative halves (ca, cb) and the smallest displacement i with state = T_i (ca zip cb)
__device__ __forceinline__ int sec_canon(const SecDev &S, uint32_t a, uint32_t b, uint32_t &ca, uint32_t &cb)
{
    const uint32_t rs = min((uint32_t)S.rep[a], (uint32_t)S.rep[b]);
    int best = 0x7fffffff, bi = -1;
    for (int i = 0; i < S.ntrans; i++) {
        uint32_t ai, bb;
        sec_move(S, S.inv_swap[i], S.inv_ja[i], S.inv_jb[i], a, b, ai, bb);
        if (ai != rs) continue;
        const int key = (int)S.dist[bb] * kMaxTrans + i;
        if (key < best) { best = key; bi = i; ca = ai; cb = bb; }
    }
    return bi;
}

__device__ __forceinline__ uint32_t sec_key(const SecDev &S, uint32_t a, uint32_t b)
{
    return S.lin_order ? ((b << S.nsub) | a) : sec_zip(S, a, b);
}
__device__ __forceinline__ void sec_halves(const SecDev &S, uint32_t key, uint32_t &a, uint32_t &b)
{
    if (S.lin_order) { a = key & ((1u << S.nsub) - 1u); b = key >> S.nsub; }
    else sec_unzip(S, key, a, b);
}
__device__ __forceinline__ int64_t sec_lookup(const SecDev &S, uint32_t key)
{
    const uint32_t h = key >> S.shift;
    uint32_t lo = S.seg[h], hi = S.seg[h + 1];
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; const uint32_t v = S.keys[mid]; if (v < key) lo = mid + 1; else hi = mid; }
    return (lo < S.seg[h + 1] && S.keys[lo] == key) ? (int64_t)lo : -1;
}

// ------------------------------------------------------------------------------------------ enumeration
// candidate c = bIdx * nreps + r  <->  (a = reps[r], b = bIdx); ascending c is Lin order
__global__ void __launch_bounds__(kSBlock) sec_flag_kernel(SecDev S, const uint16_t *__restrict__ reps, int nreps, int ndown, int64_t ncand,
                                                           uint8_t *flag)
{
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncand; c += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t b = (uint32_t)(c / nreps), a = reps[c % nreps];
        uint8_t ok = 0;
        if (__popc(a) + __popc(b) == ndown && a <= S.rep[b]) {
            ok = 1;
            const int db = S.dist[b];
            for (int i = 0; i < S.ntrans; i++) {
                uint32_t ai, bb;
                sec_move(S, S.inv_swap[i], S.inv_ja[i], S.inv_jb[i], a, b, ai, bb);
                if (ai == a && (int)S.dist[bb] < db) { ok = 0; break; }
            }
        }
        flag[c] = ok;
    }
}

__global__ void __launch_bounds__(kSBlock) sec_cand_to_key_kernel(int64_t n, const uint16_t *__restrict__ reps, int nreps, int nsub, uint32_t *keys)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t c = keys[i];
        keys[i] = ((c / nreps) << nsub) | reps[c % nreps];
    }
}

__global__ void __launch_bounds__(kSBlock) sec_lin_to_zip_kernel(int64_t n, int nsub, uint32_t *keys)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t k = keys[i];
        keys[i] = spread_bits(k & ((1u << nsub) - 1u)) | (spread_bits(k >> nsub) << 1);
    }
}

__global__ void __launch_bounds__(kSBlock) sec_seg_kernel(int64_t n, const uint32_t *__restrict__ keys, int shift, uint32_t nseg, uint32_t *seg)
{
    for (uint32_t h = blockIdx.x * blockDim.x + threadIdx.x; h <= nseg; h += gridDim.x * blockDim.x) {
        const uint64_t target = (uint64_t)h << shift;
        int64_t lo = 0, hi = n;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if ((uint64_t)keys[mid] < target) lo = mid + 1; else hi = mid; }
        seg[h] = (uint32_t)lo;
    }
}

__global__ void __launch_bounds__(kSBlock) sec_norm_kernel(SecDev S, double *nu, unsigned long long *zero_count)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S.n; r += (int64_t)gridDim.x * blockDim.x) {
        uint32_t a, b;
        sec_halves(S, S.keys[r], a, b);
        int cnt = 0, bad = 0;
        for (int i = 0; i < S.ntrans; i++) {
            uint32_t ai, bb;
            sec_move(S, S.fwd_swap[i], S.fwd_ja[i], S.fwd_jb[i], a, b, ai, bb);
            if (ai == a && bb == b) { cnt++; bad |= S.bad[i]; }
        }
        const double v = bad ? 0.0 : (double)(S.ntrans / cnt);
        nu[r] = v;
        if (bad) atomicAdd(zero_count, 1ull);
    }
}

__global__ void __launch_bounds__(kSBlock) sec_states_kernel(SecDev S, uint32_t *out)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S.n; r += (int64_t)gridDim.x * blockDim.x) {
        uint32_t a, b;
        sec_halves(S, S.keys[r], a, b);
        out[r] = sec_zip(S, a, b);
    }
}

// ------------------------------------------------------------------------------------------ single-orbital electrons
// The Weisse tables compare bit patterns, so representatives, distances and the basis order are found exactly as for spins
// (two bits per site instead of one); what fermions add (tests/repr_builders_fermion.py pins this against the compiled reference):
//   * a translation permutes the singly occupied sites and picks up the parity of that permutation
//     (mbasis_elem::transform, src/basis.cc:593-620);
//   * norm_trans_repr (src/basis.cc:2134-2147): a stabiliser t needs k.t + sgn_t/2 integer;
//   * generate_Ham_sparse_repr (src/model.cc:815-820): the element carries (-1)^sgn of the translation that maps the
//     representative onto the state the hopping term produced.
__device__ __forceinline__ int el_trans_sign(const SecDev &S, uint32_t st, int i)
{
    const uint32_t m = squeeze_bits(st ^ (st >> 1));                    // singly occupied sites
    int sg = 0;
    for (uint32_t r = m; r; r &= r - 1) sg += __popc(m & S.invmask[i * 16 + (__ffs(r) - 1)]);
    return sg & 1;
}

__global__ void __launch_bounds__(kSBlock) el_flag_kernel(SecDev S, const uint16_t *__restrict__ reps, int nreps, int nup, int ndn, int64_t ncand,
                                                          uint8_t *flag)
{
    const uint32_t MU = 0x5555u;
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < ncand; c += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t b = (uint32_t)(c / nreps), a = reps[c % nreps];
        uint8_t ok = 0;
        if (__popc(a & MU) + __popc(b & MU) == nup && __popc((a >> 1) & MU) + __popc((b >> 1) & MU) == ndn && a <= S.rep[b]) {
            ok = 1;
            const int db = S.dist[b];
            for (int i = 0; i < S.ntrans; i++) {
                uint32_t ai, bb;
                sec_move(S, S.inv_swap[i], S.inv_ja[i], S.inv_jb[i], a, b, ai, bb);
                if (ai == a && (int)S.dist[bb] < db) { ok = 0; break; }
            }
        }
        flag[c] = ok;
    }
}

__global__ void __launch_bounds__(kSBlock) el_lin_to_zip_kernel(int64_t n, int nsub, uint32_t *keys)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t k = keys[i];
        keys[i] = spread_digits(k & ((1u << nsub) - 1u)) | (spread_digits(k >> nsub) << 2);
    }
}

__global__ void __launch_bounds__(kSBlock) el_norm_kernel(SecDev S, double *nu, unsigned long long *zero_count)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S.n; r += (int64_t)gridDim.x * blockDim.x) {
        uint32_t a, b;
        sec_halves(S, S.keys[r], a, b);
        const uint32_t st = sec_zip(S, a, b);
        int cnt = 0, bad = 0;
        for (int i = 0; i < S.ntrans; i++) {
            uint32_t ai, bb;
            sec_move(S, S.fwd_swap[i], S.fwd_ja[i], S.fwd_jb[i], a, b, ai, bb);
            if (ai == a && bb == b) {
                cnt++;
                if (((int)S.kt[i] + el_trans_sign(S, st, i) * (S.nsites / 2)) % S.nsites != 0) bad = 1;
            }
        }
        const double v = bad ? 0.0 : (double)(S.ntrans / cnt);
        nu[r] = v;
        if (bad) atomicAdd(zero_count, 1ull);
    }
}

constexpr int kMaxHops = 256;
struct ElTerms {
    int nterms;
    double t, U, fake_pos;
    uint8_t to[kMaxHops], from[kMaxHops], sp[kMaxHops];      // directed hops c+_{to,sp} c_{from,sp} in the order of mopr::operator+=
};

__device__ __forceinline__ bool el_hop(uint32_t st, int to, int from, int sp, uint32_t &s2, int &sg)
{
    const uint32_t bf = 1u << (2 * from + sp), bt = 1u << (2 * to + sp);
    if (!(st & bf) || (st & bt)) return false;
    sg = __popc(st & ((1u << (2 * from)) - 1u)) & 1;                   // oprXphi's sign rule, src/basis.cc:2717-2731
    if (sp) sg ^= (st >> (2 * from)) & 1u;
    const uint32_t s1 = st ^ bf;
    sg ^= __popc(s1 & ((1u << (2 * to)) - 1u)) & 1;
    if (sp) sg ^= (s1 >> (2 * to)) & 1u;
    s2 = s1 ^ bt;
    return true;
}

// upper bound of the stored row length: the diagonal plus one entry per applicable hop
__global__ void __launch_bounds__(kSBlock) el_cap_kernel(SecDev S, const ElTerms *Tp, int64_t *cap)
{
    __shared__ ElTerms T;
    for (int i = threadIdx.x; i < (int)(sizeof(ElTerms) / 4); i += blockDim.x) ((int *)&T)[i] = ((const int *)Tp)[i];
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= S.n; r += (int64_t)gridDim.x * blockDim.x) {
        int c = 0;
        if (r < S.n) {
            c = 1;
            if (S.nu[r] != 0.0) {
                uint32_t a, b;
                sec_halves(S, S.keys[r], a, b);
                const uint32_t st = sec_zip(S, a, b);
                for (int t = 0; t < T.nterms; t++) {
                    const uint32_t bf = 1u << (2 * T.from[t] + T.sp[t]), bt = 1u << (2 * T.to[t] + T.sp[t]);
                    c += ((st & bf) && !(st & bt)) ? 1 : 0;
                }
            }
        }
        cap[r] = c;
    }
}

// generate_Ham_sparse_repr (src/model.cc:688-836) for H = -t sum c+c + U sum n_up n_dn, upper triangle, lil_mat::add's rule
__global__ void __launch_bounds__(kSBlock) el_rows_kernel(SecDev S, const ElTerms *Tp, const double2 *__restrict__ phase,
                                                          const int64_t *__restrict__ start, int64_t *row_end, int64_t *ocol, double2 *oval)
{
    __shared__ ElTerms T;
    for (int i = threadIdx.x; i < (int)(sizeof(ElTerms) / 4); i += blockDim.x) ((int *)&T)[i] = ((const int *)Tp)[i];
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S.n; r += (int64_t)gridDim.x * blockDim.x) {
        int64_t *col = ocol + start[r];
        double2 *val = oval + start[r];
        const double nu_i = S.nu[r];
        if (nu_i == 0.0) {                                             // src/model.cc:737-740
            col[0] = r; val[0] = make_double2(__dadd_rn(T.fake_pos, __ddiv_rn((double)r, (double)S.n)), 0.0);
            row_end[r] = start[r] + 1;
            continue;
        }
        uint32_t a, b;
        sec_halves(S, S.keys[r], a, b);
        const uint32_t st = sec_zip(S, a, b);
        const int ndbl = __popc(st & (st >> 1) & 0x55555555u);
        double dg = 0.0;
        for (int q = 0; q < ndbl; q++) dg = __dadd_rn(dg, T.U);
        int len = 1;
        col[0] = r; val[0] = make_double2(dg, 0.0);
        for (int t = 0; t < T.nterms; t++) {
            uint32_t s2;
            int sg;
            if (!el_hop(st, T.to[t], T.from[t], T.sp[t], s2, sg)) continue;
            uint32_t a2, b2, ca = 0, cb = 0;
            sec_unzip(S, s2, a2, b2);
            const int i = sec_canon(S, a2, b2, ca, cb);
            if (i < 0) continue;
            const int64_t j = sec_lookup(S, sec_key(S, ca, cb));
            if (j < r) continue;                                       // upper triangle (and j = -1: not in the sector)
            const double nu_j = S.nu[j];
            if (nu_j == 0.0) continue;
            const double amp = sg ? T.t : -T.t;                        // (-t) * (-1)^sg
            const double x = __dmul_rn(__dsqrt_rn(__ddiv_rn(nu_i, nu_j)), amp);
            const double2 ph = phase[i];
            double re = __dmul_rn(x, ph.x), im = __dmul_rn(x, ph.y);
            if (el_trans_sign(S, sec_zip(S, ca, cb), i)) { re = -re; im = -im; }      // src/model.cc:815-820
            int e = 0;
            while (e < len && col[e] != j) e++;
            if (e < len) {                                             // lil_mat::add, src/sparse.cc:57-81
                val[e].x = __dadd_rn(val[e].x, re); val[e].y = __dadd_rn(val[e].y, im);
                if (j != r && hypot(val[e].x, val[e].y) < 1e-14) { len--; col[e] = col[len]; val[e] = val[len]; }
            } else { col[len] = j; val[len] = make_double2(re, im); len++; }
        }
        for (int x1 = 1; x1 < len; x1++) {                             // ascending columns
            const int64_t c = col[x1]; const double2 v = val[x1];
            int y1 = x1 - 1;
            while (y1 >= 0 && col[y1] > c) { col[y1 + 1] = col[y1]; val[y1 + 1] = val[y1]; y1--; }
            col[y1 + 1] = c; val[y1 + 1] = v;
        }
        row_end[r] = start[r] + len;
    }
}

// ------------------------------------------------------------------------------------------ Hamiltonian rows
struct SecTerms {
    int nterms;
    double J, fake_pos;
    uint8_t p[kMaxTerms], q[kMaxTerms];          // site pairs sorted by (lower, higher) -- the order of mopr::operator+=
};

// upper bound of the stored row length: the diagonal plus one entry per antiparallel bond
__global__ void __launch_bounds__(kSBlock) sec_cap_kernel(SecDev S, const SecTerms *Tp, int64_t *cap)
{
    __shared__ SecTerms T;
    for (int i = threadIdx.x; i < (int)(sizeof(SecTerms) / 4); i += blockDim.x) ((int *)&T)[i] = ((const int *)Tp)[i];
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= S.n; r += (int64_t)gridDim.x * blockDim.x) {
        int c = 0;
        if (r < S.n) {
            c = 1;
            if (S.nu[r] != 0.0) {
                uint32_t a, b;
                sec_halves(S, S.keys[r], a, b);
                const uint32_t s = spread_bits(a) | (spread_bits(b) << 1);
                for (int t = 0; t < T.nterms; t++) c += (((s >> T.p[t]) ^ (s >> T.q[t])) & 1u);
            }
        }
        cap[r] = c;
    }
}

__global__ void __launch_bounds__(kSBlock) sec_rows_kernel(SecDev S, const SecTerms *Tp, const double2 *__restrict__ phase,
                                                           const int64_t *__restrict__ start, int64_t *row_end, int64_t *ocol, double2 *oval)
{
    __shared__ SecTerms T;
    for (int i = threadIdx.x; i < (int)(sizeof(SecTerms) / 4); i += blockDim.x) ((int *)&T)[i] = ((const int *)Tp)[i];
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S.n; r += (int64_t)gridDim.x * blockDim.x) {
        int64_t *col = ocol + start[r];
        double2 *val = oval + start[r];
        const double nu_i = S.nu[r];
        if (nu_i == 0.0) {                                             // src/model.cc:737-740
            col[0] = r; val[0] = make_double2(__dadd_rn(T.fake_pos, __ddiv_rn((double)r, (double)S.n)), 0.0);
            row_end[r] = start[r] + 1;
            continue;
        }
        uint32_t a, b;
        sec_halves(S, S.keys[r], a, b);
        const uint32_t s = spread_bits(a) | (spread_bits(b) << 1);
        double dg = 0.0;
        for (int t = 0; t < T.nterms; t++)
            dg = __dadd_rn(dg, (((s >> T.p[t]) ^ (s >> T.q[t])) & 1u) ? -0.25 * T.J : 0.25 * T.J);
        int len = 1;
        col[0] = r; val[0] = make_double2(dg, 0.0);
        for (int t = 0; t < T.nterms; t++) {
            if (!(((s >> T.p[t]) ^ (s >> T.q[t])) & 1u)) continue;
            const uint32_t s2 = s ^ ((1u << T.p[t]) | (1u << T.q[t]));
            uint32_t ca = 0, cb = 0;
            const int i = sec_canon(S, squeeze_bits(s2), squeeze_bits(s2 >> 1), ca, cb);
            if (i < 0) continue;
            const int64_t j = sec_lookup(S, sec_key(S, ca, cb));
            if (j < r) continue;                                       // upper triangle (and j = -1: not in the sector)
            const double nu_j = S.nu[j];
            if (nu_j == 0.0) continue;
            const double x = __dmul_rn(__dsqrt_rn(__ddiv_rn(nu_i, nu_j)), 0.5 * T.J);
            const double2 ph = phase[i];
            const double re = __dmul_rn(x, ph.x), im = __dmul_rn(x, ph.y);
            int e = 0;
            while (e < len && col[e] != j) e++;
            if (e < len) {                                             // lil_mat::add, src/sparse.cc:57-81
                val[e].x = __dadd_rn(val[e].x, re); val[e].y = __dadd_rn(val[e].y, im);
                if (j != r && hypot(val[e].x, val[e].y) < 1e-14) { len--; col[e] = col[len]; val[e] = val[len]; }
            } else { col[len] = j; val[len] = make_double2(re, im); len++; }
        }
        for (int x1 = 1; x1 < len; x1++) {                             // ascending columns
            const int64_t c = col[x1]; const double2 v = val[x1];
            int y1 = x1 - 1;
            while (y1 >= 0 && col[y1] > c) { col[y1 + 1] = col[y1]; val[y1 + 1] = val[y1]; y1--; }
            col[y1 + 1] = c; val[y1 + 1] = v;
        }
        row_end[r] = start[r] + len;
    }
}

// Matrix-free product over the sector: model<T>::MultMv2, repr branch (src/model.cc:1016-1107).  Row i is regenerated from the
// bond list exactly as sec_rows_kernel stores it, but as the FULL row seen from i (the reference does the same: every term, no
// upper-triangle filter, y[i] += x[j] * sqrt(nu_i/nu_j) * conj(c) * exp(2 pi i k.disp_i/L)), and consumed at once.  Zero-norm rows
// carry fake_pos + i/dim on the diagonal (:1022-1025).  Nothing is stored: the sector's tables (keys, norms, sublattice tables)
// are all that lives in HBM -- the reference's own answer to dimensions whose csr_mat does not fit.
template <bool DOTS>
__global__ void __launch_bounds__(kSBlock) sec_matfree_spmv_kernel(SecDev S, const SecTerms *Tp, const double2 *__restrict__ phase,
                                                                   const double2 *__restrict__ x, const double2 *z, double2 *y,
                                                                   double2 alpha, double2 gamma, double2 beta, int scal_mode,
                                                                   const double *__restrict__ sc, double *dots_out, double *partials, unsigned *ticket)
{
    using VT = VecTraits<double2>;
    __shared__ SecTerms T;
    for (int i = threadIdx.x; i < (int)(sizeof(SecTerms) / 4); i += blockDim.x) ((int *)&T)[i] = ((const int *)Tp)[i];
    __syncthreads();
    double dot_scale = 1.0;
    if (scal_mode != 0) {                                              // the fused Lanczos step (internal.hpp: FusedArgs)
        const double sx = sc[0], sz = sc[1], bprev = sc[2];
        alpha = make_double2(sx, 0.0);
        gamma = make_double2(0.0, 0.0);
        beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
        dot_scale = sx;
    }
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    double d[3] = {0.0, 0.0, 0.0};
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S.n; r += (int64_t)gridDim.x * blockDim.x) {
        const double nu_i = S.nu[r];
        const double2 xi = x[r];
        double2 acc = VT::zero();
        if (nu_i == 0.0) {
            mac(acc, __dadd_rn(T.fake_pos, __ddiv_rn((double)r, (double)S.n)), xi);
        } else {
            uint32_t a, b;
            sec_halves(S, S.keys[r], a, b);
            const uint32_t s = spread_bits(a) | (spread_bits(b) << 1);
            double dg = 0.0;
            for (int t = 0; t < T.nterms; t++)
                dg = __dadd_rn(dg, (((s >> T.p[t]) ^ (s >> T.q[t])) & 1u) ? -0.25 * T.J : 0.25 * T.J);
            mac(acc, dg, xi);
            for (int t = 0; t < T.nterms; t++) {
                if (!(((s >> T.p[t]) ^ (s >> T.q[t])) & 1u)) continue;
                const uint32_t s2 = s ^ ((1u << T.p[t]) | (1u << T.q[t]));
                uint32_t ca = 0, cb = 0;
                const int i = sec_canon(S, squeeze_bits(s2), squeeze_bits(s2 >> 1), ca, cb);
                if (i < 0) continue;
                const int64_t j = sec_lookup(S, sec_key(S, ca, cb));
                if (j < 0) continue;                                   // not in the sector
                const double nu_j = S.nu[j];
                if (nu_j == 0.0) continue;
                const double w = __dmul_rn(__dsqrt_rn(__ddiv_rn(nu_i, nu_j)), 0.5 * T.J);
                const double2 ph = phase[i];
                mac(acc, make_double2(__dmul_rn(w, ph.x), __dmul_rn(w, ph.y)), x[j]);
            }
        }
        double2 out = VT::scale(alpha, acc);
        if (gamma.x != 0.0 || gamma.y != 0.0) out = VT::add(out, VT::scale(gamma, xi));
        if (use_beta) out = VT::add(out, VT::scale(beta, z[r]));
        y[r] = out;
        if (DOTS) {
            const double2 p = VT::conj_mul(xi, out);
            d[0] += p.x; d[1] += p.y; d[2] += VT::abs2(out);
        }
    }
    if (DOTS) {
        d[0] *= dot_scale; d[1] *= dot_scale;
        block_reduce_finalize<3, kSBlock>(d, partials, ticket, dots_out);
    }
}

__global__ void __launch_bounds__(kSBlock) sec_len_kernel(int64_t n, const int64_t *start, const int64_t *end, int64_t *len)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) len[r] = end[r] - start[r];
}

// model::moprXvec_repr (src/model.cc:1716-1846) for an operator made of diagonal one-site terms, A = sum_r c_r S^z_r
// (S^z_q when c_r = exp(-i q.r)/sqrt(N)): only the momentum changes, the representative keeps its row index, and
//   y[j] = sum_r  sqrt(nu_old[j] / nu_new[j]) * x[j] * (c_r * <state_j| S^z_r |state_j>)          (:1758-1761)
// with rows skipped when |x[j]|, nu_old[j] or nu_new[j] is below lanczos_precision (:1752, :1760).
__global__ void __launch_bounds__(kSBlock) sec_apply_sz_kernel(SecDev S, const double *__restrict__ nu_new, const double2 *__restrict__ coef,
                                                               const double2 *__restrict__ x, double2 *y)
{
    __shared__ double2 c[kMaxTrans];
    if (threadIdx.x < S.nsites) c[threadIdx.x] = coef[threadIdx.x];
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S.n; r += (int64_t)gridDim.x * blockDim.x) {
        const double2 xj = x[r];
        const double nj = S.nu[r], ni = nu_new[r];
        double2 acc = make_double2(0.0, 0.0);
        if (hypot(xj.x, xj.y) >= 2e-12 && fabs(nj) >= 2e-12 && fabs(ni) > 2e-12) {
            uint32_t a, b;
            sec_halves(S, S.keys[r], a, b);
            const uint32_t st = spread_bits(a) | (spread_bits(b) << 1);
            const double w = __dsqrt_rn(__ddiv_rn(nj, ni));
            const double2 t = make_double2(__dmul_rn(w, xj.x), __dmul_rn(w, xj.y));
            for (int site = 0; site < S.nsites; site++) {
                const double sz = ((st >> site) & 1u) ? -0.5 : 0.5;
                const double2 d = make_double2(__dmul_rn(c[site].x, sz), __dmul_rn(c[site].y, sz));
                acc.x = __dadd_rn(acc.x, __dsub_rn(__dmul_rn(t.x, d.x), __dmul_rn(t.y, d.y)));
                acc.y = __dadd_rn(acc.y, __dadd_rn(__dmul_rn(t.x, d.y), __dmul_rn(t.y, d.x)));
            }
        }
        y[r] = acc;
    }
}

// model::moprXvec_repr (src/model.cc:1762-1834), off-diagonal branch, for the spin-1/2 ladder operators
// A = sum_r c_r S^-_r (lower = 1: acts on up spins, the target sector has one more down spin) or sum_r c_r S^+_r
// (lower = 0).  Every term flips one spin of the OLD representative; the produced state is brought to its representative
// in the NEW sector and
//     y[i] += sqrt(nu_old[j] / nu_new[i]) * x[j] * c_r * exp(-2 pi i k_new . disp_i / L)
// (restated and pinned to the compiled reference in tests/repr_builders.py: apply_sminus).  Scatter with fp64 atomics:
// the reference itself adds these contributions from several threads in no fixed order, so agreement is to rounding.
// y must be zero on entry.
__global__ void __launch_bounds__(kSBlock) sec_apply_ladder_kernel(SecDev So, SecDev Sn, const double2 *__restrict__ phase_new, const double2 *__restrict__ coef,
                                                                   int lower, const double2 *__restrict__ x, double2 *y)
{
    __shared__ double2 c[kMaxTrans];
    if (threadIdx.x < So.nsites) c[threadIdx.x] = coef[threadIdx.x];
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < So.n; r += (int64_t)gridDim.x * blockDim.x) {
        const double2 xj = x[r];
        const double nj = So.nu[r];
        if (!(hypot(xj.x, xj.y) >= 2e-12) || !(nj >= 2e-12)) continue;                 // :1752
        uint32_t a, b;
        sec_halves(So, So.keys[r], a, b);
        const uint32_t st = spread_bits(a) | (spread_bits(b) << 1);
        for (int site = 0; site < So.nsites; site++) {
            const uint32_t bit = 1u << site;
            if (lower ? (st & bit) != 0u : (st & bit) == 0u) continue;                 // S^- needs an up spin (digit 0), S^+ a down spin
            const uint32_t s2 = st ^ bit;
            uint32_t ca = 0, cb = 0;
            const int i = sec_canon(Sn, squeeze_bits(s2), squeeze_bits(s2 >> 1), ca, cb);
            if (i < 0) continue;
            const int64_t tgt = sec_lookup(Sn, sec_key(Sn, ca, cb));
            if (tgt < 0) continue;
            const double ni = Sn.nu[tgt];
            if (!(ni >= 2e-12)) continue;                                              // :1810
            const double w = sqrt(nj / ni);
            const double2 ph = phase_new[i];                                           // exp(+2 pi i k.disp/L): conjugated below
            const double2 t1 = make_double2(w * xj.x, w * xj.y);
            const double2 t2 = make_double2(t1.x * c[site].x - t1.y * c[site].y, t1.x * c[site].y + t1.y * c[site].x);
            atomicAdd(&y[tgt].x, t2.x * ph.x + t2.y * ph.y);
            atomicAdd(&y[tgt].y, t2.y * ph.x - t2.x * ph.y);
        }
    }
}

// ------------------------------------------------------------------------------------------ one-site electron operators
// model::moprXvec_repr (src/model.cc:1716-1846) for A = sum_r c_r O_r between electron sectors of one lattice (restated and pinned
// in tests/repr_ops_fermion.py).  Coefficients travel by value: at most 16 sites.
struct ElCoef { double2 c[2][16]; };

// Diagonal branch (:1758-1761), O_r = cu_r n_up,r + cd_r n_dn,r: the representative keeps its row and
//   y[j] = sqrt(nu_old[j] / nu_new[j]) * x[j] * sum_r (cu_r n_up,r + cd_r n_dn,r)(state_j),
// rows with |x[j]|, nu_old[j] or nu_new[j] below lanczos_precision give 0 (:1752, :1760).
__global__ void __launch_bounds__(kSBlock) el_apply_density_kernel(SecDev S, const double *__restrict__ nu_new, ElCoef C,
                                                                   const double2 *__restrict__ x, double2 *y)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S.n; r += (int64_t)gridDim.x * blockDim.x) {
        const double2 xj = x[r];
        const double nj = S.nu[r], ni = nu_new[r];
        double2 out = make_double2(0.0, 0.0);
        if (hypot(xj.x, xj.y) >= 2e-12 && nj >= 2e-12 && ni >= 2e-12) {
            uint32_t a, b;
            sec_halves(S, S.keys[r], a, b);
            const uint32_t st = sec_zip(S, a, b);
            double2 d = make_double2(0.0, 0.0);
            for (int site = 0; site < S.nsites; site++) {
                if ((st >> (2 * site)) & 1u) { d.x = __dadd_rn(d.x, C.c[0][site].x); d.y = __dadd_rn(d.y, C.c[0][site].y); }
                if ((st >> (2 * site + 1)) & 1u) { d.x = __dadd_rn(d.x, C.c[1][site].x); d.y = __dadd_rn(d.y, C.c[1][site].y); }
            }
            const double w = __dsqrt_rn(__ddiv_rn(nj, ni));
            const double2 t = make_double2(__dmul_rn(w, xj.x), __dmul_rn(w, xj.y));
            out = make_double2(__dsub_rn(__dmul_rn(t.x, d.x), __dmul_rn(t.y, d.y)), __dadd_rn(__dmul_rn(t.x, d.y), __dmul_rn(t.y, d.x)));
        }
        y[r] = out;
    }
}

// c_{r,sp} (create = 0) or c+_{r,sp} on st with oprXphi's sign (src/basis.cc:2717-2731, the halves of el_hop): parity of the
// electrons below site r, and for spin down the up electron of site r, counted on the state the operator acts on.
__device__ __forceinline__ bool el_one(uint32_t st, int r, int sp, int create, uint32_t &s2, int &sg)
{
    const uint32_t bit = 1u << (2 * r + sp);
    if (create ? (st & bit) != 0u : (st & bit) == 0u) return false;
    sg = __popc(st & ((1u << (2 * r)) - 1u)) & 1;
    if (sp) sg ^= (st >> (2 * r)) & 1u;
    s2 = st ^ bit;
    return true;
}

// Off-diagonal branch (:1762-1834) for one- and two-operator terms on one site (c, c+, S^- = c+_dn c_up, S^+ = c+_up c_dn).  The
// reference scatters every term of the OLD representative j into the new sector,
//     y[i] += sqrt(nu_old[j] / nu_new[i]) * x[j] * c_r * conj(phase_new[t]) * (-1)^(operator sign + el_trans_sign(rep_i, t)),
// which needs fp64 atomics and lands in no fixed order.  Here every output row is written once instead: the ADJOINT term
// (nops operators ops[0] then ops[1], each (spin, create)) acts on the NEW representative i, the state it produces is brought to
// its representative j in the OLD sector with the same rule, and y[i] takes the conjugate of that element:
//     y[i] = sum_r sqrt(nu_new[i] / nu_old[j]) * c_r * phase_old[t] * (-1)^(operator sign + el_trans_sign(rep_j, t)) * x[j],
// terms in site order -- the same matrix for coefficients e^{+i q.r} between K and K + q, bit-identical from run to run.
__global__ void __launch_bounds__(kSBlock) el_apply_gather_kernel(SecDev So, SecDev Sn, const double2 *__restrict__ phase_old, ElCoef C,
                                                                  int nops, int sp0, int cr0, int sp1, int cr1,
                                                                  const double2 *__restrict__ x, double2 *y)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < Sn.n; r += (int64_t)gridDim.x * blockDim.x) {
        const double ni = Sn.nu[r];
        double2 acc = make_double2(0.0, 0.0);
        if (ni >= 2e-12) {
            uint32_t a, b;
            sec_halves(Sn, Sn.keys[r], a, b);
            const uint32_t st = sec_zip(Sn, a, b);
            for (int site = 0; site < Sn.nsites; site++) {
                uint32_t s1, s2;
                int g1, g2 = 0;
                if (!el_one(st, site, sp0, cr0, s1, g1)) continue;
                s2 = s1;
                if (nops == 2 && !el_one(s1, site, sp1, cr1, s2, g2)) continue;
                uint32_t a2, b2, ca = 0, cb = 0;
                sec_unzip(So, s2, a2, b2);
                const int t = sec_canon(So, a2, b2, ca, cb);
                if (t < 0) continue;
                const int64_t j = sec_lookup(So, sec_key(So, ca, cb));
                if (j < 0) continue;
                const double nj = So.nu[j];
                if (!(nj >= 2e-12)) continue;                                          // :1810
                const double2 xj = x[j];
                if (!(hypot(xj.x, xj.y) >= 2e-12)) continue;                           // :1752
                const double w = __dsqrt_rn(__ddiv_rn(ni, nj));
                const double2 cf = C.c[0][site], ph = phase_old[t];
                const double2 cp = make_double2(__dsub_rn(__dmul_rn(cf.x, ph.x), __dmul_rn(cf.y, ph.y)),
                                                __dadd_rn(__dmul_rn(cf.x, ph.y), __dmul_rn(cf.y, ph.x)));
                double re = __dmul_rn(w, __dsub_rn(__dmul_rn(cp.x, xj.x), __dmul_rn(cp.y, xj.y)));
                double im = __dmul_rn(w, __dadd_rn(__dmul_rn(cp.x, xj.y), __dmul_rn(cp.y, xj.x)));
                if ((g1 ^ g2 ^ el_trans_sign(So, sec_zip(So, ca, cb), t)) & 1) { re = -re; im = -im; }
                acc.x = __dadd_rn(acc.x, re); acc.y = __dadd_rn(acc.y, im);
            }
        }
        y[r] = acc;
    }
}

static double wall_clock() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
struct FlagToInt { __host__ __device__ int operator()(uint8_t f) const { return (int)f; } };
static int sgrid(int64_t n) { int64_t g = (n + kSBlock - 1) / kSBlock; if (g < 1) g = 1; if (g > 148 * 64) g = 148 * 64; return (int)g; }

}  // namespace qb

using namespace qb;

struct qbgpu_sector {
    int dim = 0, L[3] = {1, 1, 1}, k[3] = {0, 0, 0}, spec = 0, nsites = 0, nsub = 0, ntrans = 0, nsubtrans = 0, ndown = 0;
    bool electron = false;                           // two bits per site (nup = ndown field, ndn below); nsub = bits of a half state
    int ndn = 0;
    uint16_t *d_invmask = nullptr;
    int64_t n = 0, zero_norm = 0;
    SecDev dev{};
    uint16_t *d_subT = nullptr, *d_rep = nullptr;
    uint8_t *d_dist = nullptr;
    uint32_t *d_keys = nullptr, *d_seg = nullptr;
    double *d_nu = nullptr;
    double2 *d_phase = nullptr;
    std::vector<std::complex<double>> phase;
    std::vector<std::vector<int>> disps;            // parent displacements, lexicographic
    std::vector<int> site_of_coor;                   // helper for bond generation / S^z_q phases
    std::vector<std::vector<int>> coor;
    double enumerate_s = 0, norms_s = 0;
};

namespace {

struct HostLattice {
    int dim, spec, N;
    std::vector<int> L, order;
    std::vector<std::vector<int>> coor, disps;
    HostLattice(int dim_, const int *L_, int spec_) : dim(dim_), spec(spec_), L(L_, L_ + dim_)
    {
        order.push_back(spec);
        for (int d = 0; d < dim; d++) if (d != spec) order.push_back(d);
        N = 1; for (int d = 0; d < dim; d++) N *= L[d];
        coor.assign(N, std::vector<int>(dim));
        for (int s = 0; s < N; s++) { int r = s; for (int d : order) { coor[s][d] = r % L[d]; r /= L[d]; } }
        std::vector<int> c(dim, 0);
        for (int t = 0; t < N; t++) {                                   // lexicographic, last index fastest
            disps.push_back(c);
            for (int d = dim - 1; d >= 0; d--) { if (++c[d] < L[d]) break; c[d] = 0; }
        }
    }
    int site(const std::vector<int> &c) const
    {
        int s = 0, mul = 1;
        for (int d : order) { int v = ((c[d] % L[d]) + L[d]) % L[d]; s += v * mul; mul *= L[d]; }
        return s;
    }
    std::vector<int> plan(const std::vector<int> &disp) const        // plan[site] = site + disp
    {
        std::vector<int> p(N), c(dim);
        for (int s = 0; s < N; s++) { for (int d = 0; d < dim; d++) c[d] = coor[s][d] + disp[d]; p[s] = site(c); }
        return p;
    }
};

// does J = Ja[ia] + Jb[ib] have a solution?  (weighted union-find over the 2 * 2^nsub labels)
bool lin_tables_exist(const std::vector<uint32_t> &keys, int nsub)
{
    const uint32_t half = 1u << nsub;
    std::vector<int32_t> parent(2 * half);
    std::vector<int64_t> off(2 * half, 0);
    for (uint32_t i = 0; i < 2 * half; i++) parent[i] = (int32_t)i;
    std::vector<int32_t> path;
    auto find = [&](int32_t x) {
        path.clear();
        while (parent[x] != x) { path.push_back(x); x = parent[x]; }
        int64_t acc = 0;
        for (size_t t = path.size(); t-- > 0;) { const int32_t y = path[t]; acc += off[y]; off[y] = acc; parent[y] = x; }
        return x;
    };
    for (size_t J = 0; J < keys.size(); J++) {
        const int32_t x = (int32_t)(keys[J] & (half - 1)), y = (int32_t)(half + (keys[J] >> nsub));
        const int32_t rx = find(x), ry = find(y);
        const int64_t px = (x != rx) ? off[x] : 0, py = (y != ry) ? off[y] : 0;
        if (rx == ry) { if (px - py != (int64_t)J) return false; }
        else { parent[rx] = ry; off[rx] = (int64_t)J + py - px; }
    }
    return true;
}

struct SecMatFree {                      // what a matrix-free sector handle owns: the term list; everything else is the sector's
    SecDev dev;
    SecTerms *d_T = nullptr;
    const double2 *phase = nullptr;
};

void sector_free(qbgpu_sector *S)
{
    if (!S) return;
    cudaFree(S->d_subT); cudaFree(S->d_rep); cudaFree(S->d_dist); cudaFree(S->d_keys); cudaFree(S->d_seg); cudaFree(S->d_nu); cudaFree(S->d_phase); cudaFree(S->d_invmask);
    delete S;
}

}  // namespace

int qb::launch_spmv_sector_matfree(const qbgpu_matrix *A, const FusedArgs &a)
{
    Context &c = ctx();
    const SecMatFree *M = (const SecMatFree *)A->mf_sec;
    if (!A->api_complex) return fail(QBGPU_ERR_STATE, "matrix-free sector handle: complex vectors only");
    auto kern = a.dots ? sec_matfree_spmv_kernel<true> : sec_matfree_spmv_kernel<false>;
    int blocks_per_sm = 0;
    QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, kSBlock, 0));
    if (blocks_per_sm < 1) blocks_per_sm = 1;
    const int64_t n = A->n;
    if (n == 0) return QBGPU_OK;
    int64_t want = (n + kSBlock - 1) / kSBlock;
    int64_t cap = (int64_t)c.num_sms * blocks_per_sm;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    const int grid = (int)(want < cap ? want : cap);
    kern<<<grid, kSBlock, 0, c.stream>>>(M->dev, M->d_T, M->phase, (const double2 *)a.x, (const double2 *)a.z, (double2 *)a.y, a.alpha, a.gamma, a.beta,
                                         a.scal_mode, a.sc, a.dots, c.partials, c.ticket);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

void qb::sector_matfree_destroy(qbgpu_matrix *A)
{
    SecMatFree *M = (SecMatFree *)A->mf_sec;
    if (!M) return;
    cudaFree(M->d_T);
    delete M;
    A->mf_sec = nullptr;
}

extern "C" {

}  // extern "C"

// spins (one bit per site, n0 = ndown) or single-orbital electrons (two bits per site, n0 = nup, n1 = ndn)
static int sector_create_impl(qbgpu_sector_t *out, int dim, const int32_t *L, bool electron, int n0, int n1, const int32_t *k)
{
    QB_TRY(ensure_init());
    Context &c = ctx();
    if (!out || !L || !k || dim < 1 || dim > 3) return fail(QBGPU_ERR_ARG, "sector_create: bad arguments");
    *out = nullptr;
    int spec = -1, N = 1;
    for (int d = 0; d < dim; d++) { if (L[d] < 1) return fail(QBGPU_ERR_ARG, "sector_create: bad lattice size"); N *= L[d]; if (spec < 0 && L[d] % 2 == 0) spec = d; }
    if (spec < 0) return fail(QBGPU_ERR_ARG, "sector_create: no even direction (the reference's divide_lattice needs one, src/lattice.cc:1076-1083)");
    if (N > (electron ? 16 : 32) || N < 2) return fail(QBGPU_ERR_ARG, electron ? "sector_create: 2..16 sites for electrons" : "sector_create: 2..32 sites");
    if (n0 < 0 || n0 > N || n1 < 0 || n1 > N) return fail(QBGPU_ERR_ARG, "sector_create: bad particle numbers");
    const int ndown = n0;
    const double t0 = wall_clock();
    auto *S = new qbgpu_sector;
    const int nhs = N / 2;                                              // sites of a half
    const int bps = electron ? 2 : 1;                                   // bits per site
    S->dim = dim; S->spec = spec; S->nsites = N; S->nsub = nhs * bps; S->ntrans = N; S->nsubtrans = N / 2; S->ndown = n0; S->ndn = n1; S->electron = electron;
    for (int d = 0; d < dim; d++) { S->L[d] = L[d]; S->k[d] = k[d]; }
    HostLattice par(dim, S->L, spec);
    int Ls[3] = {S->L[0], S->L[1], S->L[2]};
    Ls[spec] /= 2;
    HostLattice sub(dim, Ls, spec);
    const int nsub = S->nsub, nst = sub.N;                              // nsub: BITS of a half state
    const uint32_t half = 1u << nsub;
    S->disps = par.disps; S->coor = par.coor;

    // sublattice translations of every half state, their representatives and distances
    std::vector<std::vector<int>> splans;
    for (auto &d : sub.disps) splans.push_back(sub.plan(d));
    std::vector<uint16_t> subT((size_t)nst * half);
    const uint32_t dmask = (1u << bps) - 1u;
    for (int j = 0; j < nst; j++)
        for (uint32_t x = 0; x < half; x++) {
            uint32_t y = 0;
            for (int s = 0; s < nhs; s++) y |= ((x >> (bps * s)) & dmask) << (bps * splans[j][s]);
            subT[(size_t)j * half + x] = (uint16_t)y;
        }
    std::vector<uint16_t> rep(half);
    std::vector<uint8_t> dist(half), seen(half, 0);
    std::vector<uint16_t> reps;
    for (uint32_t x = 0; x < half; x++) {                               // src/basis.cc:1385-1419
        if (seen[x]) continue;
        reps.push_back((uint16_t)x);
        for (int j = 0; j < nst; j++) {
            const uint32_t y = subT[(size_t)j * half + x];
            if (!seen[y]) { seen[y] = 1; rep[y] = (uint16_t)x; dist[y] = (uint8_t)j; }
        }
    }
    // each parent translation in terms of sublattice translations of the halves
    std::map<std::vector<int>, int> sp_index;
    for (int j = 0; j < nst; j++) sp_index[splans[j]] = j;
    std::map<std::vector<int>, int> dindex;
    for (int i = 0; i < N; i++) dindex[par.disps[i]] = i;
    std::vector<int> fs(N), fa(N), fb(N);
    for (int i = 0; i < N; i++) {
        const std::vector<int> p = par.plan(par.disps[i]);
        std::vector<int> pa(nhs), pb(nhs);
        if (p[0] % 2 == 0) { fs[i] = 0; for (int t = 0; t < nhs; t++) { pa[t] = p[2 * t] / 2; pb[t] = (p[2 * t + 1] - 1) / 2; } }
        else               { fs[i] = 1; for (int t = 0; t < nhs; t++) { pa[t] = p[2 * t + 1] / 2; pb[t] = (p[2 * t] - 1) / 2; } }
        auto ia = sp_index.find(pa), ib = sp_index.find(pb);
        if (ia == sp_index.end() || ib == sp_index.end()) { sector_free(S); return fail(QBGPU_ERR_STATE, "sector_create: translation does not factor over the sublattices"); }
        fa[i] = ia->second; fb[i] = ib->second;
    }
    SecDev &D = S->dev;
    D.nsites = N; D.nsub = nsub; D.ntrans = N; D.shift = std::max(0, 2 * nsub - 16); D.lin_order = 1;
    D.electron = electron ? 1 : 0; D.invmask = nullptr;
    std::vector<uint16_t> invmask((size_t)N * 16, 0);
    for (int i = 0; i < N; i++) {
        if (electron) {                                                 // inversions of translation i: mbasis_elem::transform's bubble-sort count
            const std::vector<int> p = par.plan(par.disps[i]);
            for (int s1 = 0; s1 < N; s1++)
                for (int s2 = s1 + 1; s2 < N; s2++) if (p[s1] > p[s2]) invmask[(size_t)i * 16 + s1] |= (uint16_t)(1u << s2);
        }
        std::vector<int> m(dim);
        for (int d = 0; d < dim; d++) m[d] = (S->L[d] - par.disps[i][d]) % S->L[d];
        const int iv = dindex[m];
        D.fwd_swap[i] = (uint8_t)fs[i]; D.fwd_ja[i] = (uint8_t)fa[i]; D.fwd_jb[i] = (uint8_t)fb[i];
        D.inv_swap[i] = (uint8_t)fs[iv]; D.inv_ja[i] = (uint8_t)fa[iv]; D.inv_jb[i] = (uint8_t)fb[iv];
        long long num = 0;                                              // src/basis.cc:2129-2147
        for (int d = 0; d < dim; d++) { const int kk = ((S->k[d] % S->L[d]) + S->L[d]) % S->L[d]; num += (long long)kk * par.disps[i][d] * (N / S->L[d]); }
        D.bad[i] = (num % N != 0) ? 1 : 0;
        D.kt[i] = (int16_t)(num % N);
        double e = 0.0;                                                 // src/model.cc:808-814
        for (int d = 0; d < dim; d++) e += S->k[d] * par.disps[i][d] / static_cast<double>(S->L[d]);
        S->phase.push_back(std::exp(std::complex<double>(0.0, 2.0 * 3.1415926535897932 * e)));
    }

    uint16_t *d_reps = nullptr;
    uint8_t *d_flag = nullptr;
    void *d_tmp = nullptr;
    int *d_nsel = nullptr;
    uint32_t *d_sorted = nullptr;
    unsigned long long *d_zero = nullptr;
    auto cleanup = [&]() { cudaFree(d_reps); cudaFree(d_flag); cudaFree(d_tmp); cudaFree(d_nsel); cudaFree(d_sorted); cudaFree(d_zero); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); sector_free(S); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&S->d_subT, subT.size() * 2));
    QB_CU(cudaMalloc(&S->d_rep, half * 2));
    QB_CU(cudaMalloc(&S->d_dist, half));
    QB_CU(cudaMalloc(&d_reps, reps.size() * 2));
    QB_CU(cudaMalloc(&S->d_phase, sizeof(double2) * N));
    QB_CU(cudaMemcpyAsync(S->d_subT, subT.data(), subT.size() * 2, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(S->d_rep, rep.data(), half * 2, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(S->d_dist, dist.data(), half, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_reps, reps.data(), reps.size() * 2, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(S->d_phase, S->phase.data(), sizeof(double2) * N, cudaMemcpyHostToDevice, c.stream));
    if (electron) {
        QB_CU(cudaMalloc(&S->d_invmask, invmask.size() * 2));
        QB_CU(cudaMemcpyAsync(S->d_invmask, invmask.data(), invmask.size() * 2, cudaMemcpyHostToDevice, c.stream));
        D.invmask = S->d_invmask;
    }
    D.subT = S->d_subT; D.rep = S->d_rep; D.dist = S->d_dist;

    // representatives: flag the candidates (even half a sublattice representative), compact in Lin order
    const int nreps = (int)reps.size();
    const int64_t ncand = (int64_t)nreps << nsub;
    if (ncand > 2147483647LL) { cleanup(); sector_free(S); return fail(QBGPU_ERR_STATE, "sector_create: candidate count overflow"); }
    QB_CU(cudaMalloc(&d_flag, ncand));
    if (electron) el_flag_kernel<<<sgrid(ncand), kSBlock, 0, c.stream>>>(D, d_reps, nreps, n0, n1, ncand, d_flag);
    else sec_flag_kernel<<<sgrid(ncand), kSBlock, 0, c.stream>>>(D, d_reps, nreps, ndown, ncand, d_flag);
    QB_LAUNCH_COUNT();
    QB_CU(cudaMalloc(&d_nsel, sizeof(int)));
    uint32_t *d_all = nullptr;
    {
        // the sector size is not known before the selection: count first (a sum over the flags), then select
        size_t tb = 0;
        int *d_cnt = d_nsel;
        auto fit = thrust::make_transform_iterator((const uint8_t *)d_flag, FlagToInt());
        QB_CU(cub::DeviceReduce::Sum(nullptr, tb, fit, d_cnt, (int)ncand, c.stream));
        QB_CU(cudaMalloc(&d_tmp, tb ? tb : 1));
        QB_CU(cub::DeviceReduce::Sum(d_tmp, tb, fit, d_cnt, (int)ncand, c.stream));
        int cnt = 0;
        QB_CU(cudaMemcpyAsync(&cnt, d_cnt, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        QB_CU(cudaStreamSynchronize(c.stream));
        cudaFree(d_tmp); d_tmp = nullptr;
        if (cnt <= 0) { cleanup(); sector_free(S); return fail(QBGPU_ERR_ARG, "sector_create: empty sector"); }
        S->n = cnt;
        QB_CU(cudaMalloc(&d_all, sizeof(uint32_t) * (size_t)cnt));
        S->d_keys = d_all;
        thrust::counting_iterator<uint32_t> it(0u);
        QB_CU(cub::DeviceSelect::Flagged(nullptr, tb, it, d_flag, d_all, d_nsel, (int)ncand, c.stream));
        QB_CU(cudaMalloc(&d_tmp, tb ? tb : 1));
        QB_CU(cub::DeviceSelect::Flagged(d_tmp, tb, it, d_flag, d_all, d_nsel, (int)ncand, c.stream));
        sec_cand_to_key_kernel<<<sgrid(cnt), kSBlock, 0, c.stream>>>(cnt, d_reps, nreps, nsub, d_all);
        QB_LAUNCH_COUNT();
    }
    // Lin tables or bisection order?  (decided on the host exactly like the reference's graph search would)
    {
        std::vector<uint32_t> hk((size_t)S->n);
        QB_CU(cudaMemcpyAsync(hk.data(), S->d_keys, sizeof(uint32_t) * hk.size(), cudaMemcpyDeviceToHost, c.stream));
        QB_CU(cudaStreamSynchronize(c.stream));
        D.lin_order = lin_tables_exist(hk, nsub) ? 1 : 0;
    }
    if (!D.lin_order) {
        if (electron) el_lin_to_zip_kernel<<<sgrid(S->n), kSBlock, 0, c.stream>>>(S->n, nsub, S->d_keys);
        else sec_lin_to_zip_kernel<<<sgrid(S->n), kSBlock, 0, c.stream>>>(S->n, nsub, S->d_keys);
        QB_LAUNCH_COUNT();
        QB_CU(cudaMalloc(&d_sorted, sizeof(uint32_t) * (size_t)S->n));
        size_t tb = 0;
        cudaFree(d_tmp); d_tmp = nullptr;
        QB_CU(cub::DeviceRadixSort::SortKeys(nullptr, tb, S->d_keys, d_sorted, (int)S->n, 0, 32, c.stream));
        QB_CU(cudaMalloc(&d_tmp, tb ? tb : 1));
        QB_CU(cub::DeviceRadixSort::SortKeys(d_tmp, tb, S->d_keys, d_sorted, (int)S->n, 0, 32, c.stream));
        QB_CU(cudaStreamSynchronize(c.stream));
        std::swap(S->d_keys, d_sorted);
    }
    D.keys = S->d_keys; D.n = S->n;
    const uint32_t nseg = 1u << (2 * nsub - D.shift);
    QB_CU(cudaMalloc(&S->d_seg, sizeof(uint32_t) * ((size_t)nseg + 1)));
    sec_seg_kernel<<<sgrid(nseg + 1), kSBlock, 0, c.stream>>>(S->n, S->d_keys, D.shift, nseg, S->d_seg);
    QB_LAUNCH_COUNT();
    D.seg = S->d_seg;
    QB_CU(cudaStreamSynchronize(c.stream));
    S->enumerate_s = wall_clock() - t0;

    const double t1 = wall_clock();
    QB_CU(cudaMalloc(&S->d_nu, sizeof(double) * (size_t)S->n));
    QB_CU(cudaMalloc(&d_zero, sizeof(unsigned long long)));
    QB_CU(cudaMemsetAsync(d_zero, 0, sizeof(unsigned long long), c.stream));
    if (electron) el_norm_kernel<<<sgrid(S->n), kSBlock, 0, c.stream>>>(D, S->d_nu, d_zero);
    else sec_norm_kernel<<<sgrid(S->n), kSBlock, 0, c.stream>>>(D, S->d_nu, d_zero);
    QB_LAUNCH_COUNT();
    unsigned long long z = 0;
    QB_CU(cudaMemcpyAsync(&z, d_zero, sizeof(z), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
    S->zero_norm = (int64_t)z;
    D.nu = S->d_nu;
    S->norms_s = wall_clock() - t1;
    cleanup();
#undef QB_CU
    *out = S;
    return QBGPU_OK;
}

extern "C" {

int qbgpu_sector_create(qbgpu_sector_t *out, int dim, const int32_t *L, int ndown, const int32_t *k)
{ return sector_create_impl(out, dim, L, false, ndown, 0, k); }

/* A (N_up, N_dn, momentum) sector of single-orbital electrons on an untilted lattice of at most 16 sites: the device counterpart
 * of fill_Weisse_table + enumerate_basis_repr for the reference's "electron" orbital (src/basis.cc:49-96; two bits per site, bit 0
 * up, bit 1 down).  Same representatives, order and norms as the reference (translation signs: src/basis.cc:593-620, 2134-2147). */
int qbgpu_sector_create_electron(qbgpu_sector_t *out, int dim, const int32_t *L, int nup, int ndn, const int32_t *k)
{ return sector_create_impl(out, dim, L, true, nup, ndn, k); }

int qbgpu_sector_destroy(qbgpu_sector_t S) { sector_free(S); return QBGPU_OK; }

int qbgpu_sector_get_info(qbgpu_sector_t S, qbgpu_sector_info *info)
{
    if (!S || !info) return fail(QBGPU_ERR_ARG, "sector_get_info: null argument");
    info->dim = S->n; info->zero_norm = S->zero_norm; info->nsites = S->nsites; info->lin_order = S->dev.lin_order;
    info->enumerate_seconds = S->enumerate_s; info->norms_seconds = S->norms_s;
    return QBGPU_OK;
}

int qbgpu_sector_states(qbgpu_sector_t S, uint32_t *states_host)
{
    if (!S || !states_host) return fail(QBGPU_ERR_ARG, "sector_states: null argument");
    Context &c = ctx();
    uint32_t *d = nullptr;
    QB_CUDA(cudaMalloc(&d, sizeof(uint32_t) * (size_t)S->n));
    sec_states_kernel<<<sgrid(S->n), kSBlock, 0, c.stream>>>(S->dev, d);
    QB_LAUNCH_COUNT();
    cudaError_t e = cudaMemcpyAsync(states_host, d, sizeof(uint32_t) * (size_t)S->n, cudaMemcpyDeviceToHost, c.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
    cudaFree(d);
    QB_CUDA(e);
    return QBGPU_OK;
}

int qbgpu_sector_norms(qbgpu_sector_t S, double *nu_host)
{
    if (!S || !nu_host) return fail(QBGPU_ERR_ARG, "sector_norms: null argument");
    Context &c = ctx();
    QB_CUDA(cudaMemcpyAsync(nu_host, S->d_nu, sizeof(double) * (size_t)S->n, cudaMemcpyDeviceToHost, c.stream));
    QB_CUDA(cudaStreamSynchronize(c.stream));
    return QBGPU_OK;
}

int qbgpu_sector_apply_sz(qbgpu_sector_t S_old, qbgpu_sector_t S_new, const double *coef_reim, const void *x_old_dev, void *y_new_dev)
{
    if (!S_old || !S_new || !coef_reim || !x_old_dev || !y_new_dev) return fail(QBGPU_ERR_ARG, "sector_apply_sz: null argument");
    if (S_old->electron || S_new->electron) return fail(QBGPU_ERR_STATE, "sector_apply_sz: spin sectors only");
    if (S_old->n != S_new->n || S_old->nsites != S_new->nsites || S_old->ndown != S_new->ndown || S_old->dim != S_new->dim ||
        memcmp(S_old->L, S_new->L, sizeof(S_old->L)) != 0 || S_old->dev.lin_order != S_new->dev.lin_order)
        return fail(QBGPU_ERR_ARG, "sector_apply_sz: the two sectors must share lattice and Sz (same representatives)");
    Context &c = ctx();
    double2 *d_coef = nullptr;
    QB_CUDA(cudaMalloc(&d_coef, sizeof(double2) * kMaxTrans));
    cudaError_t e = cudaMemcpyAsync(d_coef, coef_reim, sizeof(double2) * S_old->nsites, cudaMemcpyHostToDevice, c.stream);
    if (e == cudaSuccess) {
        sec_apply_sz_kernel<<<sgrid(S_old->n), kSBlock, 0, c.stream>>>(S_old->dev, S_new->d_nu, d_coef, (const double2 *)x_old_dev, (double2 *)y_new_dev);
        QB_LAUNCH_COUNT();
        e = cudaStreamSynchronize(c.stream);
    }
    cudaFree(d_coef);
    QB_CUDA(e);
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

int qbgpu_sector_apply_ladder(qbgpu_sector_t S_old, qbgpu_sector_t S_new, int lower, const double *coef_reim, const void *x_old_dev, void *y_new_dev)
{
    if (!S_old || !S_new || !coef_reim || !x_old_dev || !y_new_dev) return fail(QBGPU_ERR_ARG, "sector_apply_ladder: null argument");
    if (S_old->electron || S_new->electron) return fail(QBGPU_ERR_STATE, "sector_apply_ladder: spin sectors only");
    if (S_old->nsites != S_new->nsites || S_old->dim != S_new->dim || memcmp(S_old->L, S_new->L, sizeof(S_old->L)) != 0)
        return fail(QBGPU_ERR_ARG, "sector_apply_ladder: the two sectors must share the lattice");
    if (S_new->ndown != S_old->ndown + (lower ? 1 : -1))
        return fail(QBGPU_ERR_ARG, "sector_apply_ladder: the target sector must have one more (S^-) or one fewer (S^+) down spin");
    Context &c = ctx();
    double2 *d_coef = nullptr;
    QB_CUDA(cudaMalloc(&d_coef, sizeof(double2) * kMaxTrans));
    cudaError_t e = cudaMemcpyAsync(d_coef, coef_reim, sizeof(double2) * S_old->nsites, cudaMemcpyHostToDevice, c.stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(y_new_dev, 0, sizeof(double2) * (size_t)S_new->n, c.stream);
    if (e == cudaSuccess && S_old->n > 0) {
        sec_apply_ladder_kernel<<<sgrid(S_old->n), kSBlock, 0, c.stream>>>(S_old->dev, S_new->dev, S_new->d_phase, d_coef, lower ? 1 : 0,
                                                                            (const double2 *)x_old_dev, (double2 *)y_new_dev);
        QB_LAUNCH_COUNT();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
    cudaFree(d_coef);
    QB_CUDA(e);
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

}  // extern "C"

// checks shared by the electron operator entries: both sectors electron sectors (else QBGPU_ERR_STATE) on one lattice, and
// S_new's particle numbers (nup, ndn) = S_old's + (dup, ddn)
static int el_op_check(const char *who, qbgpu_sector_t So, qbgpu_sector_t Sn, const void *coef, const void *x, const void *y, int dup, int ddn)
{
    char msg[160];
    if (!So || !Sn || !coef || !x || !y) { snprintf(msg, sizeof(msg), "%s: null argument", who); return fail(QBGPU_ERR_ARG, msg); }
    if (!So->electron || !Sn->electron) { snprintf(msg, sizeof(msg), "%s: electron sectors only", who); return fail(QBGPU_ERR_STATE, msg); }
    if (So->nsites != Sn->nsites || So->dim != Sn->dim || memcmp(So->L, Sn->L, sizeof(So->L)) != 0) {
        snprintf(msg, sizeof(msg), "%s: the two sectors must share the lattice", who); return fail(QBGPU_ERR_ARG, msg);
    }
    if (Sn->ndown != So->ndown + dup || Sn->ndn != So->ndn + ddn) {
        snprintf(msg, sizeof(msg), "%s: the target sector must have (N_up, N_dn) = (%d, %d), it has (%d, %d)", who, So->ndown + dup, So->ndn + ddn,
                 Sn->ndown, Sn->ndn);
        return fail(QBGPU_ERR_ARG, msg);
    }
    return QBGPU_OK;
}

static int el_gather(qbgpu_sector_t So, qbgpu_sector_t Sn, const double *c_reim, int nops, int sp0, int cr0, int sp1, int cr1, const void *x, void *y)
{
    Context &c = ctx();
    ElCoef C;
    memset(&C, 0, sizeof(C));
    memcpy(C.c[0], c_reim, sizeof(double2) * So->nsites);
    el_apply_gather_kernel<<<sgrid(Sn->n), kSBlock, 0, c.stream>>>(So->dev, Sn->dev, So->d_phase, C, nops, sp0, cr0, sp1, cr1,
                                                                   (const double2 *)x, (double2 *)y);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    QB_CUDA(cudaStreamSynchronize(c.stream));
    return QBGPU_OK;
}

extern "C" {

int qbgpu_sector_apply_density(qbgpu_sector_t S_old, qbgpu_sector_t S_new, const double *cu_reim, const double *cd_reim, const void *x_old_dev,
                               void *y_new_dev)
{
    const int rc = el_op_check("sector_apply_density", S_old, S_new, cu_reim, x_old_dev, y_new_dev, 0, 0);
    if (rc != QBGPU_OK) return rc;
    if (!cd_reim) return fail(QBGPU_ERR_ARG, "sector_apply_density: null argument");
    if (S_old->n != S_new->n || S_old->dev.lin_order != S_new->dev.lin_order) return fail(QBGPU_ERR_ARG, "sector_apply_density: different representatives");
    Context &c = ctx();
    ElCoef C;
    memset(&C, 0, sizeof(C));
    memcpy(C.c[0], cu_reim, sizeof(double2) * S_old->nsites);
    memcpy(C.c[1], cd_reim, sizeof(double2) * S_old->nsites);
    el_apply_density_kernel<<<sgrid(S_old->n), kSBlock, 0, c.stream>>>(S_old->dev, S_new->d_nu, C, (const double2 *)x_old_dev, (double2 *)y_new_dev);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    QB_CUDA(cudaStreamSynchronize(c.stream));
    return QBGPU_OK;
}

int qbgpu_sector_apply_spin_flip(qbgpu_sector_t S_old, qbgpu_sector_t S_new, int lower, const double *c_reim, const void *x_old_dev, void *y_new_dev)
{
    const int rc = el_op_check("sector_apply_spin_flip", S_old, S_new, c_reim, x_old_dev, y_new_dev, lower ? -1 : 1, lower ? 1 : -1);
    if (rc != QBGPU_OK) return rc;
    // the adjoint term acting on the new representative: S^+ = c+_up c_dn for lower, S^- = c+_dn c_up otherwise
    return lower ? el_gather(S_old, S_new, c_reim, 2, 1, 0, 0, 1, x_old_dev, y_new_dev)
                 : el_gather(S_old, S_new, c_reim, 2, 0, 0, 1, 1, x_old_dev, y_new_dev);
}

int qbgpu_sector_apply_fermion(qbgpu_sector_t S_old, qbgpu_sector_t S_new, int create, int spin, const double *c_reim, const void *x_old_dev,
                               void *y_new_dev)
{
    if (spin != 0 && spin != 1) return fail(QBGPU_ERR_ARG, "sector_apply_fermion: spin is 0 (up) or 1 (down)");
    const int d = create ? 1 : -1;
    const int rc = el_op_check("sector_apply_fermion", S_old, S_new, c_reim, x_old_dev, y_new_dev, spin == 0 ? d : 0, spin == 1 ? d : 0);
    if (rc != QBGPU_OK) return rc;
    return el_gather(S_old, S_new, c_reim, 1, spin, create ? 0 : 1, 0, 0, x_old_dev, y_new_dev);    // adjoint: c+ for c, c for c+
}

int qbgpu_sector_build_heisenberg(qbgpu_sector_t S, qbgpu_matrix_t *A, int nbonds, const int32_t *bonds, double J, double fake_pos, int flags)
{
    if (!S || !A || !bonds || nbonds < 1) return fail(QBGPU_ERR_ARG, "sector_build_heisenberg: bad arguments");
    if (S->electron) return fail(QBGPU_ERR_STATE, "sector_build_heisenberg: this is an electron sector (qbgpu_sector_build_hubbard)");
    if (nbonds > kMaxTerms) return fail(QBGPU_ERR_ARG, "sector_build_heisenberg: at most 128 bonds");
    Context &c = ctx();
    *A = nullptr;
    std::vector<std::pair<int, int>> bs;
    for (int t = 0; t < nbonds; t++) {
        const int p = bonds[2 * t], q = bonds[2 * t + 1];
        if (p < 0 || q < 0 || p >= S->nsites || q >= S->nsites || p == q) return fail(QBGPU_ERR_ARG, "sector_build_heisenberg: bad bond");
        bs.push_back({std::min(p, q), std::max(p, q)});
    }
    std::stable_sort(bs.begin(), bs.end());                             // mopr::operator+=, src/operators.cc:901-925
    SecTerms T;
    memset(&T, 0, sizeof(T));
    T.nterms = nbonds; T.J = J; T.fake_pos = fake_pos;
    for (int t = 0; t < nbonds; t++) { T.p[t] = (uint8_t)bs[t].first; T.q[t] = (uint8_t)bs[t].second; }

    SecTerms *d_T = nullptr;
    int64_t *d_cap = nullptr, *d_start = nullptr, *d_end = nullptr, *d_col = nullptr;
    double2 *d_val = nullptr;
    void *d_tmp = nullptr;
    auto cleanup = [&]() { cudaFree(d_T); cudaFree(d_cap); cudaFree(d_start); cudaFree(d_end); cudaFree(d_col); cudaFree(d_val); cudaFree(d_tmp); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    const int64_t n = S->n;
    QB_CU(cudaMalloc(&d_T, sizeof(SecTerms)));
    QB_CU(cudaMemcpyAsync(d_T, &T, sizeof(SecTerms), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMalloc(&d_cap, sizeof(int64_t) * (n + 1)));
    QB_CU(cudaMalloc(&d_start, sizeof(int64_t) * (n + 1)));
    QB_CU(cudaMalloc(&d_end, sizeof(int64_t) * (n + 1)));
    sec_cap_kernel<<<sgrid(n + 1), kSBlock, 0, c.stream>>>(S->dev, d_T, d_cap);
    QB_LAUNCH_COUNT();
    size_t tb = 0;
    QB_CU(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_cap, d_start, n + 1, c.stream));
    QB_CU(cudaMalloc(&d_tmp, tb ? tb : 1));
    QB_CU(cub::DeviceScan::ExclusiveSum(d_tmp, tb, d_cap, d_start, n + 1, c.stream));
    int64_t total = 0;
    QB_CU(cudaMemcpyAsync(&total, d_start + n, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaMalloc(&d_col, sizeof(int64_t) * (size_t)total));
    QB_CU(cudaMalloc(&d_val, sizeof(double2) * (size_t)total));
    sec_rows_kernel<<<sgrid(n), kSBlock, 0, c.stream>>>(S->dev, d_T, S->d_phase, d_start, d_end, d_col, d_val);
    QB_LAUNCH_COUNT();
    sec_len_kernel<<<sgrid(n), kSBlock, 0, c.stream>>>(n, d_start, d_end, d_cap);
    QB_LAUNCH_COUNT();
    cudaFree(d_tmp); d_tmp = nullptr;
    int64_t *d_sum = nullptr;
    QB_CU(cudaMalloc(&d_sum, sizeof(int64_t)));
    cudaError_t e1 = cub::DeviceReduce::Sum(nullptr, tb, d_cap, d_sum, n, c.stream);
    if (e1 == cudaSuccess) e1 = cudaMalloc(&d_tmp, tb ? tb : 1);
    if (e1 == cudaSuccess) e1 = cub::DeviceReduce::Sum(d_tmp, tb, d_cap, d_sum, n, c.stream);
    int64_t upper = 0;
    if (e1 == cudaSuccess) e1 = cudaMemcpyAsync(&upper, d_sum, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream);
    if (e1 == cudaSuccess) e1 = cudaStreamSynchronize(c.stream);
    cudaFree(d_sum);
    QB_CU(e1);
    QB_CU(cudaGetLastError());
#undef QB_CU
    int rc = create_from_device_csr(A, n, d_start, d_end, d_col, d_val, true, upper, 1, flags, true);
    cleanup();
    return rc;
}

/* Matrix-free handle over a sector: model<T>::MultMv / MultMv2 with matrix_free == true, repr branch (src/model.cc:1016-1107).
 * The handle borrows the sector's device tables: destroy it before the sector. */
int qbgpu_sector_matfree_heisenberg(qbgpu_sector_t S, qbgpu_matrix_t *A, int nbonds, const int32_t *bonds, double J, double fake_pos)
{
    QB_TRY(ensure_init());
    if (!S || !A || !bonds || nbonds < 1) return fail(QBGPU_ERR_ARG, "sector_matfree_heisenberg: bad arguments");
    if (S->electron) return fail(QBGPU_ERR_STATE, "sector_matfree_heisenberg: this is an electron sector");
    if (nbonds > kMaxTerms) return fail(QBGPU_ERR_ARG, "sector_matfree_heisenberg: at most 128 bonds");
    Context &c = ctx();
    *A = nullptr;
    std::vector<std::pair<int, int>> bs;
    for (int t = 0; t < nbonds; t++) {
        const int p = bonds[2 * t], q = bonds[2 * t + 1];
        if (p < 0 || q < 0 || p >= S->nsites || q >= S->nsites || p == q) return fail(QBGPU_ERR_ARG, "sector_matfree_heisenberg: bad bond");
        bs.push_back({std::min(p, q), std::max(p, q)});
    }
    std::stable_sort(bs.begin(), bs.end());                             // the term order of the stored assembly (diagonal sums bit for bit)
    SecTerms T;
    memset(&T, 0, sizeof(T));
    T.nterms = nbonds; T.J = J; T.fake_pos = fake_pos;
    for (int t = 0; t < nbonds; t++) { T.p[t] = (uint8_t)bs[t].first; T.q[t] = (uint8_t)bs[t].second; }
    auto *M = new SecMatFree;
    M->dev = S->dev; M->phase = S->d_phase;
    if (cudaMalloc(&M->d_T, sizeof(SecTerms)) != cudaSuccess) { delete M; return cuda_fail(cudaGetLastError(), "cudaMalloc(terms)", __FILE__, __LINE__); }
    if (cudaMemcpyAsync(M->d_T, &T, sizeof(SecTerms), cudaMemcpyHostToDevice, c.stream) != cudaSuccess || cudaStreamSynchronize(c.stream) != cudaSuccess) {
        cudaFree(M->d_T); delete M; return cuda_fail(cudaGetLastError(), "upload(terms)", __FILE__, __LINE__);
    }
    auto *H = new qbgpu_matrix;
    H->n = S->n; H->row_lo = 0; H->row_hi = S->n; H->api_complex = true; H->val_real = false;
    H->format = QBGPU_FORMAT_MATFREE; H->nnz = 0; H->nnz_input = 0;
    H->mf_sec = M;
    *A = H;
    return QBGPU_OK;
}

/* generate_Ham_sparse_repr (src/model.cc:688-836) for the single-orbital Hubbard model on an electron sector:
 * H = -t sum_hops c+_{to,s} c_{from,s} + U sum_i n_up,i n_dn,i.  hops[3*nhops] = (to, from, spin) DIRECTED, in the order the
 * caller's add_Ham calls insert them (the reference's example: per bond c+_up,i c_up,j ; c+_up,j c_up,i ; c+_dn,i c_dn,j ;
 * c+_dn,j c_dn,i); they are re-ordered here like mopr::operator+= does (src/operators.cc:901-925: ascending (lower site, higher
 * site), equal keys in REVERSE order of insertion) because the accumulation order decides the last bits and lil_mat's erase rule. */
int qbgpu_sector_build_hubbard(qbgpu_sector_t S, qbgpu_matrix_t *A, int nhops, const int32_t *hops, double t, double U, double fake_pos, int flags)
{
    if (!S || !A || !hops || nhops < 1) return fail(QBGPU_ERR_ARG, "sector_build_hubbard: bad arguments");
    if (!S->electron) return fail(QBGPU_ERR_STATE, "sector_build_hubbard: needs an electron sector (qbgpu_sector_create_electron)");
    if (nhops > kMaxHops) return fail(QBGPU_ERR_ARG, "sector_build_hubbard: at most 256 directed hops");
    Context &c = ctx();
    *A = nullptr;
    std::vector<int> order(nhops);
    for (int q = 0; q < nhops; q++) {
        const int to = hops[3 * q], fr = hops[3 * q + 1], sp = hops[3 * q + 2];
        if (to < 0 || fr < 0 || to >= S->nsites || fr >= S->nsites || to == fr || sp < 0 || sp > 1) return fail(QBGPU_ERR_ARG, "sector_build_hubbard: bad hop");
        order[q] = q;
    }
    std::sort(order.begin(), order.end(), [&](int x, int y) {
        const int lx = std::min(hops[3 * x], hops[3 * x + 1]), hx = std::max(hops[3 * x], hops[3 * x + 1]);
        const int ly = std::min(hops[3 * y], hops[3 * y + 1]), hy = std::max(hops[3 * y], hops[3 * y + 1]);
        if (lx != ly) return lx < ly;
        if (hx != hy) return hx < hy;
        return x > y;                                                   // equal keys: the later insertion comes first
    });
    ElTerms T;
    memset(&T, 0, sizeof(T));
    T.nterms = nhops; T.t = t; T.U = U; T.fake_pos = fake_pos;
    for (int pos = 0; pos < nhops; pos++) { const int q = order[pos]; T.to[pos] = (uint8_t)hops[3 * q]; T.from[pos] = (uint8_t)hops[3 * q + 1]; T.sp[pos] = (uint8_t)hops[3 * q + 2]; }

    ElTerms *d_T = nullptr;
    int64_t *d_cap = nullptr, *d_start = nullptr, *d_end = nullptr, *d_col = nullptr, *d_sum = nullptr;
    double2 *d_val = nullptr;
    void *d_tmp = nullptr;
    auto cleanup = [&]() { cudaFree(d_T); cudaFree(d_cap); cudaFree(d_start); cudaFree(d_end); cudaFree(d_col); cudaFree(d_val); cudaFree(d_tmp); cudaFree(d_sum); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    const int64_t n = S->n;
    QB_CU(cudaMalloc(&d_T, sizeof(ElTerms)));
    QB_CU(cudaMemcpyAsync(d_T, &T, sizeof(ElTerms), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMalloc(&d_cap, sizeof(int64_t) * (n + 1)));
    QB_CU(cudaMalloc(&d_start, sizeof(int64_t) * (n + 1)));
    QB_CU(cudaMalloc(&d_end, sizeof(int64_t) * (n + 1)));
    el_cap_kernel<<<sgrid(n + 1), kSBlock, 0, c.stream>>>(S->dev, d_T, d_cap);
    QB_LAUNCH_COUNT();
    size_t tb = 0;
    QB_CU(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_cap, d_start, n + 1, c.stream));
    QB_CU(cudaMalloc(&d_tmp, tb ? tb : 1));
    QB_CU(cub::DeviceScan::ExclusiveSum(d_tmp, tb, d_cap, d_start, n + 1, c.stream));
    int64_t total = 0;
    QB_CU(cudaMemcpyAsync(&total, d_start + n, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaMalloc(&d_col, sizeof(int64_t) * (size_t)total));
    QB_CU(cudaMalloc(&d_val, sizeof(double2) * (size_t)total));
    el_rows_kernel<<<sgrid(n), kSBlock, 0, c.stream>>>(S->dev, d_T, S->d_phase, d_start, d_end, d_col, d_val);
    QB_LAUNCH_COUNT();
    sec_len_kernel<<<sgrid(n), kSBlock, 0, c.stream>>>(n, d_start, d_end, d_cap);
    QB_LAUNCH_COUNT();
    cudaFree(d_tmp); d_tmp = nullptr;
    QB_CU(cudaMalloc(&d_sum, sizeof(int64_t)));
    QB_CU(cub::DeviceReduce::Sum(nullptr, tb, d_cap, d_sum, n, c.stream));
    QB_CU(cudaMalloc(&d_tmp, tb ? tb : 1));
    QB_CU(cub::DeviceReduce::Sum(d_tmp, tb, d_cap, d_sum, n, c.stream));
    int64_t upper = 0;
    QB_CU(cudaMemcpyAsync(&upper, d_sum, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
#undef QB_CU
    int rc = create_from_device_csr(A, n, d_start, d_end, d_col, d_val, true, upper, 1, flags, true);
    cleanup();
    return rc;
}

}  // extern "C"
