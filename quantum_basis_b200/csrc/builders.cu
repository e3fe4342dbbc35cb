// quantum_basis_b200/csrc/builders.cu -- on-device Hamiltonian generators in the reference's Lin-table order.
//
// The reference enumerates the basis on the host (src/basis.cc:998-1110), orders it by (label of the odd-numbered
// sites, label of the even-numbered sites) -- the Lin-table convention, src/basis.cc:1144-1190, labels from
// mbasis_elem::label_sub, src/basis.cc:428-450 -- and assembles H row by row by applying every Hamiltonian term
// to the row's basis state (model::generate_Ham_sparse_full, src/model.cc:619-686; fermion signs from oprXphi,
// src/basis.cc:2717-2731: parity of the fermions on sites below the operator's site, operators applied right to
// left).  At the BASELINE sizes that assembler cannot run (SURVEY F6: > 140 GB of LIL nodes for the 4x4 Hubbard
// model), so the same matrix is generated here directly in its expanded device layout: one thread per row
// re-derives the row's basis state from its index (binary search in the Jb table + class-list lookup), applies
// the bond terms with bit operations, looks the columns up through the same Ja/Jb tables, and sorts the row.
// tests/test_builders.py checks the result entry for entry against matrices assembled by the compiled reference.
#include "internal.hpp"
#include "lin_tables.hpp"
#include <cub/device/device_scan.cuh>
#include <algorithm>
#include <chrono>
#include <cstring>
#include <vector>

namespace qb {

static double wall_b() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

constexpr int kBBlock = 128;

// Tables describing the sector.  Site s lives on sublattice A (even s, position s/2) or B (odd s, position s/2);
// a sublattice label packs `bps` bits per site (bps = 1: spin-1/2 digit; bps = 2: electron digit = up + 2*dn).
struct SectorTables {
    int nsites, bps, nA, nB;
    int t0, t1;                       // conserved counts: (#digit-1 sites, 0) for spins, (N_up, N_dn) for electrons
    int64_t dim;
    const int64_t *Jb;                // [sizeB + 1] first row index of each B label (Lin_Jb)
    const int32_t *rankA;             // [sizeA] rank of an A label inside its class (Lin_Ja relative to the class)
    const uint32_t *alist;            // A labels grouped by class, ascending inside a class
    const int32_t *class_off;         // [(nA+1)*(nA+1)] offset of class (c0,c1) in alist
    uint32_t sizeB;
};

__host__ __device__ __forceinline__ void label_counts(uint32_t lab, int bps, int &c0, int &c1)
{
    if (bps == 1) { c0 = popc_hd(lab); c1 = 0; }
    else { c0 = popc_hd(lab & 0x55555555u); c1 = popc_hd(lab & 0xAAAAAAAAu); }
}

__host__ __device__ __forceinline__ void unrank_row(const SectorTables &S, int64_t row, uint32_t &la, uint32_t &lb)
{
    // largest lb with Jb[lb] <= row  (empty B labels share their successor's offset and are skipped)
    uint32_t lo = 0, hi = S.sizeB;                          // answer in [lo, hi)
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (S.Jb[mid] <= row) lo = mid; else hi = mid; }
    lb = lo;
    int cb0, cb1;
    label_counts(lb, S.bps, cb0, cb1);
    const int32_t off = S.class_off[(S.t0 - cb0) * (S.nA + 1) + (S.t1 - cb1)];
    la = S.alist[off + (int32_t)(row - S.Jb[lb])];
}

__host__ __device__ __forceinline__ int64_t col_of(const SectorTables &S, uint32_t la, uint32_t lb) { return S.Jb[lb] + S.rankA[la]; }

// parity of the fermions on sites < s (electron digits 0,1,2,3 carry 0,1,1,2 fermions: popcount of the 2-bit digit)
__host__ __device__ __forceinline__ int parity_below(uint32_t la, uint32_t lb, int s)
{
    const int ka = (s + 1) >> 1, kb = s >> 1;               // A sites 0,2,..,<s : ceil(s/2) of them; B sites: floor(s/2)
    const uint32_t ma = ka >= 16 ? 0xFFFFFFFFu : ((1u << (2 * ka)) - 1u);
    const uint32_t mb = kb >= 16 ? 0xFFFFFFFFu : ((1u << (2 * kb)) - 1u);
    return (popc_hd(la & ma) + popc_hd(lb & mb)) & 1;
}

// Enumerate the off-diagonal entries of the row whose basis state is (la, lb); returns the diagonal value.
// emit(col, val) is called once per entry; distinct calls give distinct columns.  Compiled for the host too: the sampled-row
// check of bench.py (qbgpu_debug_rows_host) recomputes rows of the BASELINE-size matrices with exactly this function.
template <class Emit>
__host__ __device__ __forceinline__ double row_entries(const SectorTables &S, const ModelParams &M, uint32_t la, uint32_t lb, Emit emit)
{
    double diag = 0.0;
    if (M.kind == 0) {
        // H = sum_b J (S_i.S_j): diagonal J*Sz_i*Sz_j (digit 0 -> +1/2, 1 -> -1/2); off-diagonal J/2 on antiparallel pairs
        for (int b = 0; b < M.nbonds; b++) {
            const int i = M.bonds[b].i, j = M.bonds[b].j;
            const uint32_t bi = 1u << (i >> 1), bj = 1u << (j >> 1);
            const int di = ((i & 1) ? lb : la) & bi ? 1 : 0;
            const int dj = ((j & 1) ? lb : la) & bj ? 1 : 0;
            const double zz = (di == dj) ? 0.25 * M.J : -0.25 * M.J;
            double off = 0.0;
            for (int r = 0; r < M.bonds[b].w; r++) { diag += zz; off += 0.5 * M.J; }
            if (di != dj) {
                uint32_t na = la, nb = lb;
                if (i & 1) nb ^= bi; else na ^= bi;
                if (j & 1) nb ^= bj; else na ^= bj;
                emit(col_of(S, na, nb), off);
            }
        }
    } else {
        // H = -t sum_{b,s} (c+_is c_js + h.c.) + U sum_i n_up n_dn ; digit = up + 2*dn
        const uint32_t dbl = (la & (la >> 1) & 0x55555555u);
        const uint32_t dbl_b = (lb & (lb >> 1) & 0x55555555u);
        const int ndbl = popc_hd(dbl) + popc_hd(dbl_b);
        for (int r = 0; r < ndbl; r++) diag += M.U;
        for (int b = 0; b < M.nbonds; b++) {
            double amp = 0.0;
            for (int r = 0; r < M.bonds[b].w; r++) amp += -M.t;
            for (int dir = 0; dir < 2; dir++) {
                const int to = dir ? M.bonds[b].j : M.bonds[b].i, from = dir ? M.bonds[b].i : M.bonds[b].j;
                for (int sp = 0; sp < 2; sp++) {            // sp 0: up (bit 0 of the digit), 1: dn (bit 1)
                    const uint32_t bf = 1u << (2 * (from >> 1) + sp), bt = 1u << (2 * (to >> 1) + sp);
                    const uint32_t lf = (from & 1) ? lb : la, lt = (to & 1) ? lb : la;
                    if (!(lf & bf) || (lt & bt)) continue;
                    // c_{from,sp}: sign from fermions below `from`; local element -1 for c_dn on a doubly occupied site
                    int sg = parity_below(la, lb, from);
                    if (sp == 1 && (lf & (1u << (2 * (from >> 1))))) sg ^= 1;
                    uint32_t na = la, nb = lb;
                    if (from & 1) nb ^= bf; else na ^= bf;
                    // c+_{to,sp} on the intermediate state
                    sg ^= parity_below(na, nb, to);
                    const uint32_t lt2 = (to & 1) ? nb : na;
                    if (sp == 1 && (lt2 & (1u << (2 * (to >> 1))))) sg ^= 1;
                    if (to & 1) nb ^= bt; else na ^= bt;
                    emit(col_of(S, na, nb), sg ? -amp : amp);
                }
            }
        }
    }
    return diag;
}

__global__ void __launch_bounds__(kBBlock) build_count_kernel(SectorTables S, const ModelParams *Mp, int64_t row_lo, int64_t nloc, int64_t *len)
{
    __shared__ ModelParams M;
    for (int k = threadIdx.x; k < (int)(sizeof(ModelParams) / 4); k += blockDim.x) ((int *)&M)[k] = ((const int *)Mp)[k];
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= nloc; r += (int64_t)gridDim.x * blockDim.x) {
        if (r == nloc) { len[r] = 0; continue; }
        uint32_t la, lb;
        unrank_row(S, row_lo + r, la, lb);
        int cnt = 1;                                        // the diagonal is always stored (src/sparse.cc:44-54)
        row_entries(S, M, la, lb, [&](int64_t, double) { cnt++; });
        len[r] = cnt;
    }
}

template <typename ValT>
__global__ void __launch_bounds__(kBBlock) build_fill_kernel(SectorTables S, const ModelParams *Mp, int64_t row_lo, int64_t nloc,
                                                             const int64_t *__restrict__ rowptr, int32_t *col, ValT *val)
{
    __shared__ ModelParams M;
    for (int k = threadIdx.x; k < (int)(sizeof(ModelParams) / 4); k += blockDim.x) ((int *)&M)[k] = ((const int *)Mp)[k];
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nloc; r += (int64_t)gridDim.x * blockDim.x) {
        uint32_t la, lb;
        unrank_row(S, row_lo + r, la, lb);
        const int64_t s = rowptr[r];
        int cnt = 1;
        auto put = [&](int64_t at, int32_t c, double v) {
            col[at] = c;
            if constexpr (sizeof(ValT) == 16) val[at] = make_double2(v, 0.0); else val[at] = v;
        };
        // insertion into the sorted prefix of the row (rows are short: 1 + number of active bond terms)
        auto insert = [&](int64_t c64, double v) {
            const int32_t c = (int32_t)c64;
            int64_t p = s + cnt - 1;
            while (p >= s && col[p] > c) { col[p + 1] = col[p]; val[p + 1] = val[p]; p--; }
            put(p + 1, c, v);
            cnt++;
        };
        put(s, (int32_t)(row_lo + r), 0.0);                 // diagonal placeholder, value patched below
        const double diag = row_entries(S, M, la, lb, insert);
        for (int64_t p = s; p < s + cnt; p++)
            if (col[p] == (int32_t)(row_lo + r)) { put(p, (int32_t)(row_lo + r), diag); break; }
    }
}

// ------------------------------------------------------------------------------------------ host-side tables
static void counts_host(uint32_t lab, int bps, int &c0, int &c1)
{
    if (bps == 1) { c0 = __builtin_popcount(lab); c1 = 0; }
    else { c0 = __builtin_popcount(lab & 0x55555555u); c1 = __builtin_popcount(lab & 0xAAAAAAAAu); }
}

int make_tables(int nsites, int bps, int t0, int t1, HostTables &T)
{
    T.nsites = nsites; T.bps = bps; T.nA = (nsites + 1) / 2; T.nB = nsites / 2; T.t0 = t0; T.t1 = t1;
    if (bps * T.nA > 24) return fail(QBGPU_ERR_ARG, "builder: sublattice label too wide (max 24 bits per sublattice)");
    const uint32_t sizeA = 1u << (bps * T.nA), sizeB = 1u << (bps * T.nB);
    const int nc = T.nA + 1;
    std::vector<int32_t> csize(nc * nc, 0);
    T.rankA.assign(sizeA, -1);
    for (uint32_t a = 0; a < sizeA; a++) { int c0, c1; counts_host(a, bps, c0, c1); T.rankA[a] = csize[c0 * nc + c1]++; }
    T.class_off.assign(nc * nc, 0);
    int32_t acc = 0;
    for (int k = 0; k < nc * nc; k++) { T.class_off[k] = acc; acc += csize[k]; }
    T.alist.assign(sizeA, 0);
    for (uint32_t a = 0; a < sizeA; a++) { int c0, c1; counts_host(a, bps, c0, c1); T.alist[T.class_off[c0 * nc + c1] + T.rankA[a]] = a; }
    T.Jb.assign((size_t)sizeB + 1, 0);
    int64_t run = 0;
    for (uint32_t b = 0; b < sizeB; b++) {
        T.Jb[b] = run;
        int c0, c1; counts_host(b, bps, c0, c1);
        const int n0 = t0 - c0, n1 = t1 - c1;
        if (n0 >= 0 && n0 <= T.nA && n1 >= 0 && n1 <= T.nA && (bps == 2 || n1 == 0)) run += csize[n0 * nc + n1];
    }
    T.Jb[sizeB] = run;
    T.dim = run;
    return QBGPU_OK;
}

int merge_bonds(int nsites, int nbonds, const int32_t *bonds, ModelParams &M)
{
    M.nbonds = 0;
    for (int b = 0; b < nbonds; b++) {
        int i = bonds[2 * b], j = bonds[2 * b + 1];
        if (i < 0 || j < 0 || i >= nsites || j >= nsites || i == j) return fail(QBGPU_ERR_ARG, "builder: bad bond");
        bool found = false;
        for (int k = 0; k < M.nbonds; k++)
            if ((M.bonds[k].i == i && M.bonds[k].j == j) || (M.bonds[k].i == j && M.bonds[k].j == i)) { M.bonds[k].w++; found = true; break; }
        if (!found) {
            if (M.nbonds == kMaxBonds) return fail(QBGPU_ERR_ARG, "builder: too many bonds");
            M.bonds[M.nbonds++] = Bond{i, j, 1};
        }
    }
    return QBGPU_OK;
}

static int build_generic(qbgpu_matrix_t *out, const HostTables &T, const ModelParams &M, int api_complex, int flags,
                         int64_t row_lo, int64_t row_hi)
{
    QB_TRY(ensure_init());
    Context &c = ctx();
    if (!out) return fail(QBGPU_ERR_ARG, "null handle pointer");
    *out = nullptr;
    if (T.dim <= 0) return fail(QBGPU_ERR_ARG, "builder: empty sector");
    if (T.dim > 2147483647LL) return fail(QBGPU_ERR_ARG, "builder: dimension exceeds the int32 column range");
    if (row_hi < 0) row_hi = T.dim;
    if (row_lo < 0 || row_lo > row_hi || row_hi > T.dim) return fail(QBGPU_ERR_ARG, "builder: bad row shard");
    const int64_t nloc = row_hi - row_lo;
    const double t0 = wall_b();
    auto *A = new qbgpu_matrix;
    A->n = T.dim; A->row_lo = row_lo; A->row_hi = row_hi; A->api_complex = api_complex != 0;
    A->val_real = !(flags & QBGPU_KEEP_COMPLEX) || !api_complex;

    int64_t *d_Jb = nullptr, *d_len = nullptr;
    int32_t *d_rank = nullptr, *d_off = nullptr;
    uint32_t *d_alist = nullptr;
    ModelParams *d_M = nullptr;
    void *d_tmp = nullptr;
    auto cleanup = [&]() { cudaFree(d_Jb); cudaFree(d_len); cudaFree(d_rank); cudaFree(d_off); cudaFree(d_alist); cudaFree(d_M); cudaFree(d_tmp); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); qbgpu_destroy(A); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&d_Jb, sizeof(int64_t) * T.Jb.size()));
    QB_CU(cudaMalloc(&d_rank, sizeof(int32_t) * T.rankA.size()));
    QB_CU(cudaMalloc(&d_alist, sizeof(uint32_t) * T.alist.size()));
    QB_CU(cudaMalloc(&d_off, sizeof(int32_t) * T.class_off.size()));
    QB_CU(cudaMalloc(&d_M, sizeof(ModelParams)));
    QB_CU(cudaMemcpyAsync(d_Jb, T.Jb.data(), sizeof(int64_t) * T.Jb.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_rank, T.rankA.data(), sizeof(int32_t) * T.rankA.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_alist, T.alist.data(), sizeof(uint32_t) * T.alist.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_off, T.class_off.data(), sizeof(int32_t) * T.class_off.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_M, &M, sizeof(ModelParams), cudaMemcpyHostToDevice, c.stream));
    SectorTables S;
    S.nsites = T.nsites; S.bps = T.bps; S.nA = T.nA; S.nB = T.nB; S.t0 = T.t0; S.t1 = T.t1; S.dim = T.dim;
    S.Jb = d_Jb; S.rankA = d_rank; S.alist = d_alist; S.class_off = d_off; S.sizeB = (uint32_t)(T.Jb.size() - 1);

    QB_CU(cudaMalloc(&d_len, sizeof(int64_t) * (nloc + 1)));
    QB_CU(cudaMalloc(&A->rowptr, sizeof(int64_t) * (nloc + 1)));
    int64_t g = (nloc + 1 + kBBlock - 1) / kBBlock;
    if (g > 148 * 64) g = 148 * 64;
    build_count_kernel<<<(int)g, kBBlock, 0, c.stream>>>(S, d_M, row_lo, nloc, d_len);
    QB_LAUNCH_COUNT();
    size_t tmp_bytes = 0;
    QB_CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_len, A->rowptr, nloc + 1, c.stream));
    QB_CU(cudaMalloc(&d_tmp, tmp_bytes ? tmp_bytes : 1));
    QB_CU(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_len, A->rowptr, nloc + 1, c.stream));
    int64_t nnz = 0;
    QB_CU(cudaMemcpyAsync(&nnz, A->rowptr + nloc, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    A->nnz = nnz;
    A->nnz_input = (nnz + T.dim) / 2;                       // what the reference would store (upper triangle incl. diagonal), full handle
    QB_CU(cudaMalloc(&A->col, sizeof(int32_t) * (nnz ? nnz : 1) + 64));
    QB_CU(cudaMalloc(&A->val, A->val_bytes() * (nnz ? nnz : 1) + 64));
    if (A->val_real) build_fill_kernel<double><<<(int)g, kBBlock, 0, c.stream>>>(S, d_M, row_lo, nloc, A->rowptr, A->col, (double *)A->val);
    else             build_fill_kernel<double2><<<(int)g, kBBlock, 0, c.stream>>>(S, d_M, row_lo, nloc, A->rowptr, A->col, (double2 *)A->val);
    QB_LAUNCH_COUNT();
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
    cleanup();
#undef QB_CU
    A->convert_s = wall_b() - t0;
    { int rc = autotune(A, flags); if (rc) { qbgpu_destroy(A); return rc; } }
    *out = A;
    return QBGPU_OK;
}


// ------------------------------------------------------------------------------------ Lin order -> species order
// perm[r] for the species-order handles of species.cu: row r of the reference's Lin order is the electron state (la, lb);
// its up / down occupancy words (site-indexed) are ranked among the words of equal popcount.
__host__ __device__ __forceinline__ int32_t species_index_of_row(const SectorTables &S, int64_t r, const int32_t *rank_in_class, int64_t Dd)
{
    uint32_t la, lb;
    unrank_row(S, r, la, lb);
    const uint32_t occ0 = (la & 0x55555555u) | ((lb & 0x55555555u) << 1);              // same words as row_entries_walk
    const uint32_t occ1 = ((la >> 1) & 0x55555555u) | (lb & 0xAAAAAAAAu);
    return (int32_t)((int64_t)rank_in_class[occ0] * Dd + rank_in_class[occ1]);
}

__global__ void __launch_bounds__(kBBlock) species_perm_kernel(SectorTables S, int64_t n, const int32_t *__restrict__ rank_in_class, int64_t Dd, int32_t *perm)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x)
        perm[r] = species_index_of_row(S, r, rank_in_class, Dd);
}

// the same row function on the host (qbgpu_debug_species_host: CPU tests of the index logic, no device involved)
void species_perm_host(const HostTables &T, const int32_t *rank_in_class, int64_t Dd, int32_t *perm)
{
    SectorTables S;
    S.nsites = T.nsites; S.bps = T.bps; S.nA = T.nA; S.nB = T.nB; S.t0 = T.t0; S.t1 = T.t1; S.dim = T.dim;
    S.Jb = T.Jb.data(); S.rankA = T.rankA.data(); S.alist = T.alist.data(); S.class_off = T.class_off.data(); S.sizeB = (uint32_t)(T.Jb.size() - 1);
    for (int64_t r = 0; r < T.dim; r++) perm[r] = species_index_of_row(S, r, rank_in_class, Dd);
}

int species_perm_build(const HostTables &T, const int32_t *d_rank_in_class, int64_t Dd, int32_t *d_perm)
{
    Context &c = ctx();
    if (T.bps != 2) return fail(QBGPU_ERR_ARG, "species order: electron sectors only");
    int64_t *d_Jb = nullptr;
    int32_t *d_rank = nullptr, *d_off = nullptr;
    uint32_t *d_alist = nullptr;
    auto cleanup = [&]() { cudaFree(d_Jb); cudaFree(d_rank); cudaFree(d_off); cudaFree(d_alist); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&d_Jb, sizeof(int64_t) * T.Jb.size()));
    QB_CU(cudaMalloc(&d_rank, sizeof(int32_t) * T.rankA.size()));
    QB_CU(cudaMalloc(&d_alist, sizeof(uint32_t) * T.alist.size()));
    QB_CU(cudaMalloc(&d_off, sizeof(int32_t) * T.class_off.size()));
    QB_CU(cudaMemcpyAsync(d_Jb, T.Jb.data(), sizeof(int64_t) * T.Jb.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_rank, T.rankA.data(), sizeof(int32_t) * T.rankA.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_alist, T.alist.data(), sizeof(uint32_t) * T.alist.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_off, T.class_off.data(), sizeof(int32_t) * T.class_off.size(), cudaMemcpyHostToDevice, c.stream));
    SectorTables S;
    S.nsites = T.nsites; S.bps = T.bps; S.nA = T.nA; S.nB = T.nB; S.t0 = T.t0; S.t1 = T.t1; S.dim = T.dim;
    S.Jb = d_Jb; S.rankA = d_rank; S.alist = d_alist; S.class_off = d_off; S.sizeB = (uint32_t)(T.Jb.size() - 1);
    int64_t g = (T.dim + kBBlock - 1) / kBBlock;
    if (g < 1) g = 1;
    if (g > 148 * 64) g = 148 * 64;
    species_perm_kernel<<<(int)g, kBBlock, 0, c.stream>>>(S, T.dim, d_rank_in_class, Dd, d_perm);
    QB_LAUNCH_COUNT();
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
#undef QB_CU
    cleanup();
    return QBGPU_OK;
}

// the inverse on a row range of the species order: out[p - lo] = the reference's row r with species index p, lo <= p < hi
__global__ void __launch_bounds__(kBBlock) species_ref_rows_kernel(SectorTables S, int64_t n, const int32_t *__restrict__ rank_in_class, int64_t Dd,
                                                                   int64_t lo, int64_t hi, int32_t *out)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = species_index_of_row(S, r, rank_in_class, Dd);
        if (p >= lo && p < hi) out[p - lo] = (int32_t)r;
    }
}

int species_ref_rows_build(const HostTables &T, const int32_t *d_rank_in_class, int64_t Dd, int64_t lo, int64_t hi, int32_t *d_out)
{
    Context &c = ctx();
    if (T.bps != 2) return fail(QBGPU_ERR_ARG, "species order: electron sectors only");
    int64_t *d_Jb = nullptr;
    int32_t *d_rank = nullptr, *d_off = nullptr;
    uint32_t *d_alist = nullptr;
    auto cleanup = [&]() { cudaFree(d_Jb); cudaFree(d_rank); cudaFree(d_off); cudaFree(d_alist); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&d_Jb, sizeof(int64_t) * T.Jb.size()));
    QB_CU(cudaMalloc(&d_rank, sizeof(int32_t) * T.rankA.size()));
    QB_CU(cudaMalloc(&d_alist, sizeof(uint32_t) * T.alist.size()));
    QB_CU(cudaMalloc(&d_off, sizeof(int32_t) * T.class_off.size()));
    QB_CU(cudaMemcpyAsync(d_Jb, T.Jb.data(), sizeof(int64_t) * T.Jb.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_rank, T.rankA.data(), sizeof(int32_t) * T.rankA.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_alist, T.alist.data(), sizeof(uint32_t) * T.alist.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_off, T.class_off.data(), sizeof(int32_t) * T.class_off.size(), cudaMemcpyHostToDevice, c.stream));
    SectorTables S;
    S.nsites = T.nsites; S.bps = T.bps; S.nA = T.nA; S.nB = T.nB; S.t0 = T.t0; S.t1 = T.t1; S.dim = T.dim;
    S.Jb = d_Jb; S.rankA = d_rank; S.alist = d_alist; S.class_off = d_off; S.sizeB = (uint32_t)(T.Jb.size() - 1);
    int64_t g = (T.dim + kBBlock - 1) / kBBlock;
    if (g < 1) g = 1;
    if (g > 148 * 64) g = 148 * 64;
    species_ref_rows_kernel<<<(int)g, kBBlock, 0, c.stream>>>(S, T.dim, d_rank_in_class, Dd, lo, hi, d_out);
    QB_LAUNCH_COUNT();
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
#undef QB_CU
    cleanup();
    return QBGPU_OK;
}

// ------------------------------------------------------------------------------------------------ matrix-free
// Neighbour tables for the matrix-free kernel: instead of testing every (bond, direction, spin) -- 128 tests per row on
// the 4x4 lattice, a quarter of which fire -- the kernel walks the set bits of "occupied site" words and, for each,
// the set bits of (neighbours of that site) & ~occupied, so that the number of trips equals the number of entries.
struct SiteTables {
    int nsites;
    uint32_t nbr[32];            // nbr[f]: bit t set when sites f and t share a bond
    uint8_t wgt[32][32];         // bond multiplicity (duplicates in the caller's list are merged)
    int wbonds;                  // sum of multiplicities (for the Heisenberg diagonal)
};

// bit k -> bit 2k (k < 16)
__host__ __device__ __forceinline__ uint32_t spread16(uint32_t x)
{
    x &= 0xFFFFu;
    x = (x | (x << 8)) & 0x00FF00FFu;
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x;
}

// Entries of the row of basis state (la, lb), generated in neighbour-walk order; returns the diagonal.
template <class Emit>
__device__ __forceinline__ double row_entries_walk(const SectorTables &S, const ModelParams &M, const SiteTables &N, uint32_t la, uint32_t lb, Emit emit)
{
    if (M.kind == 0) {
        // site-indexed "down" word: A-site k is site 2k, B-site k is site 2k+1
        const uint32_t dn = spread16(la) | (spread16(lb) << 1);
        int anti = 0;                                        // weighted number of antiparallel bonds
        uint32_t m = dn;
        while (m) {
            const int f = __ffs(m) - 1; m &= m - 1;
            uint32_t cand = N.nbr[f] & ~dn;
            while (cand) {
                const int t = __ffs(cand) - 1; cand &= cand - 1;
                const int w = N.wgt[f][t];
                anti += w;
                uint32_t na = la, nb = lb;
                if (f & 1) nb ^= 1u << (f >> 1); else na ^= 1u << (f >> 1);
                if (t & 1) nb ^= 1u << (t >> 1); else na ^= 1u << (t >> 1);
                emit(col_of(S, na, nb), 0.5 * M.J * w);
            }
        }
        return 0.25 * M.J * (double)(N.wbonds - 2 * anti);
    }
    // electrons: digit = up + 2*dn at bit pair k of a sublattice label; site-indexed occupancy words per spin
    const uint32_t occ0 = (la & 0x55555555u) | ((lb & 0x55555555u) << 1);
    const uint32_t occ1 = ((la >> 1) & 0x55555555u) | (lb & 0xAAAAAAAAu);
    const int ndbl = __popc(occ0 & occ1);
    double diag = 0.0;
    for (int r = 0; r < ndbl; r++) diag += M.U;
#pragma unroll
    for (int sp = 0; sp < 2; sp++) {
        const uint32_t occ = sp ? occ1 : occ0;
        uint32_t m = occ;
        while (m) {
            const int f = __ffs(m) - 1; m &= m - 1;
            uint32_t cand = N.nbr[f] & ~occ;
            // c_{f,sp}: fermions on sites below f (both spins); c_dn next to an up electron on the same site: -1
            const uint32_t below_f = (1u << f) - 1u;
            const int sg_f = (__popc(occ0 & below_f) + __popc(occ1 & below_f) + (sp == 1 ? (int)((occ0 >> f) & 1u) : 0)) & 1;
            while (cand) {
                const int t = __ffs(cand) - 1; cand &= cand - 1;
                // c+_{t,sp} on the state with (f,sp) removed
                const uint32_t below_t = (1u << t) - 1u;
                int sg = sg_f + __popc(occ0 & below_t) + __popc(occ1 & below_t) + (sp == 1 ? (int)((occ0 >> t) & 1u) : 0);
                if (f < t) sg += 1;                          // the removed electron sat below t
                uint32_t na = la, nb = lb;
                if (f & 1) nb ^= 1u << (2 * (f >> 1) + sp); else na ^= 1u << (2 * (f >> 1) + sp);
                if (t & 1) nb ^= 1u << (2 * (t >> 1) + sp); else na ^= 1u << (2 * (t >> 1) + sp);
                double amp = 0.0;
                for (int r = 0; r < N.wgt[f][t]; r++) amp += -M.t;
                emit(col_of(S, na, nb), (sg & 1) ? -amp : amp);
            }
        }
    }
    return diag;
}

// ------------------------------------------------------------------ one-site diagonal operators in the full basis
// model::moprXvec_full (src/model.cc:1468-1538) for A = sum_r c_r O_r with O_r diagonal in the site basis -- S^z_r for spins
// (digit 0 = up: +1/2), c0_r n_up,r + c1_r n_dn,r for electrons (S^z_q of the Hubbard model: c1 = -c0) -- on a vector in
// the reference's Lin order: y_j = x_j * sum_r c_r <state_j| O_r |state_j>, rows with |x_j| < lanczos_precision skipped
// (:1500).  With measure_full_dynamic's normalisation and qbgpu_lanczos_z(..., "dnmcs") this is src/model.cc:1697-1712, the
// dynamic part of the reference's examples/trans_absent/latt_square/square_Fermi_Hubbard.cc.
__host__ __device__ __forceinline__ double2 onsite_diag_weight(const SectorTables &S, int64_t r, const double2 *c0, const double2 *c1)
{
    uint32_t la, lb;
    unrank_row(S, r, la, lb);
    double2 w = make_double2(0.0, 0.0);
    if (S.bps == 1) {
        const uint32_t dn = spread16(la) | (spread16(lb) << 1);                          // bit s set = site s down
        for (int s = 0; s < S.nsites; s++) {
            const double sz = ((dn >> s) & 1u) ? -0.5 : 0.5;
            w.x += c0[s].x * sz; w.y += c0[s].y * sz;
        }
    } else {
        const uint32_t occ0 = (la & 0x55555555u) | ((lb & 0x55555555u) << 1);              // same words as row_entries_walk
        const uint32_t occ1 = ((la >> 1) & 0x55555555u) | (lb & 0xAAAAAAAAu);
        for (int s = 0; s < S.nsites; s++) {
            if ((occ0 >> s) & 1u) { w.x += c0[s].x; w.y += c0[s].y; }
            if ((occ1 >> s) & 1u) { w.x += c1[s].x; w.y += c1[s].y; }
        }
    }
    return w;
}

__global__ void __launch_bounds__(kBBlock) full_apply_diag_kernel(SectorTables S, int64_t n, const double2 *__restrict__ c0g, const double2 *__restrict__ c1g,
                                                                  const double2 *__restrict__ x, double2 *y)
{
    __shared__ double2 c0[32], c1[32];
    if (threadIdx.x < 32) { c0[threadIdx.x] = c0g[threadIdx.x]; c1[threadIdx.x] = c1g[threadIdx.x]; }
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
        const double2 xj = x[r];
        double2 out = make_double2(0.0, 0.0);
        if (hypot(xj.x, xj.y) >= 2e-12) {
            const double2 w = onsite_diag_weight(S, r, c0, c1);
            out = make_double2(xj.x * w.x - xj.y * w.y, xj.x * w.y + xj.y * w.x);
        }
        y[r] = out;
    }
}

// host == true: the same row function on host arrays (CPU tests), nothing touches the device
static int full_apply_diag(int kind, int nsites, int n0, int n1, const double *c0_reim, const double *c1_reim, const void *x, void *y, bool host)
{
    if (nsites < 2 || nsites > 32 || !c0_reim || !x || !y || (kind == 1 && !c1_reim) || (kind != 0 && kind != 1))
        return fail(QBGPU_ERR_ARG, "full_apply_diag: bad argument");
    HostTables T;
    QB_TRY(make_tables(nsites, kind == 0 ? 1 : 2, n0, kind == 0 ? 0 : n1, T));
    if (T.dim <= 0) return fail(QBGPU_ERR_ARG, "full_apply_diag: empty sector");
    double2 c0[32], c1[32];
    for (int s = 0; s < 32; s++) {
        c0[s] = s < nsites ? make_double2(c0_reim[2 * s], c0_reim[2 * s + 1]) : make_double2(0.0, 0.0);
        c1[s] = (s < nsites && kind == 1) ? make_double2(c1_reim[2 * s], c1_reim[2 * s + 1]) : make_double2(0.0, 0.0);
    }
    SectorTables S;
    S.nsites = T.nsites; S.bps = T.bps; S.nA = T.nA; S.nB = T.nB; S.t0 = T.t0; S.t1 = T.t1; S.dim = T.dim;
    S.sizeB = (uint32_t)(T.Jb.size() - 1);
    if (host) {
        S.Jb = T.Jb.data(); S.rankA = T.rankA.data(); S.alist = T.alist.data(); S.class_off = T.class_off.data();
        const double2 *xs = (const double2 *)x;
        double2 *ys = (double2 *)y;
        for (int64_t r = 0; r < T.dim; r++) {
            const double2 xj = xs[r];
            double2 out = make_double2(0.0, 0.0);
            if (hypot(xj.x, xj.y) >= 2e-12) {
                const double2 w = onsite_diag_weight(S, r, c0, c1);
                out = make_double2(xj.x * w.x - xj.y * w.y, xj.x * w.y + xj.y * w.x);
            }
            ys[r] = out;
        }
        return QBGPU_OK;
    }
    QB_TRY(ensure_init());
    Context &c = ctx();
    int64_t *d_Jb = nullptr;
    int32_t *d_rank = nullptr, *d_off = nullptr;
    uint32_t *d_alist = nullptr;
    double2 *d_c = nullptr;
    auto cleanup = [&]() { cudaFree(d_Jb); cudaFree(d_rank); cudaFree(d_off); cudaFree(d_alist); cudaFree(d_c); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&d_Jb, sizeof(int64_t) * T.Jb.size()));
    QB_CU(cudaMalloc(&d_rank, sizeof(int32_t) * T.rankA.size()));
    QB_CU(cudaMalloc(&d_alist, sizeof(uint32_t) * T.alist.size()));
    QB_CU(cudaMalloc(&d_off, sizeof(int32_t) * T.class_off.size()));
    QB_CU(cudaMalloc(&d_c, sizeof(double2) * 64));
    QB_CU(cudaMemcpyAsync(d_Jb, T.Jb.data(), sizeof(int64_t) * T.Jb.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_rank, T.rankA.data(), sizeof(int32_t) * T.rankA.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_alist, T.alist.data(), sizeof(uint32_t) * T.alist.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_off, T.class_off.data(), sizeof(int32_t) * T.class_off.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_c, c0, sizeof(double2) * 32, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_c + 32, c1, sizeof(double2) * 32, cudaMemcpyHostToDevice, c.stream));
    S.Jb = d_Jb; S.rankA = d_rank; S.alist = d_alist; S.class_off = d_off;
    int64_t g = (T.dim + kBBlock - 1) / kBBlock;
    if (g > 148 * 64) g = 148 * 64;
    full_apply_diag_kernel<<<(int)g, kBBlock, 0, c.stream>>>(S, T.dim, d_c, d_c + 32, (const double2 *)x, (double2 *)y);
    QB_LAUNCH_COUNT();
    QB_CU(cudaStreamSynchronize(c.stream));               // c0 / c1 live on this stack frame
    QB_CU(cudaGetLastError());
#undef QB_CU
    cleanup();
    return QBGPU_OK;
}

// The product with no stored matrix: one thread per row (32 consecutive rows per warp, like the sliced-jagged
// kernel, so one Hamiltonian term sends the lanes of a warp to neighbouring columns), the row's entries regenerated by
// row_entries() and consumed at once.  The reference's counterpart is model<T>::MultMv2 with matrix_free == true
// (src/model.cc:942-1109): same per-row recomputation, same Lin-table lookup j = Ja[i_a] + Jb[i_b] (:985-988).
struct MatFree {
    SectorTables S;                 // device pointers into the arrays below
    ModelParams *d_M = nullptr;
    int64_t *d_Jb = nullptr;
    int32_t *d_rank = nullptr, *d_off = nullptr;
    uint32_t *d_alist = nullptr;
    uint2 *d_states = nullptr;      // (la, lb) of every local row
    SiteTables *d_N = nullptr;
    // term-coded variant (QBGPU_MATFREE_TERMS): one byte per entry naming the (directed bond, spin) that produces it, so
    // the product replays the row without searching for the applicable terms.  Codes are packed four to a word and laid
    // out per 32-row slice, word k of every row side by side (padded with 0xFF to the slice's longest row).
    uint32_t *d_codes = nullptr;
    int64_t *d_sliceptr = nullptr;  // [nslices + 1] word offsets
    struct TermTable *d_terms = nullptr;
    int wbonds = 0, kind = 0;
    int64_t bytes = 0;
};

struct TermTable {
    int ncodes;
    uint32_t hop[256];              // f | t << 5 | spin << 10 | weight << 11
    double amp[256];                // Heisenberg: J/2 * weight;  Hubbard: -t added `weight` times (like the LIL accumulation)
    uint8_t code_of[32][32];        // directed pair (f, t) -> code / 2 (Hubbard) or code (Heisenberg)
    // branch-free decode for spmv_terms_kernel_v2: XOR masks on the two sublattice labels and "sites below" masks; the
    // padding code 255 has all-zero masks and amplitude 0, so it replays as "0 * x[own row]"
    uint32_t mask_a[256], mask_b[256], below_f[256], below_t[256];
};

__global__ void __launch_bounds__(kBBlock) matfree_states_kernel(SectorTables S, int64_t row_lo, int64_t nloc, uint2 *states)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nloc; r += (int64_t)gridDim.x * blockDim.x) {
        uint32_t la, lb;
        unrank_row(S, row_lo + r, la, lb);
        states[r] = make_uint2(la, lb);
    }
}

constexpr int kMFBlock = 256;

template <typename VecT, bool DOTS>
__global__ void __launch_bounds__(kMFBlock, 3)
spmv_matfree_kernel(SectorTables S, const ModelParams *Mp, const SiteTables *Np, const uint2 *__restrict__ states, int64_t nrows, int64_t row_lo,
                    const VecT *__restrict__ x, const VecT *z, VecT *y, double2 alpha, double2 gamma, double2 beta,
                    int scal_mode, const double *__restrict__ sc, double *dots_out, double *partials, unsigned *ticket)
{
    using VT = VecTraits<VecT>;
    __shared__ ModelParams M;                               // only the scalars are used here; the bonds live in N
    __shared__ SiteTables N;
    for (int k = threadIdx.x; k < 16; k += blockDim.x) ((int *)&M)[k] = ((const int *)Mp)[k];
    for (int k = threadIdx.x; k < (int)(sizeof(SiteTables) / 4); k += blockDim.x) ((int *)&N)[k] = ((const int *)Np)[k];
    __syncthreads();
    double dot_scale = 1.0;
    if (scal_mode != 0) {
        const double sx = sc[0], sz = sc[1], bprev = sc[2];
        alpha = make_double2(sx, 0.0);
        gamma = make_double2(0.0, 0.0);
        beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
        dot_scale = sx;
    }
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    double d[3] = {0.0, 0.0, 0.0};
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < nrows; row += (int64_t)gridDim.x * blockDim.x) {
        const uint2 st = states[row];
        VecT acc = VT::zero();
        const double diag = row_entries_walk(S, M, N, st.x, st.y, [&](int64_t c, double v) { mac(acc, v, ld_vec(x + c)); });
        const VecT xi = x[row_lo + row];
        mac(acc, diag, xi);
        VecT out = VT::scale(alpha, acc);
        if (gamma.x != 0.0 || gamma.y != 0.0) out = VT::add(out, VT::scale(gamma, xi));
        if (use_beta) out = VT::add(out, VT::scale(beta, z[row]));
        y[row] = out;
        if (DOTS) {
            const double2 p = VT::conj_mul(xi, out);
            d[0] += p.x; d[1] += p.y; d[2] += VT::abs2(out);
        }
    }
    if (DOTS) {
        d[0] *= dot_scale; d[1] *= dot_scale;
        block_reduce_finalize<3, kMFBlock>(d, partials, ticket, dots_out);
    }
}


// ---- term-coded rows -------------------------------------------------------------------------------------------
// count / fill: the neighbour walk once more, recording instead of multiplying
__global__ void __launch_bounds__(kBBlock) terms_count_kernel(SectorTables S, const ModelParams *Mp, const SiteTables *Np, const uint2 *__restrict__ states,
                                                              int64_t nrows, int64_t nslices, int64_t *slice_words)
{
    __shared__ ModelParams M;
    __shared__ SiteTables N;
    for (int k = threadIdx.x; k < 16; k += blockDim.x) ((int *)&M)[k] = ((const int *)Mp)[k];
    for (int k = threadIdx.x; k < (int)(sizeof(SiteTables) / 4); k += blockDim.x) ((int *)&N)[k] = ((const int *)Np)[k];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t wpb = blockDim.x / 32;
    for (int64_t s = (int64_t)blockIdx.x * wpb + (threadIdx.x >> 5); s <= nslices; s += (int64_t)gridDim.x * wpb) {
        int words = 0;
        const int64_t row = s * 32 + lane;
        if (s < nslices && row < nrows) {
            const uint2 st = states[row];
            int cnt = 0;
            row_entries_walk(S, M, N, st.x, st.y, [&](int64_t, double) { cnt++; });
            words = (cnt + 3) >> 2;
        }
        for (int o = 16; o > 0; o >>= 1) words = max(words, __shfl_xor_sync(0xffffffffu, words, o));
        if (lane == 0) slice_words[s] = s < nslices ? (int64_t)words * 32 : 0;
    }
}

// the walk of row_entries_walk, emitting (f, t, spin) instead of (column, value)
template <class Emit>
__device__ __forceinline__ void row_terms_walk(const ModelParams &M, const SiteTables &N, uint32_t la, uint32_t lb, Emit emit)
{
    if (M.kind == 0) {
        const uint32_t dn = spread16(la) | (spread16(lb) << 1);
        uint32_t m = dn;
        while (m) {
            const int f = __ffs(m) - 1; m &= m - 1;
            uint32_t cand = N.nbr[f] & ~dn;
            while (cand) { const int t = __ffs(cand) - 1; cand &= cand - 1; emit(f, t, 0); }
        }
        return;
    }
    const uint32_t occ0 = (la & 0x55555555u) | ((lb & 0x55555555u) << 1);
    const uint32_t occ1 = ((la >> 1) & 0x55555555u) | (lb & 0xAAAAAAAAu);
#pragma unroll
    for (int sp = 0; sp < 2; sp++) {
        const uint32_t occ = sp ? occ1 : occ0;
        uint32_t m = occ;
        while (m) {
            const int f = __ffs(m) - 1; m &= m - 1;
            uint32_t cand = N.nbr[f] & ~occ;
            while (cand) { const int t = __ffs(cand) - 1; cand &= cand - 1; emit(f, t, sp); }
        }
    }
}

__global__ void __launch_bounds__(kBBlock) terms_fill_kernel(const ModelParams *Mp, const SiteTables *Np, const TermTable *Tp, const uint2 *__restrict__ states,
                                                             int64_t nrows, int64_t nslices, const int64_t *__restrict__ sliceptr, uint32_t *codes)
{
    __shared__ ModelParams M;
    __shared__ SiteTables N;
    __shared__ uint8_t code_of[32][32];
    for (int k = threadIdx.x; k < 16; k += blockDim.x) ((int *)&M)[k] = ((const int *)Mp)[k];
    for (int k = threadIdx.x; k < (int)(sizeof(SiteTables) / 4); k += blockDim.x) ((int *)&N)[k] = ((const int *)Np)[k];
    for (int k = threadIdx.x; k < 1024; k += blockDim.x) ((uint8_t *)code_of)[k] = ((const uint8_t *)Tp->code_of)[k];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t wpb = blockDim.x / 32;
    for (int64_t s = (int64_t)blockIdx.x * wpb + (threadIdx.x >> 5); s < nslices; s += (int64_t)gridDim.x * wpb) {
        const int64_t base = sliceptr[s];
        const int maxw = (int)((sliceptr[s + 1] - base) >> 5);
        const int64_t row = s * 32 + lane;
        int k = 0, fill = 0;
        uint32_t word = 0;
        if (row < nrows) {
            const uint2 st = states[row];
            row_terms_walk(M, N, st.x, st.y, [&](int f, int t, int sp) {
                const uint32_t code = M.kind == 0 ? (uint32_t)code_of[f][t] : ((uint32_t)code_of[f][t] * 2u + (uint32_t)sp);
                word |= code << (8 * fill);
                if (++fill == 4) { codes[base + (int64_t)k * 32 + lane] = word; k++; fill = 0; word = 0; }
            });
        }
        if (fill) {                                           // last, partly filled word: pad with 0xFF codes
            for (; fill < 4; fill++) word |= 0xFFu << (8 * fill);
            codes[base + (int64_t)k * 32 + lane] = word; k++;
        }
        for (; k < maxw; k++) codes[base + (int64_t)k * 32 + lane] = 0xFFFFFFFFu;
    }
}

// The product from the term codes: thread = row (32 consecutive rows per warp), four codes per trip.  Nothing in a trip
// depends on a branch: every code -- padding included -- runs the same straight-line decode (XOR masks and "below"
// masks from shared memory), so the compiler issues the eight Lin-table loads of a trip together and then the four
// gathers, and the next trip's code word is fetched a trip ahead.  (A first version decoded behind a divergent
// `if (code != padding)` and chained table loads -> add -> gather per entry: 31.7 ms on config 3 against 28.6 ms for this
// one; profiles/r01_terms_coded_first_run.txt, r01_terms_coded_v2_run.txt.)
template <typename VecT, bool DOTS, int KIND>
__global__ void __launch_bounds__(kMFBlock, 3)
spmv_terms_kernel_v2(SectorTables S, const ModelParams *Mp, const TermTable *Tp, const uint2 *__restrict__ states, const int64_t *__restrict__ sliceptr,
                     const uint32_t *__restrict__ codes, int64_t nrows, int64_t nslices, int64_t row_lo, int wbonds,
                     const VecT *__restrict__ x, const VecT *z, VecT *y, double2 alpha, double2 gamma, double2 beta,
                     int scal_mode, const double *__restrict__ sc, double *dots_out, double *partials, unsigned *ticket)
{
    using VT = VecTraits<VecT>;
    __shared__ ModelParams M;
    __shared__ uint32_t hop[256], mA[256], mB[256], bF[256], bT[256];
    __shared__ double amp[256];
    for (int k = threadIdx.x; k < 16; k += blockDim.x) ((int *)&M)[k] = ((const int *)Mp)[k];
    for (int k = threadIdx.x; k < 256; k += blockDim.x) {
        hop[k] = Tp->hop[k]; amp[k] = Tp->amp[k]; mA[k] = Tp->mask_a[k]; mB[k] = Tp->mask_b[k]; bF[k] = Tp->below_f[k]; bT[k] = Tp->below_t[k];
    }
    __syncthreads();
    double dot_scale = 1.0;
    if (scal_mode != 0) {
        const double sx = sc[0], sz = sc[1], bprev = sc[2];
        alpha = make_double2(sx, 0.0);
        gamma = make_double2(0.0, 0.0);
        beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
        dot_scale = sx;
    }
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    double d[3] = {0.0, 0.0, 0.0};
    const int lane = threadIdx.x & 31;
    constexpr int WPB = kMFBlock / 32;
    for (int64_t s = (int64_t)blockIdx.x * WPB + (threadIdx.x >> 5); s < nslices; s += (int64_t)gridDim.x * WPB) {
        const int64_t base = sliceptr[s];
        const int maxw = (int)((sliceptr[s + 1] - base) >> 5);
        const int64_t row = s * 32 + lane;
        const bool live = row < nrows;
        const uint2 st = live ? states[row] : states[nrows - 1];      // padding lanes replay zeros on a valid state
        const uint32_t la = st.x, lb = st.y;
        const uint32_t occ0 = (la & 0x55555555u) | ((lb & 0x55555555u) << 1);
        const uint32_t occ1 = ((la >> 1) & 0x55555555u) | (lb & 0xAAAAAAAAu);
        VecT acc = VT::zero();
        int anti = 0;
        uint32_t wnext = maxw > 0 ? codes[base + lane] : 0xFFFFFFFFu;
        for (int k = 0; k < maxw; k++) {
            const uint32_t w4 = wnext;
            if (k + 1 < maxw) wnext = codes[base + (int64_t)(k + 1) * 32 + lane];
            uint32_t na[4], nb[4];
            double v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t code = (w4 >> (8 * u)) & 255u;
                na[u] = la ^ mA[code];
                nb[u] = lb ^ mB[code];
                const double a = amp[code];
                if (KIND == 0) {
                    anti += (int)(hop[code] >> 11);
                    v[u] = a;
                } else {
                    const uint32_t h = hop[code], bf = bF[code], bt = bT[code];
                    const int f = h & 31, t = (h >> 5) & 31, sp = (h >> 10) & 1;
                    int sg = __popc(occ0 & bf) + __popc(occ1 & bf) + __popc(occ0 & bt) + __popc(occ1 & bt);
                    sg += sp * ((int)((occ0 >> f) & 1u) + (int)((occ0 >> t) & 1u)) + (f < t ? 1 : 0);
                    v[u] = (sg & 1) ? -a : a;
                }
            }
            int64_t jb[4];
            int32_t ra[4];
#pragma unroll
            for (int u = 0; u < 4; u++) { jb[u] = __ldg(S.Jb + nb[u]); ra[u] = __ldg(S.rankA + na[u]); }
            VecT xv[4];
#pragma unroll
            for (int u = 0; u < 4; u++) xv[u] = ld_vec(x + (jb[u] + ra[u]));
#pragma unroll
            for (int u = 0; u < 4; u++) mac(acc, v[u], xv[u]);
        }
        if (live) {
            double diag;
            if (KIND == 0) diag = 0.25 * M.J * (double)(wbonds - 2 * anti);
            else { diag = 0.0; const int ndbl = __popc(occ0 & occ1); for (int r = 0; r < ndbl; r++) diag += M.U; }
            const VecT xi = x[row_lo + row];
            mac(acc, diag, xi);
            VecT out = VT::scale(alpha, acc);
            if (gamma.x != 0.0 || gamma.y != 0.0) out = VT::add(out, VT::scale(gamma, xi));
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
        block_reduce_finalize<3, kMFBlock>(d, partials, ticket, dots_out);
    }
}

template <typename VecT, bool DOTS>
static int launch_terms_variant(const qbgpu_matrix *A, const FusedArgs &a)
{
    Context &c = ctx();
    const MatFree *mf = (const MatFree *)A->mf;
    auto kern = mf->kind == 0 ? spmv_terms_kernel_v2<VecT, DOTS, 0> : spmv_terms_kernel_v2<VecT, DOTS, 1>;
    int blocks_per_sm = 0;
    QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, kMFBlock, 0));
    if (blocks_per_sm < 1) blocks_per_sm = 1;
    const int64_t nrows = A->nrows();
    if (nrows == 0) return QBGPU_OK;
    const int64_t nslices = (nrows + 31) / 32;
    int64_t want = (nslices + (kMFBlock / 32) - 1) / (kMFBlock / 32);
    int64_t cap = (int64_t)c.num_sms * blocks_per_sm;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    const int grid = (int)(want < cap ? want : cap);
    kern<<<grid, kMFBlock, 0, c.stream>>>(mf->S, mf->d_M, mf->d_terms, mf->d_states, mf->d_sliceptr, mf->d_codes, nrows, nslices, A->row_lo, mf->wbonds,
                                          (const VecT *)a.x, (const VecT *)a.z, (VecT *)a.y, a.alpha, a.gamma, a.beta, a.scal_mode, a.sc, a.dots,
                                          c.partials, c.ticket);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

template <typename VecT, bool DOTS>
static int launch_matfree_variant(const qbgpu_matrix *A, const FusedArgs &a)
{
    Context &c = ctx();
    const MatFree *mf = (const MatFree *)A->mf;
    auto kern = spmv_matfree_kernel<VecT, DOTS>;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, kMFBlock, 0));
        if (blocks_per_sm < 1) blocks_per_sm = 1;
    }
    const int64_t nrows = A->nrows();
    if (nrows == 0) return QBGPU_OK;
    int64_t want = (nrows + kMFBlock - 1) / kMFBlock;
    int64_t cap = (int64_t)c.num_sms * blocks_per_sm;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    const int grid = (int)(want < cap ? want : cap);
    kern<<<grid, kMFBlock, 0, c.stream>>>(mf->S, mf->d_M, mf->d_N, mf->d_states, nrows, A->row_lo, (const VecT *)a.x, (const VecT *)a.z, (VecT *)a.y,
                                          a.alpha, a.gamma, a.beta, a.scal_mode, a.sc, a.dots, c.partials, c.ticket);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

int launch_spmv_matfree(const qbgpu_matrix *A, const FusedArgs &a)
{
    const bool dots = a.dots != nullptr;
    if (((const MatFree *)A->mf)->d_codes) {
        if (A->api_complex) return dots ? launch_terms_variant<double2, true>(A, a) : launch_terms_variant<double2, false>(A, a);
        return dots ? launch_terms_variant<double, true>(A, a) : launch_terms_variant<double, false>(A, a);
    }
    if (A->api_complex) return dots ? launch_matfree_variant<double2, true>(A, a) : launch_matfree_variant<double2, false>(A, a);
    return dots ? launch_matfree_variant<double, true>(A, a) : launch_matfree_variant<double, false>(A, a);
}

void matfree_destroy(qbgpu_matrix *A)
{
    MatFree *mf = (MatFree *)A->mf;
    if (!mf) return;
    cudaFree(mf->d_codes); cudaFree(mf->d_sliceptr); cudaFree(mf->d_terms); cudaFree(mf->d_N); cudaFree(mf->d_M); cudaFree(mf->d_Jb); cudaFree(mf->d_rank); cudaFree(mf->d_off); cudaFree(mf->d_alist); cudaFree(mf->d_states);
    delete mf;
    A->mf = nullptr;
}

static int create_matfree(qbgpu_matrix_t *out, const HostTables &T, const ModelParams &M, int api_complex, int64_t row_lo, int64_t row_hi, int flags = 0)
{
    QB_TRY(ensure_init());
    Context &c = ctx();
    if (!out) return fail(QBGPU_ERR_ARG, "null handle pointer");
    *out = nullptr;
    if (T.dim <= 0) return fail(QBGPU_ERR_ARG, "matrix-free: empty sector");
    if (T.dim > 2147483647LL) return fail(QBGPU_ERR_ARG, "matrix-free: dimension exceeds the int32 column range");
    if (T.nsites > 32) return fail(QBGPU_ERR_ARG, "matrix-free: at most 32 sites");
    if (row_hi < 0) row_hi = T.dim;
    if (row_lo < 0 || row_lo > row_hi || row_hi > T.dim) return fail(QBGPU_ERR_ARG, "matrix-free: bad row shard");
    const int64_t nloc = row_hi - row_lo;
    auto *A = new qbgpu_matrix;
    A->n = T.dim; A->row_lo = row_lo; A->row_hi = row_hi; A->api_complex = api_complex != 0;
    A->val_real = true; A->format = QBGPU_FORMAT_MATFREE; A->nnz = 0; A->nnz_input = 0;
    auto *mf = new MatFree;
    A->mf = mf;
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { qbgpu_destroy(A); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&mf->d_Jb, sizeof(int64_t) * T.Jb.size()));
    QB_CU(cudaMalloc(&mf->d_rank, sizeof(int32_t) * T.rankA.size()));
    QB_CU(cudaMalloc(&mf->d_alist, sizeof(uint32_t) * T.alist.size()));
    QB_CU(cudaMalloc(&mf->d_off, sizeof(int32_t) * T.class_off.size()));
    QB_CU(cudaMalloc(&mf->d_M, sizeof(ModelParams)));
    QB_CU(cudaMalloc(&mf->d_states, sizeof(uint2) * (nloc ? nloc : 1)));
    QB_CU(cudaMemcpyAsync(mf->d_Jb, T.Jb.data(), sizeof(int64_t) * T.Jb.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(mf->d_rank, T.rankA.data(), sizeof(int32_t) * T.rankA.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(mf->d_alist, T.alist.data(), sizeof(uint32_t) * T.alist.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(mf->d_off, T.class_off.data(), sizeof(int32_t) * T.class_off.size(), cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(mf->d_M, &M, sizeof(ModelParams), cudaMemcpyHostToDevice, c.stream));
    static thread_local SiteTables N;
    memset(&N, 0, sizeof N);
    N.nsites = T.nsites;
    for (int b = 0; b < M.nbonds; b++) {
        const int i = M.bonds[b].i, j = M.bonds[b].j, w = M.bonds[b].w;
        N.nbr[i] |= 1u << j; N.nbr[j] |= 1u << i;
        N.wgt[i][j] = (uint8_t)w; N.wgt[j][i] = (uint8_t)w;
        N.wbonds += w;
    }
    QB_CU(cudaMalloc(&mf->d_N, sizeof(SiteTables)));
    QB_CU(cudaMemcpyAsync(mf->d_N, &N, sizeof(SiteTables), cudaMemcpyHostToDevice, c.stream));
    SectorTables &S = mf->S;
    S.nsites = T.nsites; S.bps = T.bps; S.nA = T.nA; S.nB = T.nB; S.t0 = T.t0; S.t1 = T.t1; S.dim = T.dim;
    S.Jb = mf->d_Jb; S.rankA = mf->d_rank; S.alist = mf->d_alist; S.class_off = mf->d_off; S.sizeB = (uint32_t)(T.Jb.size() - 1);
    int64_t g = (nloc + kBBlock - 1) / kBBlock;
    if (g < 1) g = 1;
    if (g > 148 * 64) g = 148 * 64;
    matfree_states_kernel<<<(int)g, kBBlock, 0, c.stream>>>(S, row_lo, nloc, mf->d_states);
    QB_LAUNCH_COUNT();
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
#undef QB_CU
    mf->bytes = (int64_t)(sizeof(uint2) * nloc + sizeof(int64_t) * T.Jb.size() + 4 * (T.rankA.size() + T.alist.size() + T.class_off.size()) + sizeof(ModelParams));
    mf->wbonds = N.wbonds; mf->kind = M.kind;
    if ((flags & QBGPU_MATFREE_TERMS) && nloc > 0) {
        // code table: one code per directed bond (x spin for electrons)
        static thread_local TermTable TT;
        memset(&TT, 0, sizeof TT);
        int npairs = 0;
        for (int f = 0; f < T.nsites; f++)
            for (int t = 0; t < T.nsites; t++)
                if ((N.nbr[f] >> t) & 1u) {
                    const int per = M.kind == 0 ? 1 : 2;
                    if ((npairs + 1) * per > 255) { qbgpu_destroy(A); return fail(QBGPU_ERR_ARG, "matrix-free terms: more than 255 (directed bond, spin) codes"); }
                    TT.code_of[f][t] = (uint8_t)npairs;
                    for (int sp = 0; sp < per; sp++) {
                        const int code = npairs * per + sp;
                        const int w = N.wgt[f][t];
                        TT.hop[code] = (uint32_t)f | ((uint32_t)t << 5) | ((uint32_t)sp << 10) | ((uint32_t)w << 11);
                        if (M.kind == 0) TT.amp[code] = 0.5 * M.J * w;
                        else { double amp = 0.0; for (int r = 0; r < w; r++) amp += -M.t; TT.amp[code] = amp; }
                    }
                    npairs++;
                }
        TT.ncodes = npairs * (M.kind == 0 ? 1 : 2);
        for (int code = 0; code < TT.ncodes; code++) {
            const uint32_t h = TT.hop[code];
            const int f = h & 31, t = (h >> 5) & 31, sp = (h >> 10) & 1;
            const int bits = M.kind == 0 ? 1 : 2;
            const uint32_t bit_f = 1u << (bits * (f >> 1) + (M.kind == 0 ? 0 : sp)), bit_t = 1u << (bits * (t >> 1) + (M.kind == 0 ? 0 : sp));
            if (f & 1) TT.mask_b[code] ^= bit_f; else TT.mask_a[code] ^= bit_f;
            if (t & 1) TT.mask_b[code] ^= bit_t; else TT.mask_a[code] ^= bit_t;
            TT.below_f[code] = (1u << f) - 1u;
            TT.below_t[code] = (1u << t) - 1u;
        }
        TT.hop[255] = 0; TT.amp[255] = 0.0;                    // padding: no flip, no weight, zero amplitude
        const int64_t nslices = (nloc + 31) / 32;
        int64_t *d_words = nullptr;
        void *d_tmp = nullptr;
        auto tclean = [&]() { cudaFree(d_words); cudaFree(d_tmp); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { tclean(); qbgpu_destroy(A); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
        QB_CU(cudaMalloc(&mf->d_terms, sizeof(TermTable)));
        QB_CU(cudaMemcpyAsync(mf->d_terms, &TT, sizeof(TermTable), cudaMemcpyHostToDevice, c.stream));
        QB_CU(cudaMalloc(&d_words, sizeof(int64_t) * (nslices + 1)));
        QB_CU(cudaMalloc(&mf->d_sliceptr, sizeof(int64_t) * (nslices + 1)));
        int64_t gs = (nslices + 1 + (kBBlock / 32) - 1) / (kBBlock / 32);
        if (gs > 148 * 64) gs = 148 * 64;
        terms_count_kernel<<<(int)gs, kBBlock, 0, c.stream>>>(S, mf->d_M, mf->d_N, mf->d_states, nloc, nslices, d_words);
        QB_LAUNCH_COUNT();
        size_t tb = 0;
        QB_CU(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_words, mf->d_sliceptr, nslices + 1, c.stream));
        QB_CU(cudaMalloc(&d_tmp, tb ? tb : 1));
        QB_CU(cub::DeviceScan::ExclusiveSum(d_tmp, tb, d_words, mf->d_sliceptr, nslices + 1, c.stream));
        int64_t total_words = 0;
        QB_CU(cudaMemcpyAsync(&total_words, mf->d_sliceptr + nslices, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
        QB_CU(cudaStreamSynchronize(c.stream));
        QB_CU(cudaMalloc(&mf->d_codes, sizeof(uint32_t) * (size_t)(total_words ? total_words : 1)));
        terms_fill_kernel<<<(int)gs, kBBlock, 0, c.stream>>>(mf->d_M, mf->d_N, mf->d_terms, mf->d_states, nloc, nslices, mf->d_sliceptr, mf->d_codes);
        QB_LAUNCH_COUNT();
        QB_CU(cudaStreamSynchronize(c.stream));
        QB_CU(cudaGetLastError());
#undef QB_CU
        tclean();
        mf->bytes += (int64_t)(4 * total_words + 8 * (nslices + 1) + sizeof(TermTable));
        A->nnz_input = 4 * total_words;                     // bytes of codes (padding included), for the bench's byte count
    }
    *out = A;
    return QBGPU_OK;
}

int64_t matfree_bytes(const qbgpu_matrix *A) { return A->mf ? ((const MatFree *)A->mf)->bytes : 0; }

}  // namespace qb

using namespace qb;

extern "C" {

int qbgpu_full_apply_diag(int kind, int nsites, int n0, int n1, const double *coef0_reim, const double *coef1_reim,
                          const void *x_dev, void *y_dev)
{ return full_apply_diag(kind, nsites, n0, n1, coef0_reim, coef1_reim, x_dev, y_dev, false); }

int qbgpu_debug_full_apply_diag_host(int kind, int nsites, int n0, int n1, const double *coef0_reim, const double *coef1_reim,
                                     const void *x_host, void *y_host)
{ return full_apply_diag(kind, nsites, n0, n1, coef0_reim, coef1_reim, x_host, y_host, true); }

/* Rows of a full-basis operator recomputed on the HOST in extended precision, no device involved: for each listed row r (the
 * reference's Lin order) the basis state is unranked from the Lin tables, the row is regenerated by row_entries() -- the
 * function the device generators run, pinned entry for entry to matrices assembled by the compiled reference
 * (tests/test_gpu_parity.py) -- and y_r = sum_c H_rc x_c is accumulated in long double.  kind 0: Heisenberg (n0 = down spins),
 * 1: Hubbard (n0, n1 = N_up, N_dn).  x_host: the full vector (complex: re,im pairs); y_out: 2 doubles per listed row. */
int qbgpu_debug_rows_host(int kind, int nsites, int n0, int n1, int nbonds, const int32_t *bonds, double J, double t, double U,
                          int64_t nrows, const int64_t *rows, const void *x_host, int x_complex, double *y_out)
{
    if (nsites < 2 || nbonds < 1 || !bonds || !rows || !x_host || !y_out || nrows < 0 || (kind != 0 && kind != 1)) return fail(QBGPU_ERR_ARG, "debug_rows_host: bad argument");
    HostTables T;
    QB_TRY(make_tables(nsites, kind == 0 ? 1 : 2, n0, kind == 0 ? 0 : n1, T));
    static thread_local ModelParams M;
    M.kind = kind; M.J = J; M.t = t; M.U = U;
    QB_TRY(merge_bonds(nsites, nbonds, bonds, M));
    SectorTables S;
    S.nsites = T.nsites; S.bps = T.bps; S.nA = T.nA; S.nB = T.nB; S.t0 = T.t0; S.t1 = T.t1; S.dim = T.dim;
    S.Jb = T.Jb.data(); S.rankA = T.rankA.data(); S.alist = T.alist.data(); S.class_off = T.class_off.data(); S.sizeB = (uint32_t)(T.Jb.size() - 1);
    const double *xr = (const double *)x_host;
    for (int64_t k = 0; k < nrows; k++) {
        const int64_t r = rows[k];
        if (r < 0 || r >= T.dim) return fail(QBGPU_ERR_ARG, "debug_rows_host: row out of range");
        uint32_t la, lb;
        unrank_row(S, r, la, lb);
        long double are = 0.0L, aim = 0.0L;
        const double diag = row_entries(S, M, la, lb, [&](int64_t c, double v) {
            if (x_complex) { are += (long double)v * xr[2 * c]; aim += (long double)v * xr[2 * c + 1]; }
            else are += (long double)v * xr[c];
        });
        if (x_complex) { are += (long double)diag * xr[2 * r]; aim += (long double)diag * xr[2 * r + 1]; }
        else are += (long double)diag * xr[r];
        y_out[2 * k] = (double)are; y_out[2 * k + 1] = (double)aim;
    }
    return QBGPU_OK;
}

int64_t qbgpu_dim_heisenberg(int nsites, int ndown)
{
    HostTables T;
    if (nsites < 2 || ndown < 0 || ndown > nsites || make_tables(nsites, 1, ndown, 0, T)) return -1;
    return T.dim;
}

int64_t qbgpu_dim_hubbard(int nsites, int nup, int ndn)
{
    HostTables T;
    if (nsites < 2 || nup < 0 || ndn < 0 || nup > nsites || ndn > nsites || make_tables(nsites, 2, nup, ndn, T)) return -1;
    return T.dim;
}

int qbgpu_create_matfree_heisenberg(qbgpu_matrix_t *A, int nsites, int ndown, int nbonds, const int32_t *bonds, double J,
                                    int api_complex, int flags, int64_t row_lo, int64_t row_hi)
{
    if (nsites < 2 || ndown < 0 || ndown > nsites || nbonds < 1 || !bonds) return fail(QBGPU_ERR_ARG, "create_matfree_heisenberg: bad argument");
    if (flags & QBGPU_SPECIES_ORDER) return fail(QBGPU_ERR_ARG, "create_matfree_heisenberg: QBGPU_SPECIES_ORDER is defined for the Hubbard model only");
    HostTables T;
    QB_TRY(make_tables(nsites, 1, ndown, 0, T));
    static thread_local ModelParams M;
    M.kind = 0; M.J = J; M.t = 0; M.U = 0;
    QB_TRY(merge_bonds(nsites, nbonds, bonds, M));
    return create_matfree(A, T, M, api_complex, row_lo, row_hi, flags);
}

int qbgpu_create_matfree_hubbard(qbgpu_matrix_t *A, int nsites, int nup, int ndn, int nbonds, const int32_t *bonds, double t, double U,
                                 int api_complex, int flags, int64_t row_lo, int64_t row_hi)
{
    if (nsites < 2 || nup < 0 || ndn < 0 || nup > nsites || ndn > nsites || nbonds < 1 || !bonds) return fail(QBGPU_ERR_ARG, "create_matfree_hubbard: bad argument");
    HostTables T;
    QB_TRY(make_tables(nsites, 2, nup, ndn, T));
    static thread_local ModelParams M;
    M.kind = 1; M.J = 0; M.t = t; M.U = U;
    QB_TRY(merge_bonds(nsites, nbonds, bonds, M));
    if (flags & QBGPU_SPECIES_ORDER) return species_build_matfree(A, T, M, api_complex, flags, row_lo, row_hi);   // shards: whole up configurations
    return create_matfree(A, T, M, api_complex, row_lo, row_hi, flags);
}

int qbgpu_build_heisenberg(qbgpu_matrix_t *A, int nsites, int ndown, int nbonds, const int32_t *bonds, double J,
                           int api_complex, int flags, int64_t row_lo, int64_t row_hi)
{
    if (nsites < 2 || ndown < 0 || ndown > nsites || nbonds < 1 || !bonds) return fail(QBGPU_ERR_ARG, "build_heisenberg: bad argument");
    if (flags & QBGPU_SPECIES_ORDER) return fail(QBGPU_ERR_ARG, "build_heisenberg: QBGPU_SPECIES_ORDER is defined for the Hubbard model only");
    HostTables T;
    QB_TRY(make_tables(nsites, 1, ndown, 0, T));
    static thread_local ModelParams M;
    M.kind = 0; M.J = J; M.t = 0; M.U = 0;
    QB_TRY(merge_bonds(nsites, nbonds, bonds, M));
    return build_generic(A, T, M, api_complex, flags, row_lo, row_hi);
}

int qbgpu_build_hubbard(qbgpu_matrix_t *A, int nsites, int nup, int ndn, int nbonds, const int32_t *bonds, double t, double U,
                        int api_complex, int flags, int64_t row_lo, int64_t row_hi)
{
    if (nsites < 2 || nup < 0 || ndn < 0 || nup > nsites || ndn > nsites || nbonds < 1 || !bonds) return fail(QBGPU_ERR_ARG, "build_hubbard: bad argument");
    HostTables T;
    QB_TRY(make_tables(nsites, 2, nup, ndn, T));
    static thread_local ModelParams M;
    M.kind = 1; M.J = 0; M.t = t; M.U = U;
    QB_TRY(merge_bonds(nsites, nbonds, bonds, M));
    if (flags & QBGPU_SPECIES_ORDER) return species_build_stored(A, T, M, api_complex, flags, row_lo, row_hi);   // shards: whole up configurations
    return build_generic(A, T, M, api_complex, flags, row_lo, row_hi);
}

}  // extern "C"
