// quantum_basis_b200/csrc/species.cu -- "species order" for the single-orbital Fermi-Hubbard model (QBGPU_SPECIES_ORDER).
//
// Why: in the reference's Lin-table order (src/basis.cc:1144-1190) every hopping term of the 4x4 Hubbard matrix sends a
// row far away in the index space -- 47 % of the off-diagonal entries lie more than 300 K rows from the diagonal -- so
// the gathers of x cost about 50 GB of DRAM traffic per product where 2.65 GB would be compulsory (DESIGN.md section 7).
// No re-ordering of ONE pass over the rows removes that (profiles/r01_cache_sim_orders_and_tiles.txt).  Two passes do,
// once the basis is indexed by the two spin species separately:
//
//     p = iu * D_dn + id ,   iu = rank of the up-occupancy word, id = rank of the down-occupancy word
//                             (words ordered by (odd-site bits, even-site bits): see build_host_tables)
//
//     H = [ U * (double occupancies) + hops of the DOWN electrons ]   "local" part: same iu, i.e. inside one contiguous
//                                                                     block x[iu, :] of D_dn entries (206 KB for 4x4)
//       + [ hops of the UP electrons ]                                "cross" part: same id, another iu
//
//   pass 1 (local part, rows ascending): every gather falls into the row's own block of x -> x is read once;
//   pass 2 (cross part, y += ...): rows traversed by TILES of down indices (all iu for id in [tau W, tau W + W)), so the
//          gathered columns x[iu', tile] of a whole tile (D_up * W entries: 26 MB for W = 128) stay in L2 -> x is read
//          once more, y is read and written once more.
//
// Vector traffic 5 n S_vec instead of ~19 n S_vec; the matrix stream is unchanged.  Every matrix element factorises as
// (amplitude and sign from the hopping species' own configuration) x (parity of the OTHER species on a site interval):
// sign rule of the reference's oprXphi, src/basis.cc:2717-2731 (fermions ordered site-major, up before down on a site);
// the factorisation is restated in tests/species_builders.py and checked there, entry for entry, against the
// reference-pinned full-basis assembler.  Two kinds of handle share the tables:
//   * stored (qbgpu_build_hubbard + QBGPU_SPECIES_ORDER): the two parts as sliced-jagged matrices, multiplied by the
//     production kernel of sjds.cu (the cross part with its tile-ordered slice traversal);
//   * matrix-free (qbgpu_create_matfree_hubbard + QBGPU_SPECIES_ORDER): nothing stored but the per-species hop tables
//     (a few MB); the counterpart of model<T>::MultMv2 with matrix_free == true, src/model.cc:942-1109.
// The reference-shaped entry points keep the reference's order at the boundary: vectors are permuted on the way in and
// out (perm[r] = internal index of the reference's row r), fused with the real/complex conversion the Krylov drivers do
// anyway.
#include "internal.hpp"
#include "lin_tables.hpp"
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace qb {

// the row functions are compiled for the host too, where g++ does not know the pragma
#ifdef __CUDA_ARCH__
#define QB_UNROLL _Pragma("unroll")
#else
#define QB_UNROLL
#endif

constexpr int kPBlock = 256;
constexpr uint32_t kHopMask = 0xFFFFFFu;      // hop entry .y = interval mask (24 bits) | own sign << 24 | bond multiplicity << 25
constexpr int kMaxWeight = 127;
constexpr int kMaxDbl = 32;

static int grid_rows(int64_t n) { int64_t g = (n + kPBlock - 1) / kPBlock; if (g < 1) g = 1; if (g > 148 * 32) g = 148 * 32; return (int)g; }

__global__ void __launch_bounds__(kPBlock) invert_perm_kernel(int64_t n, const int32_t *__restrict__ perm, int32_t *perm_inv)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x)
        perm_inv[perm[r]] = (int32_t)r;
}

__global__ void tile_descriptor_kernel(int64_t nblk, const int64_t *__restrict__ blk_start, int32_t Dd, const int32_t *__restrict__ perm, int4 *desc);

static double wall_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// Device-resident tables of a species-order handle (owned through qbgpu_matrix::sp).
struct Species {
    int nsites = 0;
    int64_t Du = 0, Dd = 0;
    int64_t tot_u = 0, tot_d = 0;                 // hop-table entries of the two species
    uint32_t *ulist = nullptr, *dlist = nullptr;  // occupancy words in the species order
    int32_t *uptr = nullptr, *dptr = nullptr;     // [D + 1] offsets into the hop tables
    uint2 *uhop = nullptr, *dhop = nullptr;       // (.x = target configuration index, .y = mask | sign | weight), sorted by target
    double *ampw = nullptr;                       // [128] amplitude of a bond of multiplicity w: -t added w times (LIL accumulation)
    double *diagk = nullptr;                      // [33]  U added k times
    double amp_uni = 0.0;                         // != 0: every bond has the same multiplicity and this is its amplitude
    int tile = 64;                                // W: down indices per tile of the cross pass (multiple of 32)
    int64_t *blk_start = nullptr;                 // [nblk + 1] first row (reference order) of every non-empty odd-site label
    int4 *blk_desc = nullptr;                     // [nblk] the rectangle of the internal order a block maps to: (iu0, id0, Cd, rows)
    int64_t nblk = 0, blk_max_rows = 0;
    bool matfree = false;
    int64_t bytes = 0;
};

// Plain-pointer view of the tables (device pointers inside kernels, host pointers in the CPU-side debug entry): the
// per-row functions below are __host__ __device__, so the index logic the kernels run is the logic the CPU tests check.
struct SpeciesView {
    int64_t Du, Dd, tot_u, tot_d;
    const uint32_t *ulist, *dlist;
    const int32_t *uptr, *dptr;
    const uint2 *uhop, *dhop;
};

// value of a hop entry given the OTHER species' occupancy word
__host__ __device__ __forceinline__ double hop_value(uint32_t meta, uint32_t other, const double *ampw)
{
    const double a = ampw[meta >> 25];
    const uint32_t sg = ((meta >> 24) ^ (uint32_t)popc_hd(other & (meta & kHopMask))) & 1u;
    // flip the sign bit with integer logic (a select on the two halves plus a negation on the fp64 pipe otherwise)
#ifdef __CUDA_ARCH__
    return __hiloint2double(__double2hiint(a) ^ (int)(sg << 31), __double2loint(a));
#else
    return sg ? -a : a;
#endif
}

// the same when every bond has the same multiplicity (the usual case): the amplitude is a kernel argument, no table lookup
__host__ __device__ __forceinline__ double hop_value_uni(uint32_t meta, uint32_t other, double amp)
{
    const uint32_t sg = ((meta >> 24) ^ (uint32_t)popc_hd(other & (meta & kHopMask))) & 1u;
#ifdef __CUDA_ARCH__
    return __hiloint2double(__double2hiint(amp) ^ (int)(sg << 31), __double2loint(amp));
#else
    return sg ? -amp : amp;
#endif
}

struct SpeciesHost {
    std::vector<uint32_t> list[2];
    std::vector<int32_t> ptr[2];
    std::vector<uint2> hop[2];
    std::vector<int32_t> rank;                    // rank of a word among the words with the same popcount
    double ampw[kMaxWeight + 1];
    double diagk[kMaxDbl + 1];
    int uniform_w = 0;                            // the common bond multiplicity, 0 when the bonds differ
};

// The hop tables, with the formulas of tests/species_builders.py: for the hop f -> t of a species on the word `w`
//   own sign = parity( popc(w & below_f) + popc(w & below_t) + [f < t] )
//   the other species flips the sign by the parity of its electrons on   [min, max)  (up hop)   or   (min, max]  (down hop).
static int build_host_tables(int nsites, int nup, int ndn, const ModelParams &M, SpeciesHost &H)
{
    if (nsites < 2 || nsites > 24) return fail(QBGPU_ERR_ARG, "species order: between 2 and 24 sites");
    const uint32_t nw = 1u << nsites;
    H.rank.assign(nw, 0);
    // Order of the configurations of one species: by (bits of the odd sites, bits of the even sites), odd sites major.  Any
    // order serves the two passes; THIS one makes the species order a block-wise refinement of the reference's Lin order
    // (label of the odd sites major, src/basis.cc:1144-1190): the rows of one odd-site label -- contiguous in the reference's
    // order -- occupy a rectangle [iu0, iu0 + Cu) x [id0, id0 + Cd) of the internal order, so the permutation at the
    // boundary (vec_to_native / vec_from_native) moves whole blocks and both of its sides stay sector-efficient.
    auto order_key = [nsites](uint32_t w) {
        uint32_t odd = 0, even = 0;
        for (int s = 0; s < nsites; s++) { const uint32_t bit = (w >> s) & 1u; if (s & 1) odd |= bit << (s >> 1); else even |= bit << (s >> 1); }
        return ((uint64_t)odd << 32) | even;
    };
    const int nel[2] = {nup, ndn};
    for (int b = 0; b < M.nbonds; b++)
        if (M.bonds[b].w > kMaxWeight) return fail(QBGPU_ERR_ARG, "species order: a bond is repeated more than 127 times");
    {   // rank of every word among the words of its popcount class, in that order
        std::vector<std::vector<uint32_t>> cls(nsites + 1);
        for (uint32_t w = 0; w < nw; w++) cls[__builtin_popcount(w)].push_back(w);
        for (auto &c : cls) {
            std::sort(c.begin(), c.end(), [&](uint32_t a, uint32_t b) { return order_key(a) < order_key(b); });
            for (size_t k = 0; k < c.size(); k++) H.rank[c[k]] = (int32_t)k;
        }
    }
    for (int sp = 0; sp < 2; sp++) {
        H.list[sp].assign((size_t)0, 0u);
        for (uint32_t w = 0; w < nw; w++) if (__builtin_popcount(w) == nel[sp]) H.list[sp].push_back(w);
        std::sort(H.list[sp].begin(), H.list[sp].end(), [&](uint32_t a, uint32_t b) { return order_key(a) < order_key(b); });
        const size_t D = H.list[sp].size();
        H.ptr[sp].assign(D + 1, 0);
        H.hop[sp].clear();
        std::vector<uint2> row;
        for (size_t c = 0; c < D; c++) {
            const uint32_t word = H.list[sp][c];
            row.clear();
            for (int b = 0; b < M.nbonds; b++) {
                for (int dir = 0; dir < 2; dir++) {
                    const int f = dir ? M.bonds[b].j : M.bonds[b].i, t = dir ? M.bonds[b].i : M.bonds[b].j;
                    if (!((word >> f) & 1u) || ((word >> t) & 1u)) continue;
                    const uint32_t below_f = (1u << f) - 1u, below_t = (1u << t) - 1u;
                    const uint32_t own = (uint32_t)(__builtin_popcount(word & below_f) + __builtin_popcount(word & below_t) + (f < t ? 1 : 0)) & 1u;
                    const uint32_t mask = sp == 0 ? (below_f ^ below_t) : (((2u << f) - 1u) ^ ((2u << t) - 1u));
                    const uint32_t nword = word ^ (1u << f) ^ (1u << t);
                    uint2 e;
                    e.x = (uint32_t)H.rank[nword];
                    e.y = (mask & kHopMask) | (own << 24) | ((uint32_t)M.bonds[b].w << 25);
                    row.push_back(e);
                }
            }
            std::sort(row.begin(), row.end(), [](const uint2 &a, const uint2 &b) { return a.x < b.x; });
            if (H.hop[sp].size() + row.size() > 2147483647ull) return fail(QBGPU_ERR_ARG, "species order: hop table exceeds the int32 range");
            H.hop[sp].insert(H.hop[sp].end(), row.begin(), row.end());
            H.ptr[sp][c + 1] = (int32_t)H.hop[sp].size();
        }
    }
    H.uniform_w = M.nbonds > 0 ? M.bonds[0].w : 0;
    for (int b = 1; b < M.nbonds; b++) if (M.bonds[b].w != H.uniform_w) H.uniform_w = 0;
    for (int w = 0; w <= kMaxWeight; w++) { double a = 0.0; for (int r = 0; r < w; r++) a += -M.t; H.ampw[w] = a; }
    for (int k = 0; k <= kMaxDbl; k++) { double d = 0.0; for (int r = 0; r < k; r++) d += M.U; H.diagk[k] = d; }
    return QBGPU_OK;
}

static void species_free(Species *S)
{
    if (!S) return;
    cudaFree(S->ulist); cudaFree(S->dlist); cudaFree(S->uptr); cudaFree(S->dptr); cudaFree(S->uhop); cudaFree(S->dhop);
    cudaFree(S->ampw); cudaFree(S->diagk); cudaFree(S->blk_start); cudaFree(S->blk_desc);
    delete S;
}

static SpeciesView view_of(const Species *S)
{
    SpeciesView V;
    V.Du = S->Du; V.Dd = S->Dd; V.tot_u = S->tot_u; V.tot_d = S->tot_d;
    V.ulist = S->ulist; V.dlist = S->dlist; V.uptr = S->uptr; V.dptr = S->dptr; V.uhop = S->uhop; V.dhop = S->dhop;
    return V;
}

template <typename T>
static cudaError_t upload(T **dst, const T *src, size_t count, cudaStream_t st)
{
    cudaError_t e = cudaMalloc(dst, sizeof(T) * (count ? count : 1));
    if (e != cudaSuccess) return e;
    if (count) e = cudaMemcpyAsync(*dst, src, sizeof(T) * count, cudaMemcpyHostToDevice, st);
    return e;
}

// Common part of both handle kinds: tables in HBM, the permutation, and a bare handle that owns them.
static int species_common(qbgpu_matrix **out, const HostTables &T, const ModelParams &M, int api_complex, SpeciesHost &H, bool with_perm = true)
{
    QB_TRY(ensure_init());
    Context &c = ctx();
    *out = nullptr;
    if (T.bps != 2 || M.kind != 1) return fail(QBGPU_ERR_ARG, "species order: only the single-orbital Hubbard model has two species");
    QB_TRY(build_host_tables(T.nsites, T.t0, T.t1, M, H));
    const int64_t Du = (int64_t)H.list[0].size(), Dd = (int64_t)H.list[1].size();
    if (Du <= 0 || Dd <= 0) return fail(QBGPU_ERR_ARG, "species order: empty sector");
    if (Du > 2147483647LL / Dd) return fail(QBGPU_ERR_ARG, "species order: dimension exceeds the int32 column range");
    if (Du * Dd != T.dim) return fail(QBGPU_ERR_STATE, "species order: dimension mismatch with the Lin tables");
    auto *A = new qbgpu_matrix;
    auto *S = new Species;
    A->sp = S;
    A->n = T.dim; A->row_lo = 0; A->row_hi = T.dim; A->api_complex = api_complex != 0; A->val_real = true;
    S->nsites = T.nsites; S->Du = Du; S->Dd = Dd; S->tot_u = (int64_t)H.hop[0].size(); S->tot_d = (int64_t)H.hop[1].size();
    int W = 64;                                            // measured on BASELINE config 3: 64 -> 14.6 ms, 128 -> 14.75, 256 -> 15.8 (fp64 vectors)
    if (const char *e = getenv("QBGPU_SPECIES_TILE")) W = atoi(e);
    if (W < 32) W = 32;
    W = (W + 31) / 32 * 32;
    S->tile = W;
    int32_t *d_rank = nullptr;
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cudaFree(d_rank); qbgpu_destroy(A); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(upload(&S->ulist, H.list[0].data(), H.list[0].size(), c.stream));
    QB_CU(upload(&S->dlist, H.list[1].data(), H.list[1].size(), c.stream));
    QB_CU(upload(&S->uptr, H.ptr[0].data(), H.ptr[0].size(), c.stream));
    QB_CU(upload(&S->dptr, H.ptr[1].data(), H.ptr[1].size(), c.stream));
    QB_CU(upload(&S->uhop, H.hop[0].data(), H.hop[0].size(), c.stream));
    QB_CU(upload(&S->dhop, H.hop[1].data(), H.hop[1].size(), c.stream));
    QB_CU(upload(&S->ampw, H.ampw, (size_t)kMaxWeight + 1, c.stream));
    QB_CU(upload(&S->diagk, H.diagk, (size_t)kMaxDbl + 1, c.stream));
    if (with_perm) {
        QB_CU(upload(&d_rank, H.rank.data(), H.rank.size(), c.stream));
        QB_CU(cudaMalloc(&A->perm, sizeof(int32_t) * (size_t)T.dim));
        int rc = species_perm_build(T, d_rank, Dd, A->perm);
        if (rc) { cudaFree(d_rank); qbgpu_destroy(A); return rc; }
        QB_CU(cudaMalloc(&A->perm_inv, sizeof(int32_t) * (size_t)T.dim));
        invert_perm_kernel<<<grid_rows(T.dim), kPBlock, 0, c.stream>>>(T.dim, A->perm, A->perm_inv);
        QB_LAUNCH_COUNT();
        // the non-empty blocks of the reference's order (rows of one odd-site label): the tiles of the way in
        std::vector<int64_t> blk;
        int64_t max_rows = 0;
        for (size_t b = 0; b + 1 < T.Jb.size(); b++)
            if (T.Jb[b + 1] > T.Jb[b]) { blk.push_back(T.Jb[b]); max_rows = std::max(max_rows, T.Jb[b + 1] - T.Jb[b]); }
        blk.push_back(T.dim);
        S->nblk = (int64_t)blk.size() - 1;
        S->blk_max_rows = max_rows;
        QB_CU(upload(&S->blk_start, blk.data(), blk.size(), c.stream));
        QB_CU(cudaMalloc(&S->blk_desc, sizeof(int4) * (size_t)(S->nblk ? S->nblk : 1)));
        tile_descriptor_kernel<<<(int)std::min<int64_t>(S->nblk > 0 ? S->nblk : 1, 148 * 8), kPBlock, 0, c.stream>>>(S->nblk, S->blk_start, (int32_t)Dd, A->perm, S->blk_desc);
        QB_LAUNCH_COUNT();
    }
    QB_CU(cudaStreamSynchronize(c.stream));
    cudaFree(d_rank); d_rank = nullptr;
#undef QB_CU
    S->amp_uni = H.uniform_w > 0 ? H.ampw[H.uniform_w] : 0.0;
    S->bytes = (int64_t)(4 * (Du + Dd) + 4 * (Du + Dd + 2) + 8 * (S->tot_u + S->tot_d) + 8 * (kMaxWeight + 1 + kMaxDbl + 1) + (with_perm ? 8 * T.dim : 0));
    *out = A;
    return QBGPU_OK;
}

// ------------------------------------------------------------------------------------------- stored parts (generator)
// Row offsets are closed-form:  local part  len(iu,id) = 1 + #down hops(id)   ->  iu * (tot_d + Dd) + dptr[id] + id
//                               cross part  len(iu,id) = #up hops(iu)         ->  Dd * uptr[iu] + id * len
__host__ __device__ __forceinline__ void species_rowptr_at(const SpeciesView &V, int64_t n, int64_t p, int64_t &rl, int64_t &rc)
{
    const int64_t iu = p / V.Dd, id = p - iu * V.Dd;        // p == n: iu = Du, id = 0 -> the totals
    rl = iu * (V.tot_d + V.Dd) + (int64_t)V.dptr[id] + id;
    const int64_t u0 = V.uptr[iu];
    const int64_t len = p < n ? (int64_t)V.uptr[iu + 1] - u0 : 0;
    rc = V.Dd * u0 + id * len;
}

// rows [p0, p1] of the full operator (a row shard: whole up configurations); offsets relative to the shard's first entry
__global__ void __launch_bounds__(kPBlock) species_rowptr_kernel(SpeciesView V, int64_t n, int64_t p0, int64_t p1, int64_t base_l, int64_t base_c,
                                                                 int64_t *rp_local, int64_t *rp_cross)
{
    for (int64_t p = p0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p <= p1; p += (int64_t)gridDim.x * blockDim.x) {
        int64_t rl, rc;
        species_rowptr_at(V, n, p, rl, rc);
        rp_local[p - p0] = rl - base_l; rp_cross[p - p0] = rc - base_c;
    }
}

template <typename ValT> __host__ __device__ __forceinline__ void put_entry(int32_t *col, ValT *val, int64_t at, int32_t c, double v)
{
    col[at] = c;
    if constexpr (sizeof(ValT) == 16) val[at] = make_double2(v, 0.0); else val[at] = v;
}

// both parts of row p, columns ascending
template <typename ValT>
__host__ __device__ __forceinline__ void species_fill_row(const SpeciesView &V, const double *ampw, const double *diagk, int64_t p,
                                                          int32_t *col_l, ValT *val_l, int32_t *col_c, ValT *val_c,
                                                          int64_t base_l = 0, int64_t base_c = 0)
{
    const int64_t iu = p / V.Dd, id = p - iu * V.Dd;
    const uint32_t U = V.ulist[iu], D = V.dlist[id];
    // local part: down hops sorted by target, the diagonal (always stored, src/sparse.cc:44-54) at its sorted position
    int64_t at = iu * (V.tot_d + V.Dd) + (int64_t)V.dptr[id] + id - base_l;
    bool diag_done = false;
    for (int e = V.dptr[id]; e < V.dptr[id + 1]; e++) {
        const uint2 h = V.dhop[e];
        if (!diag_done && (int64_t)h.x > id) { put_entry(col_l, val_l, at++, (int32_t)p, diagk[popc_hd(U & D)]); diag_done = true; }
        put_entry(col_l, val_l, at++, (int32_t)(iu * V.Dd + (int64_t)h.x), hop_value(h.y, U, ampw));
    }
    if (!diag_done) put_entry(col_l, val_l, at++, (int32_t)p, diagk[popc_hd(U & D)]);
    // cross part: up hops, sorted by target
    const int64_t u0 = V.uptr[iu], len = (int64_t)V.uptr[iu + 1] - u0;
    at = V.Dd * u0 + id * len - base_c;
    for (int64_t e = u0; e < u0 + len; e++) {
        const uint2 h = V.uhop[e];
        put_entry(col_c, val_c, at++, (int32_t)((int64_t)h.x * V.Dd + id), hop_value(h.y, D, ampw));
    }
}

template <typename ValT>
__global__ void __launch_bounds__(kPBlock) species_fill_kernel(SpeciesView V, int64_t p0, int64_t p1, int64_t base_l, int64_t base_c,
                                                               const double *__restrict__ ampw_g, const double *__restrict__ diagk_g,
                                                               int32_t *col_l, ValT *val_l, int32_t *col_c, ValT *val_c)
{
    __shared__ double ampw[kMaxWeight + 1], diagk[kMaxDbl + 1];
    for (int k = threadIdx.x; k <= kMaxWeight; k += blockDim.x) ampw[k] = ampw_g[k];
    for (int k = threadIdx.x; k <= kMaxDbl; k += blockDim.x) diagk[k] = diagk_g[k];
    __syncthreads();
    for (int64_t p = p0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < p1; p += (int64_t)gridDim.x * blockDim.x)
        species_fill_row<ValT>(V, ampw, diagk, p, col_l, val_l, col_c, val_c, base_l, base_c);
}


// the packed layout of a stored part: col[i] = col[i] | code[i] << cbits (qbgpu_matrix::cbits)
__global__ void __launch_bounds__(kPBlock) pack_codes_kernel(int64_t nnz, uint32_t *col, const uint8_t *__restrict__ code, int cbits)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x)
        col[i] = packed_word((int32_t)col[i], code[i], cbits);
}

static void make_slice_order(int64_t n, int64_t Dd, int W, std::vector<int32_t> &order)
{
    const int64_t ns = (n + 31) / 32;
    const int64_t ntile = (Dd + W - 1) / W;
    std::vector<int64_t> start(ntile + 1, 0);
    for (int64_t s = 0; s < ns; s++) start[((s * 32) % Dd) / W + 1]++;
    for (int64_t t = 0; t < ntile; t++) start[t + 1] += start[t];
    order.assign(ns, 0);
    for (int64_t s = 0; s < ns; s++) order[start[((s * 32) % Dd) / W]++] = (int32_t)s;
}

// row_lo/row_hi: a row shard (multi-GPU) -- whole up configurations only, rows [u_lo * D_dn, u_hi * D_dn); it has no
// permutation: its vectors (x full length, y and z the local rows) are in the internal order, as every sharded handle's are
// in "row order".  The local part of a shard references only columns of the shard's own rows.
int species_build_stored(qbgpu_matrix_t *out, const HostTables &T, const ModelParams &M, int api_complex, int flags, int64_t row_lo, int64_t row_hi)
{
    if (!out) return fail(QBGPU_ERR_ARG, "null handle pointer");
    *out = nullptr;
    const double t0 = wall_s();
    SpeciesHost H;
    qbgpu_matrix *A = nullptr;
    const bool rows_given = row_hi >= 0;                    // built as a row shard of a multi-GPU run (also one covering all rows)
    if (row_hi < 0) row_hi = T.dim;
    const bool shard = !(row_lo == 0 && row_hi == T.dim);
    QB_TRY(species_common(&A, T, M, api_complex, H, !shard));
    Context &c = ctx();
    Species *S = (Species *)A->sp;
    const int64_t n = A->n, Dd = S->Dd;
    if (shard) {
        if (row_lo < 0 || row_lo > row_hi || row_hi > n || row_lo % Dd != 0 || row_hi % Dd != 0)
        { qbgpu_destroy(A); return fail(QBGPU_ERR_ARG, "species order: a row shard must consist of whole up configurations (multiples of D_dn rows)"); }
        A->row_lo = row_lo; A->row_hi = row_hi;
    }
    const int64_t nloc = row_hi - row_lo, u_lo = row_lo / Dd, u_hi = row_hi / Dd;
    auto *C = new qbgpu_matrix;                             // the cross part
    A->second = C;
    C->n = n; C->row_lo = row_lo; C->row_hi = row_hi; C->api_complex = A->api_complex;
    A->val_real = C->val_real = !(flags & QBGPU_KEEP_COMPLEX) || !api_complex;
    const int64_t base_l = u_lo * (S->tot_d + Dd), base_c = Dd * (int64_t)H.ptr[0][u_lo];
    A->nnz = (u_hi - u_lo) * (S->tot_d + Dd);
    C->nnz = Dd * ((int64_t)H.ptr[0][u_hi] - (int64_t)H.ptr[0][u_lo]);
    A->nnz_input = (A->nnz + C->nnz + nloc) / 2;            // what the reference would store: upper triangle incl. the diagonal
    C->nnz_input = C->nnz;
    A->block_D = Dd;                                        // pass 1 may keep the block of x in shared memory (sjds_bulk.cu)
    {   // every block of the local part has the same rows (lengths depend on the down configuration only): periodic metadata
        int64_t g = 32, r = Dd % 32;
        while (r) { const int64_t t = g % r; g = r; r = t; }               // gcd(32, Dd)
        const int64_t pb = 32 / g;                                          // blocks per period
        if ((u_hi - u_lo) >= 2 * pb) { A->period_slices = pb * Dd / 32; A->period_entries = pb * (S->tot_d + Dd); }
    }
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { qbgpu_destroy(A); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&A->rowptr, sizeof(int64_t) * (nloc + 1)));
    QB_CU(cudaMalloc(&C->rowptr, sizeof(int64_t) * (nloc + 1)));
    QB_CU(cudaMalloc(&A->col, sizeof(int32_t) * (size_t)(A->nnz ? A->nnz : 1) + 64));
    QB_CU(cudaMalloc(&A->val, A->val_bytes() * (size_t)(A->nnz ? A->nnz : 1) + 64));
    QB_CU(cudaMalloc(&C->col, sizeof(int32_t) * (size_t)(C->nnz ? C->nnz : 1) + 64));
    QB_CU(cudaMalloc(&C->val, C->val_bytes() * (size_t)(C->nnz ? C->nnz : 1) + 64));
    const SpeciesView V = view_of(S);
    species_rowptr_kernel<<<grid_rows(nloc + 1), kPBlock, 0, c.stream>>>(V, n, row_lo, row_hi, base_l, base_c, A->rowptr, C->rowptr);
    QB_LAUNCH_COUNT();
    if (nloc > 0) {
        if (A->val_real)
            species_fill_kernel<double><<<grid_rows(nloc), kPBlock, 0, c.stream>>>(V, row_lo, row_hi, base_l, base_c, S->ampw, S->diagk, A->col, (double *)A->val, C->col, (double *)C->val);
        else
            species_fill_kernel<double2><<<grid_rows(nloc), kPBlock, 0, c.stream>>>(V, row_lo, row_hi, base_l, base_c, S->ampw, S->diagk, A->col, (double2 *)A->val, C->col, (double2 *)C->val);
        QB_LAUNCH_COUNT();
    }
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
    // layout: always the sliced-jagged kernels (the traversal order of the cross part exists only there).  A part of a handle
    // built without a row range, with real values, stores packed words (qbgpu_matrix::cbits) when its table of distinct values
    // fits beside the columns: 4 bytes per entry instead of 12, and the products are bound by the matrix stream.  Handles built
    // as row shards -- a one-rank shard covering all rows too -- keep separate fp64 values: the multi-GPU drivers split their
    // cross parts by columns and rows (qbgpu_species_split_cross, qbgpu_row_view).  So do complex values.
    const int cbits = packed_col_bits(n);
    if (!rows_given && A->val_real) {
        const int max_table = (int)std::min<int64_t>(kPackedMaxTable, (int64_t)1 << (32 - cbits));
        int rc = value_dict_encode(A, max_table);           // (leaves a part whose table would not fit as it is)
        if (rc == QBGPU_OK) rc = value_dict_encode(C, max_table);
        if (rc) { qbgpu_destroy(A); return rc; }
    }
    { int rc = sjds_convert(A, true); if (rc == QBGPU_OK) rc = sjds_convert(C, true); if (rc) { qbgpu_destroy(A); return rc; } }
    for (qbgpu_matrix *P : {A, C}) {
        if (!P->ndict) continue;
        pack_codes_kernel<<<grid_rows(P->nnz), kPBlock, 0, c.stream>>>(P->nnz, (uint32_t *)P->col, (const uint8_t *)P->val, cbits);
        QB_LAUNCH_COUNT();
        QB_CU(cudaStreamSynchronize(c.stream));
        QB_CU(cudaGetLastError());
        cudaFree(P->val); P->val = nullptr; P->cbits = cbits;
    }
    std::vector<int32_t> order;
    make_slice_order(nloc, Dd, S->tile, order);
    QB_CU(upload(&C->slice_order, order.data(), order.size(), c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
#undef QB_CU
    S->matfree = false;
    A->convert_s = wall_s() - t0;
    *out = A;
    return QBGPU_OK;
}

// Row shards (multi-GPU): whole up configurations only, rows [u_lo * D_dn, u_hi * D_dn).  A shard has no permutation: its
// vectors -- x full length, y and z the local rows -- are in the internal order, like every sharded handle's are in "row order".
int species_build_matfree(qbgpu_matrix_t *out, const HostTables &T, const ModelParams &M, int api_complex, int flags, int64_t row_lo, int64_t row_hi)
{
    (void)flags;
    if (!out) return fail(QBGPU_ERR_ARG, "null handle pointer");
    *out = nullptr;
    const double t0 = wall_s();
    SpeciesHost H;
    qbgpu_matrix *A = nullptr;
    if (row_hi < 0) row_hi = T.dim;
    const bool shard = !(row_lo == 0 && row_hi == T.dim);
    QB_TRY(species_common(&A, T, M, api_complex, H, !shard));
    Species *S = (Species *)A->sp;
    if (shard) {
        if (row_lo < 0 || row_lo > row_hi || row_hi > T.dim || row_lo % S->Dd != 0 || (row_hi % S->Dd != 0))
        { qbgpu_destroy(A); return fail(QBGPU_ERR_ARG, "species order: a row shard must consist of whole up configurations (multiples of D_dn rows)"); }
        A->row_lo = row_lo; A->row_hi = row_hi;
    }
    S->matfree = true;
    if (!getenv("QBGPU_SPECIES_TILE")) S->tile = 128;       // (the matrix-free cross pass prefers the wider tile: 14.1 ms against 15.0)
    A->format = QBGPU_FORMAT_MATFREE;
    A->nnz = 0; A->nnz_input = 0;
    A->convert_s = wall_s() - t0;
    *out = A;
    return QBGPU_OK;
}

void species_destroy(qbgpu_matrix *A)
{
    if (!A || !A->sp) return;
    species_free((Species *)A->sp);
    A->sp = nullptr;
    cudaFree(A->perm); A->perm = nullptr;
    cudaFree(A->perm_inv); A->perm_inv = nullptr;
    if (A->second) { qbgpu_destroy(A->second); A->second = nullptr; }
}

int64_t species_bytes(const qbgpu_matrix *A)
{
    const Species *S = (const Species *)A->sp;
    int64_t b = S ? S->bytes : 0;
    if (A->second) {
        const int64_t ns = (A->n + 31) / 32;
        b += A->nnz * (int64_t)(4 + A->val_bytes()) + A->second->nnz * (int64_t)(4 + A->second->val_bytes());
        b += 2 * 8 * (A->n + 1) + 2 * 4 * ns * 32 + 4 * ns;        // two rowptr, two rowinfo, the slice order
    }
    return b;
}

// ------------------------------------------------------------------------------------------ matrix-free product
// pass 1: y = alpha * (diagonal + down hops) x + gamma x + beta z.  One thread per row, rows ascending: the gathers of a
// row fall into its own block x[iu, :].  Four hop entries per trip: their table loads, then their gathers, are issued
// together; past the end of the list the trip replays "0 * x[own row]".
// The block x[iu, :] of the row is xb[col0 .. col0 + D_dn): xb = x and col0 = iu * D_dn in global memory (GLOBAL: read-only
// path; n < 2^31, so the column fits 32 bits), or xb = the block staged in shared memory and col0 = 0.
template <typename VecT, bool GLOBAL, bool UNI = false>
__host__ __device__ __forceinline__ VecT kron_local_acc(const SpeciesView &V, const double *ampw, const double *diagk, uint32_t U, int32_t id,
                                                        const VecT *xb, uint32_t col0, VecT xi, double amp_uni = 0.0)
{
    using VT = VecTraits<VecT>;
    const uint32_t D = ld_ro(V.dlist + id);
    VecT acc = VT::zero();
    mac(acc, diagk[popc_hd(U & D)], xi);
    const int e1 = ld_ro(V.dptr + id + 1);
    int e = ld_ro(V.dptr + id);
    // full trips, no bounds checks; the next trip's table entries are fetched while this trip's gathers are in flight (a lane
    // reads its own list here, so a table load costs an L2 round trip that would otherwise sit in front of every gather)
    uint2 hn[4];
    bool more = e + 4 <= e1;
    if (more) {
QB_UNROLL
        for (int u = 0; u < 4; u++) hn[u] = ld_ro(V.dhop + e + u);
    }
    while (more) {
        uint2 h[4];
        VecT xv[4];
QB_UNROLL
        for (int u = 0; u < 4; u++) h[u] = hn[u];
        e += 4;
        more = e + 4 <= e1;
QB_UNROLL
        for (int u = 0; u < 4; u++) { if (GLOBAL) xv[u] = ld_ro(xb + (col0 + h[u].x)); else xv[u] = xb[col0 + h[u].x]; }
        if (more) {
QB_UNROLL
            for (int u = 0; u < 4; u++) hn[u] = ld_ro(V.dhop + e + u);
        }
QB_UNROLL
        for (int u = 0; u < 4; u++) mac(acc, UNI ? hop_value_uni(h[u].y, U, amp_uni) : hop_value(h[u].y, U, ampw), xv[u]);
    }
    if (e < e1) {                                           // the last, partial trip: past the end it replays 0 * x[own row]
        uint2 h[4];
        VecT xv[4];
QB_UNROLL
        for (int u = 0; u < 4; u++) h[u] = (e + u < e1) ? ld_ro(V.dhop + e + u) : make_uint2((uint32_t)id, 0u);
QB_UNROLL
        for (int u = 0; u < 4; u++) { if (GLOBAL) xv[u] = ld_ro(xb + (col0 + h[u].x)); else xv[u] = xb[col0 + h[u].x]; }
QB_UNROLL
        for (int u = 0; u < 4; u++) mac(acc, hop_value(h[u].y, U, ampw), xv[u]);
    }
    return acc;
}

// epilogue scalars of pass 1 (Lanczos step a like the stored kernels, spmv.cu)
__device__ __forceinline__ void local_scalars(int scal_mode, const double *sc, double2 &alpha, double2 &gamma, double2 &beta)
{
    if (scal_mode != 0) {
        const double sx = sc[0], sz = sc[1], bprev = sc[2];
        alpha = make_double2(sx, 0.0);
        gamma = make_double2(0.0, 0.0);
        beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
    }
}

// BLOCK = 256, grid-stride (default), or BLOCK = 1024 with one contiguous range of rows per CTA (variant 1: one
// CTA per SM then walks through the blocks x[iu, :] one after the other, so that L1 holds the block being gathered from).
// Rows [row0, row0 + nloc) of the operator (a shard: whole up configurations); x is the full vector, y and z the local rows.
template <typename VecT, int BLOCK, bool RANGES, bool UNI>
__global__ void __launch_bounds__(BLOCK, 1024 / BLOCK)
kron_local_kernel(SpeciesView V, int64_t row0, int64_t nloc, const double *__restrict__ ampw_g, const double *__restrict__ diagk_g, double amp_uni,
                  const VecT *__restrict__ x, const VecT *z, VecT *y,
                  double2 alpha, double2 gamma, double2 beta, int scal_mode, const double *__restrict__ sc)
{
    using VT = VecTraits<VecT>;
    __shared__ double ampw[kMaxWeight + 1], diagk[kMaxDbl + 1];
    for (int k = threadIdx.x; k <= kMaxWeight; k += blockDim.x) ampw[k] = ampw_g[k];
    for (int k = threadIdx.x; k <= kMaxDbl; k += blockDim.x) diagk[k] = diagk_g[k];
    __syncthreads();
    local_scalars(scal_mode, sc, alpha, gamma, beta);
    const bool use_gamma = (gamma.x != 0.0 || gamma.y != 0.0);
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    int64_t q0, q1, step;                                   // local row indices
    if (RANGES) {
        const int64_t chunk = ((nloc + gridDim.x - 1) / gridDim.x + BLOCK - 1) / BLOCK * BLOCK;
        q0 = (int64_t)blockIdx.x * chunk + threadIdx.x; q1 = min(nloc, ((int64_t)blockIdx.x + 1) * chunk); step = BLOCK;
    } else {
        q0 = (int64_t)blockIdx.x * BLOCK + threadIdx.x; q1 = nloc; step = (int64_t)gridDim.x * BLOCK;
    }
    for (int64_t q = q0; q < q1; q += step) {
        const int64_t p = row0 + q;
        const int64_t iu = p / V.Dd;
        const int32_t id = (int32_t)(p - iu * V.Dd);
        const VecT xi = ld_ro(x + p);
        const VecT acc = kron_local_acc<VecT, true, UNI>(V, ampw, diagk, ld_ro(V.ulist + iu), id, x, (uint32_t)(iu * V.Dd), xi, amp_uni);
        VecT out = VT::scale(alpha, acc);
        if (use_gamma) out = VT::add(out, VT::scale(gamma, xi));
        if (use_beta) out = VT::add(out, VT::scale(beta, z[q]));
        y[q] = out;
    }
}

// variant 2: one CTA of 1024 threads per up configuration; the block x[iu, :] (D_dn entries: 206 KB of complex
// numbers for the 4x4 lattice) is staged in shared memory once and every gather of the block's rows reads it from there.
template <typename VecT, bool UNI>
__global__ void __launch_bounds__(1024, 1)
kron_local_smem_kernel(SpeciesView V, int64_t u_lo, int64_t u_cnt, const double *__restrict__ ampw_g, const double *__restrict__ diagk_g, double amp_uni,
                       const VecT *__restrict__ x, const VecT *z, VecT *y,
                       double2 alpha, double2 gamma, double2 beta, int scal_mode, const double *__restrict__ sc)
{
    using VT = VecTraits<VecT>;
    extern __shared__ double2 kron_smem_raw[];              // 16-byte aligned for either vector type
    VecT *xs = reinterpret_cast<VecT *>(kron_smem_raw);
    __shared__ double ampw[kMaxWeight + 1], diagk[kMaxDbl + 1];
    for (int k = threadIdx.x; k <= kMaxWeight; k += blockDim.x) ampw[k] = ampw_g[k];
    for (int k = threadIdx.x; k <= kMaxDbl; k += blockDim.x) diagk[k] = diagk_g[k];
    local_scalars(scal_mode, sc, alpha, gamma, beta);
    const bool use_gamma = (gamma.x != 0.0 || gamma.y != 0.0);
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    const int32_t Dd = (int32_t)V.Dd;
    for (int64_t il = blockIdx.x; il < u_cnt; il += gridDim.x) {
        const int64_t iu = u_lo + il;
        __syncthreads();                                    // the previous block's gathers are done (and the tables are loaded)
        const VecT *xg = x + iu * V.Dd;
        for (int32_t k = threadIdx.x; k < Dd; k += 1024) xs[k] = ld_ro(xg + k);
        __syncthreads();
        const uint32_t U = ld_ro(V.ulist + iu);
        for (int32_t id = threadIdx.x; id < Dd; id += 1024) {
            const VecT xi = xs[id];
            const VecT acc = kron_local_acc<VecT, false, UNI>(V, ampw, diagk, U, id, xs, 0u, xi, amp_uni);
            VecT out = VT::scale(alpha, acc);
            if (use_gamma) out = VT::add(out, VT::scale(gamma, xi));
            if (use_beta) out = VT::add(out, VT::scale(beta, z[il * V.Dd + id]));
            y[il * V.Dd + id] = out;
        }
    }
}

// pass 2: y += alpha * (up hops) x, with the running dots of the finished y.  One warp per 32 consecutive down indices
// of one up configuration; the hop list is warp-uniform (broadcast loads) and every gather is a contiguous 32-entry
// segment x[iu', id .. id+31].  Items are enumerated tile by tile (all iu for the down indices of one tile), so the
// columns a tile gathers stay in L2.
struct CrossItems {
    int64_t nitems, full_items, per_tile;   // per_tile = Du * cpt warp items in every tile but the last
    int W, cpt, cpt_last, ntile;            // tile width, 32-wide chunks per tile row (last tile: cpt_last)
};

__host__ __device__ __forceinline__ CrossItems cross_items(int64_t Du, int64_t Dd, int W)
{
    CrossItems I;
    I.W = W; I.cpt = W / 32;
    I.ntile = (int)((Dd + W - 1) / W);
    const int64_t w_last = Dd - (int64_t)(I.ntile - 1) * W;
    I.cpt_last = (int)((w_last + 31) / 32);
    I.per_tile = Du * I.cpt;
    I.full_items = (int64_t)(I.ntile - 1) * I.per_tile;
    I.nitems = I.full_items + Du * I.cpt_last;
    return I;
}

// warp item `it`, lane -> (iu, id); id may be >= Dd in the last chunk of a tile row (idle lane)
__host__ __device__ __forceinline__ void cross_item_at(const CrossItems &I, int64_t it, int lane, int64_t &iu, int64_t &id)
{
    int64_t tau, ch;
    if (it < I.full_items) { tau = it / I.per_tile; const int64_t rem = it - tau * I.per_tile; iu = rem / I.cpt; ch = rem - iu * I.cpt; }
    else { const int64_t k2 = it - I.full_items; tau = I.ntile - 1; iu = k2 / I.cpt_last; ch = k2 - iu * I.cpt_last; }
    id = tau * I.W + ch * 32 + lane;
}

// FILTER: only the hops whose target configuration lies in [c_lo, c_hi) (a column part of a shard)
template <typename VecT, bool FILTER = false, bool UNI = false>
__host__ __device__ __forceinline__ VecT kron_cross_acc(const SpeciesView &V, const double *ampw, int64_t iu, int64_t idc, const VecT *x,
                                                        int64_t c_lo = 0, int64_t c_hi = 0, double amp_uni = 0.0)
{
    using VT = VecTraits<VecT>;
    const uint32_t D = ld_ro(V.dlist + idc);
    const uint32_t Dd32 = (uint32_t)V.Dd, idc32 = (uint32_t)idc;
    const int e1 = ld_ro(V.uptr + iu + 1);
    VecT acc = VT::zero();
    int e = ld_ro(V.uptr + iu);
    for (; e + 4 <= e1; e += 4) {                           // full trips: no bounds checks (the list is warp-uniform)
        uint2 h[4];
        VecT xv[4];
QB_UNROLL
        for (int u = 0; u < 4; u++) {
            h[u] = ld_ro(V.uhop + e + u);
            if (FILTER && ((int64_t)h[u].x < c_lo || (int64_t)h[u].x >= c_hi)) h[u] = make_uint2((uint32_t)iu, 0u);   // replays 0 * x[own row]
        }
QB_UNROLL
        for (int u = 0; u < 4; u++) xv[u] = ld_ro(x + (h[u].x * Dd32 + idc32));      // n < 2^31: the column fits 32 bits
QB_UNROLL
        for (int u = 0; u < 4; u++) mac(acc, (UNI && !FILTER) ? hop_value_uni(h[u].y, D, amp_uni) : hop_value(h[u].y, D, ampw), xv[u]);
    }
    if (e < e1) {                                           // the last, partial trip
        uint2 h[4];
        VecT xv[4];
QB_UNROLL
        for (int u = 0; u < 4; u++) {
            h[u] = (e + u < e1) ? ld_ro(V.uhop + e + u) : make_uint2((uint32_t)iu, 0u);
            if (FILTER && ((int64_t)h[u].x < c_lo || (int64_t)h[u].x >= c_hi)) h[u] = make_uint2((uint32_t)iu, 0u);
        }
QB_UNROLL
        for (int u = 0; u < 4; u++) xv[u] = ld_ro(x + (h[u].x * Dd32 + idc32));      // n < 2^31: the column fits 32 bits
QB_UNROLL
        for (int u = 0; u < 4; u++) mac(acc, hop_value(h[u].y, D, ampw), xv[u]);
    }
    return acc;
}

// The items enumerate the LOCAL up configurations [u_lo, u_lo + u_cnt) of the handle.  FIRST: y = alpha acc + beta z (a
// column part without the local pass that opens the product); otherwise y += alpha acc.
template <typename VecT, bool DOTS, bool FILTER, bool FIRST, bool UNI>
__global__ void __launch_bounds__(kPBlock, 4)
kron_cross_kernel(SpeciesView V, CrossItems I, int64_t u_lo, int64_t c_lo, int64_t c_hi, const double *__restrict__ ampw_g, double amp_uni,
                  const VecT *__restrict__ x, const VecT *z, VecT *y, double2 alpha, double2 beta, int scal_mode,
                  const double *__restrict__ sc, double *dots_out, double *partials, unsigned *ticket)
{
    using VT = VecTraits<VecT>;
    __shared__ double ampw[kMaxWeight + 1];
    for (int k = threadIdx.x; k <= kMaxWeight; k += blockDim.x) ampw[k] = ampw_g[k];
    __syncthreads();
    double dot_scale = 1.0;
    if (scal_mode != 0) {
        alpha = make_double2(sc[0], 0.0); dot_scale = sc[0];
        beta = scal_mode == 1 ? make_double2(-sc[2] * sc[1], 0.0) : make_double2(1.0, 0.0);
    }
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    constexpr int WPB = kPBlock / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double d[3] = {0.0, 0.0, 0.0};
    for (int64_t it = (int64_t)blockIdx.x * WPB + warp; it < I.nitems; it += (int64_t)gridDim.x * WPB) {
        int64_t il, id;
        cross_item_at(I, it, lane, il, id);
        const int64_t iu = u_lo + il;
        const bool live = id < V.Dd;
        const int64_t idc = live ? id : V.Dd - 1;           // idle lanes of the last chunk replay a valid column
        const VecT acc = kron_cross_acc<VecT, FILTER, UNI>(V, ampw, iu, idc, x, c_lo, c_hi, amp_uni);
        if (live) {
            const int64_t q = il * V.Dd + id;               // local row
            VecT out = VT::scale(alpha, acc);
            if (FIRST) { if (use_beta) out = VT::add(out, VT::scale(beta, z[q])); }
            else out = VT::add(y[q], out);
            y[q] = out;
            if (DOTS) {
                const double2 qd = VT::conj_mul(ld_ro(x + iu * V.Dd + id), out);
                d[0] += qd.x; d[1] += qd.y; d[2] += VT::abs2(out);
            }
        }
    }
    if (DOTS) {
        d[0] *= dot_scale; d[1] *= dot_scale;
        block_reduce_finalize<3, kPBlock>(d, partials, ticket, dots_out);
    }
}

static int g_kron_local_variant = 0;       // qbgpu_debug_set_variant(1000 + v)
void set_kron_local_variant(int v) { g_kron_local_variant = v; }

template <typename VecT, bool DOTS, bool FILTER, bool FIRST, bool UNI = false>
static int launch_kron_cross(const qbgpu_matrix *A, const FusedArgs &a, const SpeciesView &V, const CrossItems &I, int64_t u_lo)
{
    Context &c = ctx();
    const Species *S = (const Species *)A->sp;
    auto kern = kron_cross_kernel<VecT, DOTS, FILTER, FIRST, UNI>;
    static int bps = 0;
    if (bps == 0) { QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, kPBlock, 0)); if (bps < 1) bps = 1; }
    const int64_t want = (I.nitems + (kPBlock / 32) - 1) / (kPBlock / 32);
    int64_t cap = (int64_t)c.num_sms * bps;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    if (want < 1) return QBGPU_OK;
    kern<<<(int)(want < cap ? want : cap), kPBlock, 0, c.stream>>>(V, I, u_lo, A->sp_col_lo, A->sp_col_hi, S->ampw, S->amp_uni, (const VecT *)a.x, (const VecT *)a.z,
                                                                    (VecT *)a.y, a.alpha, a.beta, a.scal_mode, a.sc, a.dots, c.partials, c.ticket);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

template <typename VecT>
static int launch_kron(const qbgpu_matrix *A, const FusedArgs &a)
{
    Context &c = ctx();
    const Species *S = (const Species *)A->sp;
    const int64_t nloc = A->nrows(), row0 = A->row_lo;
    if (nloc == 0) return QBGPU_OK;
    const int64_t u_lo = row0 / S->Dd, u_cnt = nloc / S->Dd;
    const SpeciesView V = view_of(S);
    const bool filter = A->sp_col_lo >= 0;
    if (A->sp_has_local) {
        // pass 1 variants: 0 grid-stride / 256 threads (default), 1 contiguous row ranges / 1024 threads,
        // 2 block staged in shared memory (falls back to 0 when D_dn entries do not fit)
        const int variant = g_kron_local_variant;
        const size_t stage_bytes = sizeof(VecT) * (size_t)S->Dd;
        const bool uni = S->amp_uni != 0.0;              // every bond with the same multiplicity: amplitude as an argument
        if (variant == 2 && stage_bytes <= 225 * 1024) {
            auto kern = uni ? kron_local_smem_kernel<VecT, true> : kron_local_smem_kernel<VecT, false>;
            QB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
            const int64_t grid = u_cnt < c.num_sms ? u_cnt : c.num_sms;
            kern<<<(int)grid, 1024, stage_bytes, c.stream>>>(V, u_lo, u_cnt, S->ampw, S->diagk, S->amp_uni, (const VecT *)a.x, (const VecT *)a.z, (VecT *)a.y,
                                                             a.alpha, a.gamma, a.beta, a.scal_mode, a.sc);
        } else if (variant == 1) {
            auto kern = uni ? kron_local_kernel<VecT, 1024, true, true> : kron_local_kernel<VecT, 1024, true, false>;
            kern<<<c.num_sms, 1024, 0, c.stream>>>(V, row0, nloc, S->ampw, S->diagk, S->amp_uni, (const VecT *)a.x, (const VecT *)a.z, (VecT *)a.y,
                                                   a.alpha, a.gamma, a.beta, a.scal_mode, a.sc);
        } else {
            auto kern = uni ? kron_local_kernel<VecT, kPBlock, false, true> : kron_local_kernel<VecT, kPBlock, false, false>;
            int bps = 0;
            QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, kPBlock, 0));
            if (bps < 1) bps = 1;
            const int64_t want = (nloc + kPBlock - 1) / kPBlock, cap = (int64_t)c.num_sms * bps;
            kern<<<(int)(want < cap ? want : cap), kPBlock, 0, c.stream>>>(V, row0, nloc, S->ampw, S->diagk, S->amp_uni, (const VecT *)a.x, (const VecT *)a.z,
                                                                            (VecT *)a.y, a.alpha, a.gamma, a.beta, a.scal_mode, a.sc);
        }
        QB_LAUNCH_COUNT();
        QB_CUDA(cudaGetLastError());
    } else if (a.scal_mode == 0 && (a.gamma.x != 0.0 || a.gamma.y != 0.0)) {
        return fail(QBGPU_ERR_ARG, "a column part without the diagonal block cannot carry the gamma*x term");
    }
    const CrossItems I = cross_items(u_cnt, S->Dd, S->tile);
    // does this call open the product (y = ... + beta z) or continue it (y += ...)?  After the local pass it always continues.
    const bool accumulate = A->sp_has_local || a.scal_mode == 2 ||
                            (a.scal_mode == 0 && a.z == a.y && a.beta.x == 1.0 && a.beta.y == 0.0);
    if (!accumulate && (a.beta.x != 0.0 || a.beta.y != 0.0 || a.scal_mode == 1) && !a.z) return fail(QBGPU_ERR_ARG, "beta != 0 needs z");
    if (a.dots) {
        if (filter) return accumulate ? launch_kron_cross<VecT, true, true, false>(A, a, V, I, u_lo) : launch_kron_cross<VecT, true, true, true>(A, a, V, I, u_lo);
        if (S->amp_uni != 0.0) return launch_kron_cross<VecT, true, false, false, true>(A, a, V, I, u_lo);
        return launch_kron_cross<VecT, true, false, false>(A, a, V, I, u_lo);
    }
    if (filter) return accumulate ? launch_kron_cross<VecT, false, true, false>(A, a, V, I, u_lo) : launch_kron_cross<VecT, false, true, true>(A, a, V, I, u_lo);
    if (S->amp_uni != 0.0) return launch_kron_cross<VecT, false, false, false, true>(A, a, V, I, u_lo);
    return launch_kron_cross<VecT, false, false, false>(A, a, V, I, u_lo);
}

// Both handle kinds: pass 1 carries the caller's epilogue (alpha, gamma, beta*z) without the dots, pass 2 accumulates
// into the same y and carries the dots -- exactly the first / later column blocks of a sharded product (spmv.cu).
int launch_spmv_species(const qbgpu_matrix *A, const FusedArgs &a)
{
    const Species *S = (const Species *)A->sp;
    if (!S) return fail(QBGPU_ERR_STATE, "not a species-order handle");
    if (S->matfree) return A->api_complex ? launch_kron<double2>(A, a) : launch_kron<double>(A, a);
    if (!A->second) return fail(QBGPU_ERR_STATE, "species-order handle without its cross part");
    qbgpu_matrix L = *A;                                    // plain views: the production kernels see two ordinary matrices
    L.sp = nullptr; L.second = nullptr; L.perm = nullptr; L.perm_inv = nullptr;
    FusedArgs a1 = a;
    a1.dots = nullptr;
    a1.y_ref = nullptr;                                     // (the fused way out belongs to pass 2)
    // pass 1: every gather stays inside the block of one up configuration -> the block of x lives in shared memory
    QB_TRY(launch_spmv(&L, a1));                            // (block_D set: launch_spmv_sjds takes the block-local kernel when it fits)
    qbgpu_matrix C = *A->second;
    C.api_complex = A->api_complex;                        // a real view of the handle (fp64 vectors) covers both parts
    FusedArgs a2;
    a2.x = a.x; a2.y = a.y; a2.z = a.y; a2.dots = a.dots;
    a2.beta = make_double2(1.0, 0.0);
    if (a.scal_mode != 0) { a2.scal_mode = 2; a2.sc = a.sc; }
    else a2.alpha = a.alpha;
    if (a.y_ref) { a2.y_ref = a.y_ref; a2.out_alpha = a.out_alpha; a2.perm_inv = A->perm_inv; }
    return launch_spmv(&C, a2);
}

// Column parts of a matrix-free handle or shard (qbgpu_split_columns; the pipelined / peer-pull exchanges of dist.py multiply
// part p as soon as the slice of x owned by rank p has arrived): views that share the tables.  Part p keeps the up-hops whose
// target configuration lies in [bounds[p], bounds[p+1]) / D_dn; the part whose range contains the handle's first row also runs
// the whole local pass (its gathers never leave the handle's own rows).  Bounds must be multiples of D_dn.
int species_split_columns(qbgpu_matrix *A, int nparts, const int64_t *bounds, qbgpu_matrix_t *parts)
{
    QB_TRY(ensure_init());
    if (!A || !bounds || !parts || nparts < 1) return fail(QBGPU_ERR_ARG, "split_columns: bad argument");
    const Species *S = (const Species *)A->sp;
    if (!S || !S->matfree) return fail(QBGPU_ERR_STATE, "split_columns: of the species-order handles only the matrix-free ones can be split");
    if (A->sp_col_lo >= 0) return fail(QBGPU_ERR_STATE, "split_columns: already a column part");
    if (bounds[0] != 0 || bounds[nparts] != A->n) return fail(QBGPU_ERR_ARG, "split_columns: bounds must run from 0 to n");
    for (int p = 0; p <= nparts; p++) {
        if (bounds[p] % S->Dd != 0) return fail(QBGPU_ERR_ARG, "split_columns: species-order bounds must be multiples of D_dn (whole up configurations)");
        if (p && bounds[p] < bounds[p - 1]) return fail(QBGPU_ERR_ARG, "split_columns: bounds must be non-decreasing");
    }
    bool local_given = false;
    for (int p = 0; p < nparts; p++) {
        auto *V = new qbgpu_matrix(*A);
        V->borrowed = true;
        V->perm = nullptr; V->perm_inv = nullptr; V->perm_x = V->perm_y = nullptr;
        V->sp_col_lo = bounds[p] / S->Dd; V->sp_col_hi = bounds[p + 1] / S->Dd;
        V->sp_has_local = !local_given && bounds[p] <= A->row_lo && A->row_lo < bounds[p + 1];
        local_given = local_given || V->sp_has_local;
        parts[p] = V;
    }
    if (!local_given) {                                     // (an empty shard: no rows, no local pass needed)
        if (A->nrows() != 0) { for (int p = 0; p < nparts; p++) { qbgpu_destroy(parts[p]); parts[p] = nullptr; } return fail(QBGPU_ERR_STATE, "split_columns: no part contains the shard's rows"); }
    }
    return QBGPU_OK;
}

// --------------------------------------------------------------------------------------- order of the vectors
template <typename DstT, typename SrcT> __device__ __forceinline__ DstT cvt(SrcT v);
template <> __device__ __forceinline__ double cvt<double, double>(double v) { return v; }
template <> __device__ __forceinline__ double2 cvt<double2, double>(double v) { return make_double2(v, 0.0); }
template <> __device__ __forceinline__ double cvt<double, double2>(double2 v) { return v.x; }
template <> __device__ __forceinline__ double2 cvt<double2, double2>(double2 v) { return v; }

// Both ways GATHER (coalesced writes, reads that stay inside the rectangle one block of the reference's order maps to, so the
// sectors they touch are complete within the L2's reach): a scattering way in wrote partial sectors -- 1.55 ms against 0.9 ms
// for the way out on BASELINE config 3 (profiles/r02_mv_reference_order_launches.csv).
template <typename SrcT, typename DstT>
__global__ void __launch_bounds__(kPBlock) to_native_kernel(int64_t n, const int32_t *__restrict__ perm_inv, const SrcT *__restrict__ src, DstT *dst)
{
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x)
        dst[p] = cvt<DstT, SrcT>(src[perm_inv[p]]);
}

// The way in, tile by tile: one CTA takes one block of the reference's order (the rows of one odd-site label: contiguous there,
// a rectangle [iu0, iu0 + Cu) x [id0, id0 + Cd) of the internal order, see build_host_tables), reads it coalesced, transposes it
// into the rectangle's own row-major order in shared memory and writes Cu runs of Cd contiguous entries.  Both sides touch
// every sector once (the element-wise gather read 7.2 GB for a 2.65 GB vector on BASELINE config 3).  CHECK: *flag = 1 as soon
// as one imaginary part of the source is not zero (the real-content route of mv_species).
// per block of the reference's order: the rectangle it maps to (computed once, when the handle is created)
__global__ void __launch_bounds__(kPBlock) tile_descriptor_kernel(int64_t nblk, const int64_t *__restrict__ blk_start, int32_t Dd,
                                                                  const int32_t *__restrict__ perm, int4 *desc)
{
    __shared__ int s_lo_u, s_hi_u, s_lo_d, s_hi_d;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const int64_t r0 = blk_start[blk];
        const int na = (int)(blk_start[blk + 1] - r0);
        if (threadIdx.x == 0) { s_lo_u = 0x7fffffff; s_hi_u = -1; s_lo_d = 0x7fffffff; s_hi_d = -1; }
        __syncthreads();
        int lo_u = 0x7fffffff, hi_u = -1, lo_d = 0x7fffffff, hi_d = -1;
        for (int t = threadIdx.x; t < na; t += kPBlock) {
            const int32_t p = perm[r0 + t];
            const int iu = p / Dd, id = p - iu * Dd;
            lo_u = min(lo_u, iu); hi_u = max(hi_u, iu); lo_d = min(lo_d, id); hi_d = max(hi_d, id);
        }
        lo_u = __reduce_min_sync(0xffffffffu, lo_u); hi_u = __reduce_max_sync(0xffffffffu, hi_u);
        lo_d = __reduce_min_sync(0xffffffffu, lo_d); hi_d = __reduce_max_sync(0xffffffffu, hi_d);
        if ((threadIdx.x & 31) == 0) { atomicMin(&s_lo_u, lo_u); atomicMax(&s_hi_u, hi_u); atomicMin(&s_lo_d, lo_d); atomicMax(&s_hi_d, hi_d); }
        __syncthreads();
        if (threadIdx.x == 0) {
            const int cu = s_hi_u - s_lo_u + 1, cd = s_hi_d - s_lo_d + 1;
            desc[blk] = make_int4(s_lo_u, s_lo_d, ((int64_t)cu * cd == na) ? cd : 0, na);     // .z == 0: not a rectangle (never, by construction)
        }
        __syncthreads();
    }
}

constexpr int kTBlock = 512;
template <typename SrcT, typename DstT, bool CHECK>
__global__ void __launch_bounds__(kTBlock) to_native_tiled_kernel(int64_t nblk, const int64_t *__restrict__ blk_start, const int4 *__restrict__ desc, int32_t Dd,
                                                                  const int32_t *__restrict__ perm, const SrcT *__restrict__ src, DstT *dst, int *flag)
{
    extern __shared__ __align__(16) unsigned char tile_raw[];
    DstT *tile = (DstT *)tile_raw;
    bool any = false;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const int64_t r0 = blk_start[blk];
        const int4 d = desc[blk];
        const int iu0 = d.x, id0 = d.y, cd = d.z, na = d.w;
        constexpr int UN = 4;                               // loads of four rounds first, then their scatters
        for (int t0 = threadIdx.x; t0 < na; t0 += UN * kTBlock) {
            int32_t p[UN];
            SrcT v[UN];
#pragma unroll
            for (int u = 0; u < UN; u++) { const int t = t0 + u * kTBlock; if (t < na) { p[u] = perm[r0 + t]; v[u] = src[r0 + t]; } }
#pragma unroll
            for (int u = 0; u < UN; u++) {
                const int t = t0 + u * kTBlock;
                if (t < na) {
                    if constexpr (CHECK) any = any || (v[u].y != 0.0);
                    if (cd) { const int iu = p[u] / Dd, id = p[u] - iu * Dd; tile[(iu - iu0) * cd + (id - id0)] = cvt<DstT, SrcT>(v[u]); }
                    else dst[p[u]] = cvt<DstT, SrcT>(v[u]);
                }
            }
        }
        __syncthreads();
        if (cd) {
            for (int t = threadIdx.x; t < na; t += kTBlock) {
                const int row = t / cd, col = t - row * cd;
                dst[(int64_t)(iu0 + row) * Dd + id0 + col] = tile[t];
            }
        }
        __syncthreads();
    }
    if constexpr (CHECK) { if (any) *(volatile int *)flag = 1; }
}

template <typename SrcT, typename DstT, bool CHECK>
static int launch_to_native_tiled(const qbgpu_matrix *A, const void *src, void *dst, int *flag)
{
    Context &c = ctx();
    const Species *S = (const Species *)A->sp;
    auto kern = to_native_tiled_kernel<SrcT, DstT, CHECK>;
    const size_t smem = sizeof(DstT) * (size_t)S->blk_max_rows;
    static size_t smem_set = 0;
    if (smem > smem_set) { QB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); smem_set = smem; }
    static int bps = 0;
    static size_t bps_smem = 0;
    if (bps == 0 || bps_smem != smem) { QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, kTBlock, smem)); bps_smem = smem; if (bps < 1) bps = 1; }
    int64_t g = S->nblk < (int64_t)c.num_sms * bps ? S->nblk : (int64_t)c.num_sms * bps;      // one wave of resident CTAs, blocks round-robin
    if (g < 1) g = 1;
    kern<<<(int)g, kTBlock, smem, c.stream>>>(S->nblk, S->blk_start, S->blk_desc, (int32_t)S->Dd, A->perm, (const SrcT *)src, (DstT *)dst, flag);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}
// the tiles fit in shared memory and the handle carries the block table
static bool to_native_tiled_ok(const qbgpu_matrix *A, size_t elem)
{
    const Species *S = (const Species *)A->sp;
    return S && S->blk_start && S->blk_desc && S->nblk > 0 && elem * (size_t)S->blk_max_rows <= 200 * 1024;
}

// the way in of the real-content product: dst[p] = Re src[perm_inv[p]]; *flag = 1 as soon as one imaginary part is not zero
__global__ void __launch_bounds__(kPBlock) to_native_real_check_kernel(int64_t n, const int32_t *__restrict__ perm_inv, const double2 *__restrict__ src,
                                                                       double *dst, int *flag)
{
    bool any = false;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
        const double2 v = src[perm_inv[p]];
        dst[p] = v.x;
        any = any || (v.y != 0.0);
    }
    if (any) *(volatile int *)flag = 1;
}

template <typename SrcT, typename DstT, bool ACC>
__global__ void __launch_bounds__(kPBlock) from_native_kernel(int64_t n, const int32_t *__restrict__ perm, const SrcT *__restrict__ src, DstT *dst,
                                                              double2 a, double2 b)
{
    using VT = VecTraits<DstT>;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
        DstT v = VT::scale(a, cvt<DstT, SrcT>(src[perm[r]]));
        if (ACC) v = VT::add(v, VT::scale(b, dst[r]));
        dst[r] = v;
    }
}

int vec_to_native(const qbgpu_matrix *A, bool src_cplx, bool dst_cplx, const void *src, void *dst)
{
    if (!A || !A->perm || !A->perm_inv) return fail(QBGPU_ERR_STATE, "vec_to_native: the handle has no internal order");
    Context &c = ctx();
    const int64_t n = A->n;
    const int g = grid_rows(n);
    if (to_native_tiled_ok(A, dst_cplx ? 16 : 8)) {
        if (src_cplx && dst_cplx) return launch_to_native_tiled<double2, double2, false>(A, src, dst, nullptr);
        if (src_cplx) return launch_to_native_tiled<double2, double, false>(A, src, dst, nullptr);
        if (dst_cplx) return launch_to_native_tiled<double, double2, false>(A, src, dst, nullptr);
        return launch_to_native_tiled<double, double, false>(A, src, dst, nullptr);
    }
    if (src_cplx && dst_cplx) to_native_kernel<double2, double2><<<g, kPBlock, 0, c.stream>>>(n, A->perm_inv, (const double2 *)src, (double2 *)dst);
    else if (src_cplx) to_native_kernel<double2, double><<<g, kPBlock, 0, c.stream>>>(n, A->perm_inv, (const double2 *)src, (double *)dst);
    else if (dst_cplx) to_native_kernel<double, double2><<<g, kPBlock, 0, c.stream>>>(n, A->perm_inv, (const double *)src, (double2 *)dst);
    else to_native_kernel<double, double><<<g, kPBlock, 0, c.stream>>>(n, A->perm_inv, (const double *)src, (double *)dst);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

template <typename SrcT, typename DstT>
static int from_native_typed(const qbgpu_matrix *A, const void *src, void *dst, double2 a, double2 b)
{
    Context &c = ctx();
    const int64_t n = A->n;
    const int g = grid_rows(n);
    if (b.x != 0.0 || b.y != 0.0) from_native_kernel<SrcT, DstT, true><<<g, kPBlock, 0, c.stream>>>(n, A->perm, (const SrcT *)src, (DstT *)dst, a, b);
    else from_native_kernel<SrcT, DstT, false><<<g, kPBlock, 0, c.stream>>>(n, A->perm, (const SrcT *)src, (DstT *)dst, a, b);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

int vec_from_native(const qbgpu_matrix *A, bool src_cplx, bool dst_cplx, const void *src, void *dst, double2 a, double2 b)
{
    if (!A || !A->perm) return fail(QBGPU_ERR_STATE, "vec_from_native: the handle has no internal order");
    if (src_cplx && dst_cplx) return from_native_typed<double2, double2>(A, src, dst, a, b);
    if (src_cplx) return from_native_typed<double2, double>(A, src, dst, a, b);
    if (dst_cplx) return from_native_typed<double, double2>(A, src, dst, a, b);
    return from_native_typed<double, double>(A, src, dst, a, b);
}

// y = alpha * H x + beta * y with the vectors in the REFERENCE's order (qbgpu_{d,z}mv): permute in, two passes, permute
// out (the scaling and the beta*y term ride in the way out).
int mv_species(qbgpu_matrix *A, double2 alpha, const void *x, double2 beta, void *y, int where)
{
    Context &c = ctx();
    const bool cplx = A->api_complex;
    const size_t vb = cplx ? 16 : 8;
    const size_t bytes = vb * (size_t)A->n;
    // staging vectors in the internal order: the handle's own (lazily allocated, freed by destroy); a view (e.g. the fp64
    // view of qbgpu_real_view) owns nothing and borrows the context's staging vectors, which host-vector products need themselves
    void *px = nullptr, *py = nullptr;
    if (!A->borrowed) {
        if (!A->perm_x) QB_CUDA(cudaMalloc(&A->perm_x, bytes));
        if (!A->perm_y) QB_CUDA(cudaMalloc(&A->perm_y, bytes));
        px = A->perm_x; py = A->perm_y;
    } else {
        if (where != QBGPU_DEVICE) return fail(QBGPU_ERR_STATE, "host-vector products on a view of a species-order handle: use the owning handle");
        if (c.stage_x_bytes < bytes) { if (c.stage_x) QB_CUDA(cudaFree(c.stage_x)); c.stage_x = nullptr; c.stage_x_bytes = 0; QB_CUDA(cudaMalloc(&c.stage_x, bytes)); c.stage_x_bytes = bytes; }
        if (c.stage_y_bytes < bytes) { if (c.stage_y) QB_CUDA(cudaFree(c.stage_y)); c.stage_y = nullptr; c.stage_y_bytes = 0; QB_CUDA(cudaMalloc(&c.stage_y, bytes)); c.stage_y_bytes = bytes; }
        px = c.stage_x; py = c.stage_y;
    }
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    const void *xd = x;
    void *yd = y;
    if (where == QBGPU_HOST) {
        if (c.stage_x_bytes < bytes) { if (c.stage_x) QB_CUDA(cudaFree(c.stage_x)); c.stage_x = nullptr; c.stage_x_bytes = 0; QB_CUDA(cudaMalloc(&c.stage_x, bytes)); c.stage_x_bytes = bytes; }
        if (c.stage_y_bytes < bytes) { if (c.stage_y) QB_CUDA(cudaFree(c.stage_y)); c.stage_y = nullptr; c.stage_y_bytes = 0; QB_CUDA(cudaMalloc(&c.stage_y, bytes)); c.stage_y_bytes = bytes; }
        QB_CUDA(cudaMemcpyAsync(c.stage_x, x, bytes, cudaMemcpyHostToDevice, c.stream));
        if (use_beta) QB_CUDA(cudaMemcpyAsync(c.stage_y, y, bytes, cudaMemcpyHostToDevice, c.stream));
        xd = c.stage_x; yd = c.stage_y;
    } else if (where != QBGPU_DEVICE) return fail(QBGPU_ERR_ARG, "where must be QBGPU_HOST or QBGPU_DEVICE");
    // Real content behind the complex API: through model<complex<double>> every vector is complex<double>, but with real
    // couplings H is real (val_real) and so is every vector the reference's flows produce (SURVEY F3).  The way in looks at
    // the imaginary parts while it permutes (one pass either way); if they are all exactly zero the two passes run on the
    // fp64 copy -- half the vector bytes, half the gather sectors, the block of x fits the shared memory of pass 1 -- and the
    // way out widens the result.  Exact: the real parts go through the identical fma sequence, the imaginary parts are exact
    // zeros either way.  A vector with any non-zero imaginary part takes the complex passes (QBGPU_MV_REAL_MODE=0: always).
    static const bool real_mode_on = !(getenv("QBGPU_MV_REAL_MODE") && atoi(getenv("QBGPU_MV_REAL_MODE")) == 0);
    const Species *S = (const Species *)A->sp;
    int *flag = (int *)(c.scal_dev + 57);
    auto complex_route = [&]() -> int {
        QB_TRY(vec_to_native(A, cplx, cplx, xd, px));
        FusedArgs fa;
        fa.x = px; fa.y = py;
        QB_TRY(launch_spmv(A, fa));
        return vec_from_native(A, cplx, cplx, py, yd, alpha, beta);
    };
    auto read_flag = [&](int &h) -> int {
        h = 1;
        QB_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        QB_CUDA(cudaStreamSynchronize(c.stream));
        return QBGPU_OK;
    };
    if (cplx && A->val_real && real_mode_on) {
        qbgpu_matrix R = *A;                                // same arrays, fp64 vectors
        R.api_complex = false;
        QB_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), c.stream));
        if (to_native_tiled_ok(A, 8)) QB_TRY((launch_to_native_tiled<double2, double, true>(A, xd, px, flag)));
        else {
            to_native_real_check_kernel<<<grid_rows(A->n), kPBlock, 0, c.stream>>>(A->n, A->perm_inv, (const double2 *)xd, (double *)px, flag);
            QB_LAUNCH_COUNT();
            QB_CUDA(cudaGetLastError());
        }
        // The closing pass can write the reference's order itself (sjds_bulk.cu, OUT) when y is not read: the separate way
        // out -- 0.9 ms of 17 on BASELINE config 3 -- is gone for 2 GB more traffic in pass 2.
        const bool fuse_out = !use_beta && !S->matfree && A->second && A->row_lo == 0 && A->row_hi == A->n && sjds_bulk_out_fusable(A->second);
        auto real_route = [&]() -> int {
            FusedArgs fa;
            fa.x = px; fa.y = py;
            if (fuse_out) { fa.y_ref = yd; fa.out_alpha = alpha; }
            QB_TRY(launch_spmv(&R, fa));
            if (!fuse_out) QB_TRY(vec_from_native(A, false, true, py, yd, alpha, beta));
            return QBGPU_OK;
        };
        int h;
        if (!use_beta && !A->last_x_had_imag) {
            // y is not read: run the fp64 passes at once and look at the flag afterwards (the read-back then costs no idle
            // time on the device); a vector with imaginary parts simply repeats the product on the complex route -- and
            // the handle remembers it: the next call looks at the flag first (a caller with complex vectors pays the wasted
            // passes once, not per product)
            QB_TRY(real_route());
            QB_TRY(read_flag(h));
            A->last_x_had_imag = h != 0;
            if (h != 0) QB_TRY(complex_route());
        } else {
            QB_TRY(read_flag(h));
            A->last_x_had_imag = h != 0;
            if (h == 0) QB_TRY(real_route()); else QB_TRY(complex_route());
        }
    } else {
        QB_TRY(complex_route());
    }
    if (where == QBGPU_HOST) {
        QB_CUDA(cudaMemcpyAsync(y, yd, bytes, cudaMemcpyDeviceToHost, c.stream));
        QB_CUDA(cudaStreamSynchronize(c.stream));
    }
    return QBGPU_OK;
}

}  // namespace qb

using namespace qb;

extern "C" {

/* The two parts of a STORED species-order handle or shard as handles of their own (views: they share the arrays, destroy
 * frees nothing): `local` = diagonal + hops of the down electrons -- its gathers stay inside the handle's own rows, so on a
 * row shard it needs NO remote data; `cross` = hops of the up electrons, traversed by tiles, gathers from every rank's rows.
 * A sharded product is then: start the exchange; local part (y = ...); wait for the slices; cross part (y += ...). */
int qbgpu_species_parts(qbgpu_matrix_t A, qbgpu_matrix_t *local, qbgpu_matrix_t *cross)
{
    QB_TRY(ensure_init());
    if (!A || !local || !cross) return fail(QBGPU_ERR_ARG, "null argument");
    const Species *S = (const Species *)A->sp;
    if (!S || S->matfree || !A->second) return fail(QBGPU_ERR_STATE, "species_parts: needs a stored species-order handle");
    auto *Lv = new qbgpu_matrix(*A);
    Lv->borrowed = true; Lv->sp = nullptr; Lv->second = nullptr; Lv->perm = nullptr; Lv->perm_inv = nullptr; Lv->perm_x = Lv->perm_y = nullptr;
    auto *Cv = new qbgpu_matrix(*A->second);
    Cv->borrowed = true; Cv->api_complex = A->api_complex; Cv->perm_x = Cv->perm_y = nullptr;
    *local = Lv; *cross = Cv;
    return QBGPU_OK;
}

/* The CROSS part of a stored species-order handle or shard cut by column ranges: parts[p] holds the entries with columns in
 * [bounds[p], bounds[p+1]) (bounds[0] = 0, bounds[nparts] = n; owning handles with the same rows, the same tile-ordered
 * traversal and the sliced-jagged layout).  On a row shard the part whose columns are the shard's own rows needs no remote
 * data: about 60 % of the cross entries of BASELINE config 3 on eight ranks (qbgpu_dist_set_parts). */
int qbgpu_species_split_cross(qbgpu_matrix_t A, int nparts, const int64_t *bounds, qbgpu_matrix_t *parts)
{
    QB_TRY(ensure_init());
    if (!A || !bounds || !parts || nparts < 1) return fail(QBGPU_ERR_ARG, "species_split_cross: bad argument");
    const Species *S = (const Species *)A->sp;
    if (!S || S->matfree || !A->second || A->borrowed) return fail(QBGPU_ERR_STATE, "species_split_cross: needs the owning stored species-order handle");
    qbgpu_matrix *Cx = A->second;
    if (Cx->cbits) return fail(QBGPU_ERR_STATE, "species_split_cross: the cross part stores packed entry words (a handle built without a row range); build it as a row shard to split it");
    if (Cx->ndict) return fail(QBGPU_ERR_STATE, "species_split_cross: not available with dictionary-coded values");
    QB_TRY(split_columns(Cx, nparts, bounds, parts, QBGPU_FORMAT_SELL | QBGPU_NO_AUTOTUNE));
    const int64_t ns = (Cx->nrows() + 31) / 32;
    for (int p = 0; p < nparts; p++) {
        parts[p]->api_complex = A->api_complex;
        if (ns > 0) {
            cudaError_t e = cudaMalloc(&parts[p]->slice_order, sizeof(int32_t) * (size_t)ns);
            if (e == cudaSuccess) e = cudaMemcpyAsync(parts[p]->slice_order, Cx->slice_order, sizeof(int32_t) * (size_t)ns, cudaMemcpyDeviceToDevice, ctx().stream);
            if (e != cudaSuccess) { for (int q = 0; q < nparts; q++) { qbgpu_destroy(parts[q]); parts[q] = nullptr; } return cuda_fail(e, "copy of the slice order", __FILE__, __LINE__); }
        }
    }
    QB_CUDA(cudaStreamSynchronize(ctx().stream));
    return QBGPU_OK;
}

/* A view of a sliced-jagged handle restricted to its local rows [r0, r1) (both multiples of 32; for a tile-ordered cross part
 * also multiples of tile_period = D_dn, so that the view's first row is the first down configuration again): same arrays, its
 * own traversal order.  Products through the view read and write y / z at the VIEW's rows (the caller offsets the pointers by
 * r0 entries, or uses the multi-GPU drivers, which do).  A late part cut by rows lets the first half start as soon as ITS
 * slices have arrived (qbgpu_dist_set_pull_plan: wait points). */
int qbgpu_row_view(qbgpu_matrix_t A, int64_t r0, int64_t r1, int64_t tile_period, int tile, qbgpu_matrix_t *view)
{
    QB_TRY(ensure_init());
    if (!A || !view) return fail(QBGPU_ERR_ARG, "null argument");
    *view = nullptr;
    if (A->sp || A->mf || A->mf_sec || A->format != QBGPU_FORMAT_SELL) return fail(QBGPU_ERR_STATE, "row_view: needs a stored sliced-jagged handle (a part of a species handle, a shard)");
    if (A->cbits) return fail(QBGPU_ERR_STATE, "row_view: the part stores packed entry words (a species handle built without a row range); only the parts of row shards can be cut");
    const int64_t nl = A->nrows();
    if (r0 < 0 || r1 < r0 || r1 > nl || r0 % 32 != 0 || (r1 % 32 != 0 && r1 != nl)) return fail(QBGPU_ERR_ARG, "row_view: the row range must consist of whole 32-row slices");
    if (A->slice_order && (tile_period <= 0 || r0 % tile_period != 0)) return fail(QBGPU_ERR_ARG, "row_view: a tile-ordered part must be cut at multiples of its tile period (D_dn)");
    auto *V = new qbgpu_matrix(*A);
    V->borrowed = true; V->owns_order = false;
    V->perm_x = V->perm_y = nullptr;
    V->row_lo = A->row_lo + r0; V->row_hi = A->row_lo + r1;
    V->rowptr = A->rowptr + r0;
    V->rowinfo = A->rowinfo + r0;
    V->nnz = 0; V->nnz_input = 0;
    if (A->slice_order) {
        std::vector<int32_t> order;
        make_slice_order(r1 - r0, tile_period, tile < 32 ? 64 : tile, order);
        V->slice_order = nullptr;
        cudaError_t e = upload(&V->slice_order, order.data(), order.size(), ctx().stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx().stream);
        if (e != cudaSuccess) { cudaFree(V->slice_order); delete V; return cuda_fail(e, "row_view: slice order", __FILE__, __LINE__); }
        V->owns_order = true;
    }
    *view = V;
    return QBGPU_OK;
}

/* For a row range [row_lo, row_hi) of the species order of the Hubbard sector (nsites, N_up, N_dn): ref_rows_dev[p - row_lo] =
 * the row of the reference's Lin order that has internal index p.  What a rank of a sharded run needs to fill its slice of a
 * vector that is defined in the reference's order (qbgpu_dist_randomize: the start vector vec_randomize(seed)). */
int qbgpu_species_ref_rows(int nsites, int nup, int ndn, int64_t row_lo, int64_t row_hi, int32_t *ref_rows_dev)
{
    QB_TRY(ensure_init());
    if (nsites < 2 || nup < 0 || ndn < 0 || nup > nsites || ndn > nsites || !ref_rows_dev) return fail(QBGPU_ERR_ARG, "species_ref_rows: bad argument");
    HostTables T;
    QB_TRY(make_tables(nsites, 2, nup, ndn, T));
    static thread_local ModelParams M;
    M.kind = 1; M.J = 0; M.t = 0; M.U = 0; M.nbonds = 0;
    SpeciesHost H;
    QB_TRY(build_host_tables(nsites, nup, ndn, M, H));
    const int64_t Dd = (int64_t)H.list[1].size();
    if (row_lo < 0 || row_hi < row_lo || row_hi > T.dim) return fail(QBGPU_ERR_ARG, "species_ref_rows: bad row range");
    int32_t *d_rank = nullptr;
    QB_CUDA(cudaMalloc(&d_rank, sizeof(int32_t) * H.rank.size()));
    cudaError_t e = cudaMemcpyAsync(d_rank, H.rank.data(), sizeof(int32_t) * H.rank.size(), cudaMemcpyHostToDevice, ctx().stream);
    int rc = e == cudaSuccess ? species_ref_rows_build(T, d_rank, Dd, row_lo, row_hi, ref_rows_dev) : cuda_fail(e, "upload rank table", __FILE__, __LINE__);
    cudaFree(d_rank);
    return rc;
}

int qbgpu_native_order(qbgpu_matrix_t A, int *has_internal_order)
{
    if (!A || !has_internal_order) return fail(QBGPU_ERR_ARG, "null argument");
    *has_internal_order = A->perm ? 1 : 0;
    return QBGPU_OK;
}

int qbgpu_vec_to_native(qbgpu_matrix_t A, const void *x_ref_dev, void *x_native_dev)
{
    QB_TRY(ensure_init());
    if (!A || !x_ref_dev || !x_native_dev) return fail(QBGPU_ERR_ARG, "null argument");
    if (x_ref_dev == x_native_dev) return fail(QBGPU_ERR_ARG, "vec_to_native works out of place");
    return vec_to_native(A, A->api_complex, A->api_complex, x_ref_dev, x_native_dev);
}

int qbgpu_vec_from_native(qbgpu_matrix_t A, const void *x_native_dev, void *x_ref_dev)
{
    QB_TRY(ensure_init());
    if (!A || !x_ref_dev || !x_native_dev) return fail(QBGPU_ERR_ARG, "null argument");
    if (x_ref_dev == x_native_dev) return fail(QBGPU_ERR_ARG, "vec_from_native works out of place");
    return vec_from_native(A, A->api_complex, A->api_complex, x_native_dev, x_ref_dev, make_double2(1.0, 0.0), make_double2(0.0, 0.0));
}

/* CPU-side execution of the species-order index logic: the SAME __host__ __device__ row functions the kernels call, on host
 * arrays, with no device involved (tests/test_species_cpu.py compares the results with the reference-pinned numpy
 * restatement).  sizes[4] = {Du, Dd, up-hop entries, down-hop entries}; every other pointer may be NULL (skipped):
 *   perm[n]; the two stored parts as CSR (rowptr[n+1], col, val: nnz_local = Du*(tot_d+Dd), nnz_cross = Dd*tot_u);
 *   slice_order[ceil(n/32)]; y[n] = H x through the two matrix-free passes with x, y in the internal order; the warp items
 *   of the cross pass visited in the kernel's order, touched[p] counting how often row p was written (must end as all 1). */
int qbgpu_debug_species_host(int nsites, int nup, int ndn, int nbonds, const int32_t *bonds, double t, double U, int tile,
                             int64_t *sizes, int32_t *perm, int64_t *rp_local, int32_t *col_local, double *val_local,
                             int64_t *rp_cross, int32_t *col_cross, double *val_cross, int32_t *slice_order,
                             const double *x, double *y, int32_t *touched)
{
    if (nsites < 2 || nup < 0 || ndn < 0 || nup > nsites || ndn > nsites || nbonds < 1 || !bonds || !sizes) return fail(QBGPU_ERR_ARG, "debug_species_host: bad argument");
    HostTables T;
    QB_TRY(make_tables(nsites, 2, nup, ndn, T));
    static thread_local ModelParams M;
    M.kind = 1; M.J = 0; M.t = t; M.U = U;
    QB_TRY(merge_bonds(nsites, nbonds, bonds, M));
    SpeciesHost H;
    QB_TRY(build_host_tables(nsites, nup, ndn, M, H));
    SpeciesView V;
    V.Du = (int64_t)H.list[0].size(); V.Dd = (int64_t)H.list[1].size(); V.tot_u = (int64_t)H.hop[0].size(); V.tot_d = (int64_t)H.hop[1].size();
    V.ulist = H.list[0].data(); V.dlist = H.list[1].data(); V.uptr = H.ptr[0].data(); V.dptr = H.ptr[1].data();
    V.uhop = H.hop[0].data(); V.dhop = H.hop[1].data();
    sizes[0] = V.Du; sizes[1] = V.Dd; sizes[2] = V.tot_u; sizes[3] = V.tot_d;
    const int64_t n = V.Du * V.Dd;
    if (n != T.dim) return fail(QBGPU_ERR_STATE, "debug_species_host: dimension mismatch with the Lin tables");
    int W = tile < 32 ? 32 : (tile + 31) / 32 * 32;
    if (perm) species_perm_host(T, H.rank.data(), V.Dd, perm);
    if (rp_local && rp_cross) for (int64_t p = 0; p <= n; p++) species_rowptr_at(V, n, p, rp_local[p], rp_cross[p]);
    if (col_local && val_local && col_cross && val_cross)
        for (int64_t p = 0; p < n; p++) species_fill_row<double>(V, H.ampw, H.diagk, p, col_local, val_local, col_cross, val_cross);
    if (slice_order) { std::vector<int32_t> o; make_slice_order(n, V.Dd, W, o); memcpy(slice_order, o.data(), sizeof(int32_t) * o.size()); }
    if (x && y) {
        for (int64_t p = 0; p < n; p++) {
            const int64_t iu = p / V.Dd;
            const int32_t idl = (int32_t)(p - iu * V.Dd);
            y[p] = H.uniform_w > 0 ? kron_local_acc<double, false, true>(V, H.ampw, H.diagk, V.ulist[iu], idl, x, (uint32_t)(iu * V.Dd), x[p], H.ampw[H.uniform_w])
                                   : kron_local_acc<double, false, false>(V, H.ampw, H.diagk, V.ulist[iu], idl, x, (uint32_t)(iu * V.Dd), x[p]);
        }
        const CrossItems I = cross_items(V.Du, V.Dd, W);
        for (int64_t it = 0; it < I.nitems; it++)
            for (int lane = 0; lane < 32; lane++) {
                int64_t iu, id;
                cross_item_at(I, it, lane, iu, id);
                if (iu < 0 || iu >= V.Du || id < 0) return fail(QBGPU_ERR_STATE, "debug_species_host: warp item out of range");
                const bool live = id < V.Dd;
                const double acc = H.uniform_w > 0 ? kron_cross_acc<double, false, true>(V, H.ampw, iu, live ? id : V.Dd - 1, x, 0, 0, H.ampw[H.uniform_w])
                                                   : kron_cross_acc<double, false, false>(V, H.ampw, iu, live ? id : V.Dd - 1, x);
                if (live) { y[iu * V.Dd + id] += acc; if (touched) touched[iu * V.Dd + id]++; }
            }
    }
    return QBGPU_OK;
}

/* The packed layout of the two stored parts (qbgpu_matrix::cbits), computed on the host with the build's rules: the entries of
 * species_fill_row in CSR order, each part's table of distinct values ordered by value_table_less, words packed_word(col,
 * code, cbits).  cbits <= 0: the build's own width, packed_col_bits(n).  out[0] = cbits; out[1], out[2] = table entries of the
 * local / cross part; out[3], out[4] = 1 when that part is packed (its table fits beside the columns), 0 when it keeps separate
 * fp64 values.  table_* (256 entries each) and words_* (nnz_local / nnz_cross of qbgpu_debug_species_host) may be NULL. */
int qbgpu_debug_species_packed_host(int nsites, int nup, int ndn, int nbonds, const int32_t *bonds, double t, double U, int cbits,
                                    int64_t *out, double *table_local, uint32_t *words_local, double *table_cross, uint32_t *words_cross)
{
    if (nsites < 2 || nup < 0 || ndn < 0 || nup > nsites || ndn > nsites || nbonds < 1 || !bonds || !out || cbits > 31)
        return fail(QBGPU_ERR_ARG, "debug_species_packed_host: bad argument");
    HostTables T;
    QB_TRY(make_tables(nsites, 2, nup, ndn, T));
    static thread_local ModelParams M;
    M.kind = 1; M.J = 0; M.t = t; M.U = U;
    QB_TRY(merge_bonds(nsites, nbonds, bonds, M));
    SpeciesHost H;
    QB_TRY(build_host_tables(nsites, nup, ndn, M, H));
    SpeciesView V;
    V.Du = (int64_t)H.list[0].size(); V.Dd = (int64_t)H.list[1].size(); V.tot_u = (int64_t)H.hop[0].size(); V.tot_d = (int64_t)H.hop[1].size();
    V.ulist = H.list[0].data(); V.dlist = H.list[1].data(); V.uptr = H.ptr[0].data(); V.dptr = H.ptr[1].data();
    V.uhop = H.hop[0].data(); V.dhop = H.hop[1].data();
    const int64_t n = V.Du * V.Dd;
    if (n != T.dim) return fail(QBGPU_ERR_STATE, "debug_species_packed_host: dimension mismatch with the Lin tables");
    if (cbits <= 0) cbits = packed_col_bits(n);
    std::vector<int32_t> col[2] = {std::vector<int32_t>((size_t)(V.Du * (V.tot_d + V.Dd))), std::vector<int32_t>((size_t)(V.Dd * V.tot_u))};
    std::vector<double> val[2] = {std::vector<double>(col[0].size()), std::vector<double>(col[1].size())};
    for (int64_t p = 0; p < n; p++) species_fill_row<double>(V, H.ampw, H.diagk, p, col[0].data(), val[0].data(), col[1].data(), val[1].data());
    out[0] = cbits;
    double *tables[2] = {table_local, table_cross};
    uint32_t *words[2] = {words_local, words_cross};
    for (int part = 0; part < 2; part++) {
        std::vector<double> tab;
        {   // distinct bit patterns, in the order of the build's table
            std::vector<uint64_t> bits(val[part].size());
            memcpy(bits.data(), val[part].data(), 8 * bits.size());
            std::sort(bits.begin(), bits.end());
            bits.erase(std::unique(bits.begin(), bits.end()), bits.end());
            for (uint64_t b : bits) { double v; memcpy(&v, &b, 8); tab.push_back(v); }
            std::sort(tab.begin(), tab.end(), value_table_less);
        }
        const bool packed = packed_table_fits((int64_t)tab.size(), cbits);
        out[1 + part] = (int64_t)tab.size();
        out[3 + part] = packed ? 1 : 0;
        if (tables[part]) for (size_t j = 0; j < kPackedMaxTable; j++) tables[part][j] = j < tab.size() ? tab[j] : 0.0;
        if (words[part] && packed)
            for (size_t i = 0; i < val[part].size(); i++) {
                const uint32_t code = (uint32_t)(std::lower_bound(tab.begin(), tab.end(), val[part][i], value_table_less) - tab.begin());
                words[part][i] = packed_word(col[part][i], code, cbits);
            }
    }
    return QBGPU_OK;
}

/* The same for a ROW SHARD cut into COLUMN PARTS (what the multi-GPU exchanges of dist.py multiply): rows = the up
 * configurations [u_lo, u_hi), parts p = the hops whose target lies in [part_bounds[p], part_bounds[p+1]) (units: up
 * configurations), executed in the given order; the part containing u_lo also runs the local pass; the first executed part
 * opens the product (y = ...), the others accumulate.  x: full vector, y_local: (u_hi - u_lo) * D_dn entries. */
int qbgpu_debug_species_parts_host(int nsites, int nup, int ndn, int nbonds, const int32_t *bonds, double t, double U, int tile,
                                   int64_t u_lo, int64_t u_hi, int nparts, const int64_t *part_bounds, const int32_t *order,
                                   const double *x, double *y_local)
{
    if (nsites < 2 || nup < 0 || ndn < 0 || nup > nsites || ndn > nsites || nbonds < 1 || !bonds || !part_bounds || !order || !x || !y_local || nparts < 1)
        return fail(QBGPU_ERR_ARG, "debug_species_parts_host: bad argument");
    HostTables T;
    QB_TRY(make_tables(nsites, 2, nup, ndn, T));
    static thread_local ModelParams M;
    M.kind = 1; M.J = 0; M.t = t; M.U = U;
    QB_TRY(merge_bonds(nsites, nbonds, bonds, M));
    SpeciesHost H;
    QB_TRY(build_host_tables(nsites, nup, ndn, M, H));
    SpeciesView V;
    V.Du = (int64_t)H.list[0].size(); V.Dd = (int64_t)H.list[1].size(); V.tot_u = (int64_t)H.hop[0].size(); V.tot_d = (int64_t)H.hop[1].size();
    V.ulist = H.list[0].data(); V.dlist = H.list[1].data(); V.uptr = H.ptr[0].data(); V.dptr = H.ptr[1].data();
    V.uhop = H.hop[0].data(); V.dhop = H.hop[1].data();
    if (u_lo < 0 || u_hi < u_lo || u_hi > V.Du) return fail(QBGPU_ERR_ARG, "debug_species_parts_host: bad row range");
    const int W = tile < 32 ? 32 : (tile + 31) / 32 * 32;
    const int64_t u_cnt = u_hi - u_lo;
    const CrossItems I = cross_items(u_cnt, V.Dd, W);
    bool local_done = false;
    for (int k = 0; k < nparts; k++) {
        const int p = order[k];
        if (p < 0 || p >= nparts) return fail(QBGPU_ERR_ARG, "debug_species_parts_host: bad order");
        const int64_t c_lo = part_bounds[p], c_hi = part_bounds[p + 1];
        const bool has_local = !local_done && c_lo <= u_lo && u_lo < c_hi;
        bool first = (k == 0);
        if (has_local) {
            for (int64_t q = 0; q < u_cnt * V.Dd; q++) {
                const int64_t pg = u_lo * V.Dd + q, iu = pg / V.Dd;
                const double acc = kron_local_acc<double, false>(V, H.ampw, H.diagk, V.ulist[iu], (int32_t)(pg - iu * V.Dd), x, (uint32_t)(iu * V.Dd), x[pg]);
                y_local[q] = first ? acc : y_local[q] + acc;
            }
            local_done = true;
            first = false;                                  // the cross pass of this part continues the product
        }
        for (int64_t it = 0; it < I.nitems; it++)
            for (int lane = 0; lane < 32; lane++) {
                int64_t il, id;
                cross_item_at(I, it, lane, il, id);
                if (il < 0 || il >= u_cnt || id < 0) return fail(QBGPU_ERR_STATE, "debug_species_parts_host: warp item out of range");
                const bool live = id < V.Dd;
                const double acc = kron_cross_acc<double, true>(V, H.ampw, u_lo + il, live ? id : V.Dd - 1, x, c_lo, c_hi);
                if (live) { const int64_t q = il * V.Dd + id; y_local[q] = first ? acc : y_local[q] + acc; }
            }
    }
    return QBGPU_OK;
}

int qbgpu_native_perm(qbgpu_matrix_t A, int32_t *perm_host)
{
    QB_TRY(ensure_init());
    if (!A || !perm_host) return fail(QBGPU_ERR_ARG, "null argument");
    if (!A->perm) return fail(QBGPU_ERR_STATE, "the handle has no internal order");
    QB_CUDA(cudaStreamSynchronize(ctx().stream));
    QB_CUDA(cudaMemcpy(perm_host, A->perm, sizeof(int32_t) * (size_t)A->n, cudaMemcpyDeviceToHost));
    return QBGPU_OK;
}

}  // extern "C"
