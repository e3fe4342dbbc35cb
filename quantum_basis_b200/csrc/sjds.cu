// quantum_basis_b200/csrc/sjds.cu -- the "sliced jagged" H*v kernel and its in-place format conversion.
//
// Why a second layout: in the reference's Lin-table order (src/basis.cc:1144-1190) consecutive rows are basis states
// that differ only in the even-site label, so a given Hamiltonian term sends consecutive rows to (nearly) consecutive
// columns.  The CSR-vector kernel assigns LANES threads to ONE row, so the 32 gathers of a warp instruction hit 32
// unrelated cache lines; assigning one thread per row makes the gathers of a warp fall into a few contiguous
// segments of x (coalesced 128-byte lines instead of 32 separate sectors), which is what bounds the kernel once the
// matrix stream itself is coalesced.  Thread-per-row over plain CSR would un-coalesce the matrix stream, and ELL/SELL
// padding would add bytes, so the entries of every 32-row slice are re-ordered jagged-diagonal-wise:
//     rank the slice's rows by length (descending);  for k = 0,1,2,...: the k-th entry of every row with length > k,
//     in rank order.
// The rows active at step k are always ranks [0, cnt_k), so lane `rank` reads entry off_k + rank: contiguous,
// unpadded, and off_{k+1} = off_k + popc(ballot(k < len)).  A slice occupies exactly the CSR range of its 32 rows,
// so the conversion is an in-place (chunk-buffered) permutation and the algorithmic bytes do not change
// (4 bytes of rowinfo per row replace nothing: rowptr is still read once per slice).
#include "internal.hpp"
#include <algorithm>
#include <type_traits>
#include <vector>

namespace qb {

constexpr int kSBlock = 256;
constexpr uint32_t kLenMask = 0xFFFFFFu;

// ---- cache-policy helpers (PTX): the matrix stream should leave L2 first, the gathered vector last ------------
__device__ __forceinline__ uint64_t l2_policy_evict_first() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ uint64_t l2_policy_evict_last()  { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p; }

// All loads of the inner loop are volatile asm so that they are issued in program order -- first the U column and
// value loads of a trip, then the U gathers -- instead of ptxas' register-frugal "load, gather, fma" chain per
// diagonal, which leaves a warp with a single dependent pair of loads in flight.  The matrix stream is read through the
// non-coherent path with an L2 evict_first policy operand.
__device__ __forceinline__ int ld_i32(const int *p, uint64_t pol)
{ int v; asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol)); return v; }
__device__ __forceinline__ double ld_f64(const double *p, uint64_t pol)
{ double v; asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol)); return v; }
__device__ __forceinline__ uint8_t ld_f64(const uint8_t *p, uint64_t pol)      // dictionary codes
{ unsigned v; asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol)); return (uint8_t)v; }
__device__ __forceinline__ double2 ld_f64(const double2 *p, uint64_t pol)
{ double2 v; asm volatile("ld.global.nc.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol)); return v; }
// gathered vector: XPOL 0 = read-only path, default policy; 1 = read-only path + L2 evict_last
template <int XPOL> __device__ __forceinline__ double ld_x(const double *p, uint64_t pol)
{
    double v;
    if (XPOL == 0) asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));  // XPOL 1: policy operand
    else asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
    return v;
}
template <int XPOL> __device__ __forceinline__ double2 ld_x(const double2 *p, uint64_t pol)
{
    double2 v;
    if (XPOL == 0) asm volatile("ld.global.nc.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    else asm volatile("ld.global.nc.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol));
    return v;
}

// U = jagged diagonals per trip (U independent col/val loads, then U gathers); XPOL = cache policy of the gathers above;
// UL = unconditional loads: lanes whose row has ended re-read the slice's first entry (always valid, L1-resident)
// instead of branching around the loads, so that all 3U loads of a trip can be in flight together;
// MINB = __launch_bounds__ min blocks/SM: without it ptxas schedules for 32 registers (full occupancy) and chains
// "load column, load value, gather, fma" one diagonal at a time -- a single dependent pair of loads in flight per
// warp; with MINB <= 4 it batches the U column loads, the U value loads and the U gathers (checked in the SASS).
template <typename ValT, typename VecT, bool DOTS, int U, int XPOL, bool UL, int MINB, bool KEEP = false>
__global__ void __launch_bounds__(kSBlock, MINB)
spmv_sjds_kernel(int64_t nslices, int64_t nrows, int64_t row_lo, const int64_t *__restrict__ rowptr,
                 const uint32_t *__restrict__ rowinfo, const int32_t *__restrict__ col, const ValT *__restrict__ val,
                 const VecT *__restrict__ x, const VecT *z, VecT *y, double2 alpha, double2 gamma, double2 beta,
                 int scal_mode, const double *__restrict__ sc, double *dots_out, double *partials, unsigned *ticket,
                 const double *__restrict__ vdict, int cbits)
{
    using VT = VecTraits<VecT>;
    constexpr bool kDict = sizeof(ValT) == 1;               // 1-byte codes into a <= 256-entry fp64 dictionary
    constexpr bool kPacked = std::is_same<ValT, uint32_t>::value;   // packed words col | code << cbits (no val array)
    using ArithT = typename std::conditional<kDict || kPacked, double, ValT>::type;
    __shared__ double sdict[kDict || kPacked ? 256 : 1];
    if (kDict || kPacked) { sdict[threadIdx.x] = vdict[threadIdx.x]; __syncthreads(); }      // kSBlock == 256 threads
    const uint32_t cmask = kPacked ? (1u << cbits) - 1u : ~0u;
    constexpr int WPB = kSBlock / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t pol_s = l2_policy_evict_first(), pol_x = XPOL >= 1 ? l2_policy_evict_last() : 0;
    double dot_scale = 1.0;
    if (scal_mode != 0) {                                  // Lanczos step a: 1 = first column block, 2 = a later one
        const double sx = sc[0], sz = sc[1], bprev = sc[2];
        alpha = make_double2(sx, 0.0);
        gamma = make_double2(0.0, 0.0);
        beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
        dot_scale = sx;
    }
    const bool use_gamma = (gamma.x != 0.0 || gamma.y != 0.0);
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    // KEEP: y += H_block x (a later column block of a sharded product, chosen by the launcher when beta == 1, z == y and
    // there is no epilogue): rows without entries in this block keep their y -- neither read nor written.  A template
    // parameter, not a run-time test: the plain instantiation must stay instruction-for-instruction what ptxas schedules
    // well (a run-time flag here cost 15-25 % on the unsplit product).
    double d[3] = {0.0, 0.0, 0.0};

    for (int64_t s = (int64_t)blockIdx.x * WPB + warp; s < nslices; s += (int64_t)gridDim.x * WPB) {
        const uint32_t info = rowinfo[s * 32 + lane];
        const int len = (int)(info & kLenMask);
        const int64_t row = s * 32 + (info >> 24);
        const int maxlen = __shfl_sync(0xffffffffu, len, 0);
        if constexpr (KEEP) { if (maxlen == 0) continue; }   // warp-uniform: the whole slice is empty
        const int64_t base = rowptr[s * 32];
        int64_t off = base + lane;                          // this lane's entry at step k is off_k + lane
        VecT acc0 = VT::zero(), acc1 = VT::zero();
        for (int k = 0; k < maxlen; k += U) {              // U jagged diagonals per trip; the tail is predicated off
            bool a[U];
            int64_t o[U];
            int c[U];
            ValT v[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                a[u] = k + u < len;
                o[u] = (UL && !a[u]) ? base : off;
                off += __popc(__ballot_sync(0xffffffffu, a[u]));
            }
            if (UL) {
                VecT xv[U];
#pragma unroll
                for (int u = 0; u < U; u++) c[u] = ld_i32(col + o[u], pol_s);
                if constexpr (!kPacked) {
#pragma unroll
                    for (int u = 0; u < U; u++) v[u] = ld_f64(val + o[u], pol_s);
                }
#pragma unroll
                for (int u = 0; u < U; u++) xv[u] = ld_x<XPOL>(x + ((uint32_t)c[u] & cmask), pol_x);
#pragma unroll
                for (int u = 0; u < U; u++) {
                    VecT t = (u & 1) ? acc1 : acc0;
                    ArithT w;
                    if constexpr (kPacked) w = sdict[(uint32_t)c[u] >> cbits]; else if constexpr (kDict) w = sdict[v[u]]; else w = v[u];
                    mac(t, w, xv[u]);
                    if (a[u]) { if (u & 1) acc1 = t; else acc0 = t; }
                }
            } else {
#pragma unroll
                for (int u = 0; u < U; u++) {
                    c[u] = 0; v[u] = ValT{};
                    if (a[u]) { c[u] = ld_i32(col + o[u], pol_s); if constexpr (!kPacked) v[u] = ld_f64(val + o[u], pol_s); }
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    if (a[u]) {
                        ArithT w;
                        if constexpr (kPacked) w = sdict[(uint32_t)c[u] >> cbits]; else if constexpr (kDict) w = sdict[v[u]]; else w = v[u];
                        const VecT xv = ld_x<XPOL>(x + ((uint32_t)c[u] & cmask), pol_x);
                        if (u & 1) mac(acc1, w, xv); else mac(acc0, w, xv);
                    }
                }
            }
        }
        if (row < nrows && !(KEEP && len == 0)) {           // padding ranks of the last slice point past the last row
            const VecT acc = VT::add(acc0, acc1);
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
        block_reduce_finalize<3, kSBlock>(d, partials, ticket, dots_out);
    }
}

template <typename ValT, typename VecT, bool DOTS, int U, int XPOL, bool UL, int MINB, bool KEEP = false>
static int launch_sjds_cfg(const qbgpu_matrix *A, const FusedArgs &a)
{
    Context &c = ctx();
    auto kern = spmv_sjds_kernel<ValT, VecT, DOTS, U, XPOL, UL, MINB, KEEP>;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, kSBlock, 0));
        if (blocks_per_sm < 1) blocks_per_sm = 1;
    }
    const int64_t nrows = A->nrows();
    if (nrows == 0) return QBGPU_OK;
    const int64_t nslices = (nrows + 31) / 32;
    constexpr int WPB = kSBlock / 32;
    int64_t want = (nslices + WPB - 1) / WPB;
    int64_t cap = (int64_t)c.num_sms * blocks_per_sm;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    const int grid = (int)(want < cap ? want : cap);
    kern<<<grid, kSBlock, 0, c.stream>>>(nslices, nrows, A->row_lo, A->rowptr, A->rowinfo, A->col, (const ValT *)A->val,
                                         (const VecT *)a.x, (const VecT *)a.z, (VecT *)a.y, a.alpha, a.gamma, a.beta,
                                         a.scal_mode, a.sc, a.dots, c.partials, c.ticket, A->vdict, A->cbits);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

template <typename ValT, typename VecT>
static int launch_sjds_typed(const qbgpu_matrix *A, const FusedArgs &a)
{
    // configuration of the template, chosen from the measurements in profiles/r01_kbench_*.txt: complex vectors take 4
    // diagonals per trip, a branchy tail, L2 evict_last on the gathers and 4 blocks/SM; fp64 vectors take 8 per trip with
    // unconditional loads (with the epilogue of the dots that needs a few more registers: 3 blocks/SM keeps its loads batched)
    constexpr bool kCplx = sizeof(VecT) == 16;
    constexpr int U = kCplx ? 4 : 8, X = kCplx ? 1 : 0, MinB = 4, DotsMinB = kCplx ? 4 : 3;
    constexpr bool UL = !kCplx;
    const bool dots = a.dots != nullptr;
    // accumulating column block of a sharded product (y += H_p x, immediates only): skip the rows this block does not touch
    if (!dots && a.scal_mode == 0 && a.z == a.y && a.beta.x == 1.0 && a.beta.y == 0.0 && a.gamma.x == 0.0 && a.gamma.y == 0.0)
        return launch_sjds_cfg<ValT, VecT, false, U, X, UL, MinB, true>(A, a);
    return dots ? launch_sjds_cfg<ValT, VecT, true, U, X, UL, DotsMinB>(A, a)
                : launch_sjds_cfg<ValT, VecT, false, U, X, UL, MinB>(A, a);
}


// ------------------------------------------------------------------------------------------ ring-fused product
// One kernel for "exchange, then multiply" on a row shard (SURVEY 8e): the vector slices of the other ranks are pulled
// over NVLink by copy engines while this kernel runs; each pull ends by setting flags[d] (d = ring distance of the
// owner).  The rows of the shard were rotated into ring order by ring_prepare, so a row meets its own rank's columns
// first and the others in the order of their arrival; before gathering x[c] a lane makes sure the slice c belongs to
// has landed.  No column blocks, no partial y, no extra passes over rowptr/rowinfo: the unsplit shard is read once.
__device__ __forceinline__ int ld_acquire_sys(const int *p) { int v; asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }

template <typename ValT, typename VecT, bool DOTS, int U>
__global__ void __launch_bounds__(kSBlock, 4)
spmv_sjds_ring_kernel(int64_t nslices, int64_t nrows, int64_t row_lo, const int64_t *__restrict__ rowptr,
                      const uint32_t *__restrict__ rowinfo, const int32_t *__restrict__ col, const ValT *__restrict__ val,
                      const VecT *x, const VecT *z, VecT *y, double2 alpha, double2 gamma, double2 beta,
                      int scal_mode, const double *__restrict__ sc, double *dots_out, double *partials, unsigned *ticket,
                      const double *__restrict__ vdict, const int *flags, int *timed_out, unsigned chunk, int rank, int world)
{
    using VT = VecTraits<VecT>;
    constexpr bool kDict = sizeof(ValT) == 1;
    using ArithT = typename std::conditional<kDict, double, ValT>::type;
    __shared__ double sdict[kDict ? 256 : 1];
    if (kDict) { sdict[threadIdx.x] = vdict[threadIdx.x]; __syncthreads(); }
    constexpr int WPB = kSBlock / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t pol_s = l2_policy_evict_first(), pol_x = l2_policy_evict_last();
    double dot_scale = 1.0;
    if (scal_mode != 0) {
        const double sx = sc[0], sz = sc[1], bprev = sc[2];
        alpha = make_double2(sx, 0.0);
        gamma = make_double2(0.0, 0.0);
        beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
        dot_scale = sx;
    }
    const bool use_gamma = (gamma.x != 0.0 || gamma.y != 0.0);
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    double d[3] = {0.0, 0.0, 0.0};
    int have = 0;                                           // flags[0 .. have] have been seen set by this lane (0 = own slice)

    for (int64_t s = (int64_t)blockIdx.x * WPB + warp; s < nslices; s += (int64_t)gridDim.x * WPB) {
        const uint32_t info = rowinfo[s * 32 + lane];
        const int len = (int)(info & kLenMask);
        const int64_t row = s * 32 + (info >> 24);
        const int maxlen = __shfl_sync(0xffffffffu, len, 0);
        const int64_t base = rowptr[s * 32];
        int64_t off = base + lane;
        VecT acc0 = VT::zero(), acc1 = VT::zero();
        for (int k = 0; k < maxlen; k += U) {
            bool a[U];
            int64_t o[U];
            int c[U];
            ValT v[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                a[u] = k + u < len;
                o[u] = off;
                off += __popc(__ballot_sync(0xffffffffu, a[u]));
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                c[u] = 0; v[u] = ValT{};
                if (a[u]) { c[u] = ld_i32(col + o[u], pol_s); v[u] = ld_f64(val + o[u], pol_s); }
            }
            // the furthest slice this trip needs (ring order inside a row: the distance never decreases)
            int need = 0;
#pragma unroll
            for (int u = 0; u < U; u++) {
                if (a[u]) {
                    int owner = (int)((unsigned)c[u] / chunk);
                    owner = owner < world ? owner : world - 1;
                    int dist = owner - rank; dist += dist < 0 ? world : 0;
                    need = dist > need ? dist : need;
                }
            }
            if (need > have) {
                for (int f = have + 1; f <= need; f++) {
                    const long long t0 = clock64();
                    while (ld_acquire_sys(flags + f) == 0) {
                        if (clock64() - t0 > (1LL << 31)) { atomicExch(timed_out, 1); break; }     // ~1 s: never hang the GPU
                        __nanosleep(200);
                    }
                }
                have = need;
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                if (a[u]) {
                    ArithT w;
                    if constexpr (kDict) w = sdict[v[u]]; else w = v[u];
                    if (u & 1) mac(acc1, w, ld_x<1>(x + c[u], pol_x)); else mac(acc0, w, ld_x<1>(x + c[u], pol_x));
                }
            }
        }
        if (row < nrows) {
            const VecT acc = VT::add(acc0, acc1);
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
        block_reduce_finalize<3, kSBlock>(d, partials, ticket, dots_out);
    }
}

template <typename ValT, typename VecT, bool DOTS>
static int launch_sjds_ring(const qbgpu_matrix *A, const FusedArgs &a)
{
    Context &c = ctx();
    constexpr int U = sizeof(VecT) == 16 ? 4 : 8;
    auto kern = spmv_sjds_ring_kernel<ValT, VecT, DOTS, U>;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, kSBlock, 0));
        if (blocks_per_sm < 1) blocks_per_sm = 1;
    }
    const int64_t nrows = A->nrows();
    if (nrows == 0) return QBGPU_OK;
    const int *flags = nullptr; int *timed_out = nullptr;
    QB_TRY(peer_ring_flags(&flags, &timed_out));
    const int64_t nslices = (nrows + 31) / 32;
    constexpr int WPB = kSBlock / 32;
    int64_t want = (nslices + WPB - 1) / WPB;
    int64_t cap = (int64_t)c.num_sms * blocks_per_sm;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    const int grid = (int)(want < cap ? want : cap);
    kern<<<grid, kSBlock, 0, c.stream>>>(nslices, nrows, A->row_lo, A->rowptr, A->rowinfo, A->col, (const ValT *)A->val,
                                         (const VecT *)a.x, (const VecT *)a.z, (VecT *)a.y, a.alpha, a.gamma, a.beta,
                                         a.scal_mode, a.sc, a.dots, c.partials, c.ticket, A->vdict, flags, timed_out,
                                         (unsigned)A->ring_chunk, A->ring_rank, A->ring_world);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

template <typename ValT, typename VecT>
static int launch_sjds_ring_typed(const qbgpu_matrix *A, const FusedArgs &a)
{
    return a.dots ? launch_sjds_ring<ValT, VecT, true>(A, a) : launch_sjds_ring<ValT, VecT, false>(A, a);
}

int launch_spmv_sjds(const qbgpu_matrix *A, const FusedArgs &a)
{
    if (A->block_D > 0 && !a.dots && A->ring_world <= 1 && block_smem_applicable(A, A->block_D)) return launch_spmv_block_smem(A, a, A->block_D);
    // tile-ordered cross parts: the matrix stream through cp.async.bulk + mbarrier rings (sjds_bulk.cu).  Measured on BASELINE
    // config 3 (profiles/r02_bulk_sweep_*.txt): on the one-pass product in the reference's order the bulk-streamed kernel equals
    // the register-fed one at best (the gathers need the L1 the rings take); on the tile-ordered cross part -- gathers in whole
    // 512-byte segments that hit L2 -- it runs at 88 % of the copy peak.
    if (A->ring_world <= 1 && A->slice_order) return launch_spmv_sjds_bulk(A, a);
    if (a.y_ref) return fail(QBGPU_ERR_STATE, "fused way out: only the bulk-streamed kernel writes the reference's order (internal)");
    if (A->ring_world > 1) {
        if (A->cbits) return fail(QBGPU_ERR_STATE, "ring-fused product: not available for packed entry words");
        if (A->ndict) return A->api_complex ? launch_sjds_ring_typed<uint8_t, double2>(A, a) : launch_sjds_ring_typed<uint8_t, double>(A, a);
        if (!A->api_complex) return launch_sjds_ring_typed<double, double>(A, a);
        if (A->val_real) return launch_sjds_ring_typed<double, double2>(A, a);
        return launch_sjds_ring_typed<double2, double2>(A, a);
    }
    if (A->cbits) return A->api_complex ? launch_sjds_typed<uint32_t, double2>(A, a) : launch_sjds_typed<uint32_t, double>(A, a);
    if (A->ndict) return A->api_complex ? launch_sjds_typed<uint8_t, double2>(A, a) : launch_sjds_typed<uint8_t, double>(A, a);
    if (!A->api_complex) return launch_sjds_typed<double, double>(A, a);
    if (A->val_real) return launch_sjds_typed<double, double2>(A, a);
    return launch_sjds_typed<double2, double2>(A, a);
}

// ------------------------------------------------------------------------------------------ format conversion
// One warp per slice.  forward: CSR order -> jagged order (and fills rowinfo); backward: the inverse.
// `tmp` receives the re-ordered entries of slices [s0, s1) at offset (position - base0).
template <typename ValT, bool FORWARD>
__global__ void __launch_bounds__(kSBlock)
sjds_permute_kernel(int64_t s0, int64_t s1, int64_t nrows, const int64_t *__restrict__ rowptr, uint32_t *rowinfo,
                    const int32_t *__restrict__ col, const ValT *__restrict__ val, int64_t base0, int32_t *tcol, ValT *tval)
{
    constexpr int WPB = kSBlock / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t s = s0 + (int64_t)blockIdx.x * WPB + warp; s < s1; s += (int64_t)gridDim.x * WPB) {
        const int64_t r = s * 32 + lane;
        const int64_t rs = r < nrows ? rowptr[r] : 0;
        const int64_t len64 = r < nrows ? rowptr[r + 1] - rs : 0;
        const int len = (int)len64;                         // (< 2^24: checked by sjds_rows_fit before any entry moves)
        int rank = 0, maxlen = 0;
        for (int j = 0; j < 32; j++) {                      // rank by (length desc, lane asc): a stable sort of 32 keys
            const int lj = __shfl_sync(0xffffffffu, len, j);
            rank += (lj > len) || (lj == len && j < lane);
            maxlen = max(maxlen, lj);
        }
        if (FORWARD) rowinfo[s * 32 + rank] = ((uint32_t)lane << 24) | (uint32_t)len;
        int64_t off = rowptr[s * 32] - base0;
        for (int k = 0; k < maxlen; k++) {
            const bool act = k < len;
            const int cnt = __popc(__ballot_sync(0xffffffffu, act));
            if (act) {
                const int64_t jag = off + rank, csr = rs + k;           // jag is relative to base0, csr absolute
                if (FORWARD) { tcol[jag] = col[csr]; tval[jag] = val[csr]; }
                else         { tcol[csr - base0] = col[base0 + jag]; tval[csr - base0] = val[base0 + jag]; }
            }
            off += cnt;
        }
    }
}

__global__ void __launch_bounds__(kSBlock) sjds_row_too_long_kernel(int64_t nrows, const int64_t *__restrict__ rowptr, int *too_long)
{
    for (int64_t r = (int64_t)blockIdx.x * kSBlock + threadIdx.x; r < nrows; r += (int64_t)gridDim.x * kSBlock)
        if (rowptr[r + 1] - rowptr[r] > (int64_t)kLenMask) *too_long = 1;
}

// Does every row fit the 24-bit length field of the sliced-jagged row metadata?  (Asked before the conversion moves any entry:
// a refused conversion leaves the CSR arrays as they were.)
int sjds_rows_fit(const qbgpu_matrix *A, bool *fits)
{
    Context &c = ctx();
    *fits = true;
    const int64_t nrows = A->nrows();
    if (nrows == 0) return QBGPU_OK;
    int *d_flag = nullptr;
    int flag = 0;
    QB_CUDA(cudaMalloc(&d_flag, sizeof(int)));
    cudaError_t e = cudaMemsetAsync(d_flag, 0, sizeof(int), c.stream);
    if (e == cudaSuccess) {
        sjds_row_too_long_kernel<<<(int)std::min<int64_t>((nrows + kSBlock - 1) / kSBlock, 148 * 16), kSBlock, 0, c.stream>>>(nrows, A->rowptr, d_flag);
        QB_LAUNCH_COUNT();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, c.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
    cudaFree(d_flag);
    QB_CUDA(e);
    *fits = flag == 0;
    return QBGPU_OK;
}

template <typename ValT>
static int sjds_convert_typed(qbgpu_matrix *A, bool forward)
{
    Context &c = ctx();
    const int64_t nrows = A->nrows();
    const int64_t nslices = (nrows + 31) / 32;
    if (nslices == 0) return QBGPU_OK;
    if (forward) {
        bool fits = true;
        QB_TRY(sjds_rows_fit(A, &fits));
        if (!fits) return fail(QBGPU_ERR_STATE, "sliced-jagged layout: a row is longer than 2^24-1 entries");
    }
    if (forward && !A->rowinfo) QB_CUDA(cudaMalloc(&A->rowinfo, sizeof(uint32_t) * nslices * 32));
    // batches of slices re-ordered through a bounded temporary, then copied back over the same range
    const int64_t batch = 1 << 16;                          // 65,536 slices = 2,097,152 rows per batch
    const int64_t nb = (nslices + batch - 1) / batch;
    std::vector<int64_t> bidx(nb + 1), bofs(nb + 1);
    for (int64_t b = 0; b <= nb; b++) bidx[b] = std::min(nrows, b * batch * 32);
    int32_t *tcol = nullptr;
    ValT *tval = nullptr;
    auto cleanup = [&]() { cudaFree(tcol); cudaFree(tval); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    // boundary offsets rowptr[bidx[b]]
    for (int64_t b = 0; b <= nb; b++) QB_CU(cudaMemcpyAsync(&bofs[b], A->rowptr + bidx[b], sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    int64_t maxspan = 1;
    for (int64_t b = 0; b < nb; b++) maxspan = std::max(maxspan, bofs[b + 1] - bofs[b]);
    QB_CU(cudaMalloc(&tcol, sizeof(int32_t) * maxspan));
    QB_CU(cudaMalloc(&tval, sizeof(ValT) * maxspan));
    for (int64_t b = 0; b < nb; b++) {
        const int64_t s0 = b * batch, s1 = std::min(nslices, (b + 1) * batch);
        const int64_t span = bofs[b + 1] - bofs[b];
        if (span == 0 && !forward) continue;               // (forward still has to write rowinfo for all-empty slices)
        const int grid = (int)std::min<int64_t>((s1 - s0 + 7) / 8, 148 * 16);
        if (forward) sjds_permute_kernel<ValT, true><<<grid, kSBlock, 0, c.stream>>>(s0, s1, nrows, A->rowptr, A->rowinfo, A->col, (const ValT *)A->val, bofs[b], tcol, tval);
        else         sjds_permute_kernel<ValT, false><<<grid, kSBlock, 0, c.stream>>>(s0, s1, nrows, A->rowptr, A->rowinfo, A->col, (const ValT *)A->val, bofs[b], tcol, tval);
        QB_LAUNCH_COUNT();
        if (span) {
            QB_CU(cudaMemcpyAsync(A->col + bofs[b], tcol, sizeof(int32_t) * span, cudaMemcpyDeviceToDevice, c.stream));
            QB_CU(cudaMemcpyAsync((ValT *)A->val + bofs[b], tval, sizeof(ValT) * span, cudaMemcpyDeviceToDevice, c.stream));
        }
    }
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
    cleanup();
#undef QB_CU
    A->format = forward ? QBGPU_FORMAT_SELL : QBGPU_FORMAT_CSR;
    return QBGPU_OK;
}

int sjds_convert(qbgpu_matrix *A, bool forward)
{
    if (forward == (A->format == QBGPU_FORMAT_SELL)) return QBGPU_OK;
    if (A->cbits) return fail(QBGPU_ERR_STATE, "packed entry words stay in the sliced-jagged layout");
    if (A->ndict) return sjds_convert_typed<uint8_t>(A, forward);
    return A->val_real ? sjds_convert_typed<double>(A, forward) : sjds_convert_typed<double2>(A, forward);
}

// ------------------------------------------------------------------------------------------ ring order of a shard
// CSR layout, one thread per row: rotate the (ascending) entries so that the first one is the first column >= pivot
// (three reversals, in place).
template <typename ValT>
__global__ void __launch_bounds__(kSBlock) ring_rotate_kernel(int64_t nrows, const int64_t *__restrict__ rowptr, int32_t *col, ValT *val, int32_t pivot_col)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = rowptr[r], e = rowptr[r + 1];
        int64_t lo = s, hi = e;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (col[mid] < pivot_col) lo = mid + 1; else hi = mid; }
        const int64_t p = lo;                               // entries [s, p) move behind [p, e)
        if (p == s || p == e) continue;
        auto rev = [&](int64_t i, int64_t j) {              // reverse [i, j)
            for (j--; i < j; i++, j--) { const int32_t tc = col[i]; col[i] = col[j]; col[j] = tc; const ValT tv = val[i]; val[i] = val[j]; val[j] = tv; }
        };
        rev(s, p); rev(p, e); rev(s, e);
    }
}

int ring_prepare(qbgpu_matrix *A, int rank, int world, int64_t chunk, qbgpu_matrix **view)
{
    Context &c = ctx();
    if (!A || A->mf || A->mf_sec || A->borrowed) return fail(QBGPU_ERR_ARG, "ring_prepare: needs an owning, stored matrix handle");
    if (!view) return fail(QBGPU_ERR_ARG, "ring_prepare: null view pointer");
    *view = nullptr;
    if (A->ring_world) return fail(QBGPU_ERR_STATE, "ring_prepare: already in ring order");
    if (world < 2 || rank < 0 || rank >= world || chunk <= 0 || chunk > 0x7fffffff) return fail(QBGPU_ERR_ARG, "ring_prepare: bad rank/world/chunk");
    if (chunk % 4) return fail(QBGPU_ERR_ARG, "ring_prepare: the slice length must be a multiple of 4 rows (32-byte sectors must not straddle two owners)");
    if (A->row_lo != (int64_t)rank * chunk) return fail(QBGPU_ERR_ARG, "ring_prepare: the shard does not start at rank * chunk");
    const bool was_sell = A->format == QBGPU_FORMAT_SELL;
    if (was_sell) QB_TRY(sjds_convert(A, false));
    const int64_t nrows = A->nrows();
    const int grid = (int)std::min<int64_t>((nrows + kSBlock - 1) / kSBlock, 148 * 32);
    const int32_t pivot = (int32_t)A->row_lo;
    if (nrows) {
        if (A->ndict) ring_rotate_kernel<uint8_t><<<grid, kSBlock, 0, c.stream>>>(nrows, A->rowptr, A->col, (uint8_t *)A->val, pivot);
        else if (A->val_real) ring_rotate_kernel<double><<<grid, kSBlock, 0, c.stream>>>(nrows, A->rowptr, A->col, (double *)A->val, pivot);
        else ring_rotate_kernel<double2><<<grid, kSBlock, 0, c.stream>>>(nrows, A->rowptr, A->col, (double2 *)A->val, pivot);
        QB_LAUNCH_COUNT();
        QB_CUDA(cudaGetLastError());
    }
    QB_TRY(sjds_convert(A, true));                          // the ring kernel exists for the sliced-jagged layout only
    QB_CUDA(cudaStreamSynchronize(c.stream));
    // The waiting kernel is selected through a VIEW that shares A's arrays; A itself keeps working (its rows are merely in
    // a different order) with the ordinary kernels, e.g. behind an all-gather.
    auto *V = new qbgpu_matrix(*A);
    V->borrowed = true;
    V->ring_world = world; V->ring_rank = rank; V->ring_chunk = chunk;
    *view = V;
    return QBGPU_OK;
}

}  // namespace qb
