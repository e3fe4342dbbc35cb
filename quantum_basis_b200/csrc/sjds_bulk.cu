// quantum_basis_b200/csrc/sjds_bulk.cu -- the sliced-jagged H*v with the matrix stream moved by the copy engine of the SM
// (cp.async.bulk + mbarrier, sm_100a), and the block-local product with the gathered vector staged in shared memory.
//
// Why (profiles/r02_ncu_species_stored_two_pass_hubbard4x4.csv): with the register-fed kernel of sjds.cu a warp has one
// trip of U jagged diagonals in flight -- column load -> gather is a dependent chain of two long latencies -- and 32 warps
// per SM then sustain only 4.2-4.7 TB/s of DRAM traffic (long-scoreboard stalls: 21-33 per issue), although nothing is
// saturated.  Two remedies, one per access pattern:
//
//  (1) spmv_sjds_bulk_kernel -- every warp owns a ring of NST stages in shared memory.  A stage receives one SEGMENT of a
//      32-row slice: KSEG consecutive jagged diagonals, which are one contiguous range of col[] and of val[] (sjds.cu), so a
//      segment is two bulk copies (UBLKCP in the SASS; one for packed words) that complete on the stage's mbarrier.  NST-1
//      segments are in flight per warp while one is consumed: the stream is fetched exactly once, in whole lines, with no
//      registers held, and the only long-latency instructions left in the loop are the gathers of x, issued KSEG at a time.
//      The producer is the consumer warp itself (lane 0 issues): no CTA-wide synchronisation, ragged slices are natural.
//
//  (2) sjds_block_smem_kernel -- for a matrix whose rows [u*D, (u+1)*D) only reference columns of the same block (the
//      "local" part of a species-order Hubbard handle: diagonal + hops of the down electrons, species.cu).  Gathers of 16-byte
//      elements scattered over a 206 KB block cost one L1 tag wavefront per distinct line (about 2 cycles each inside one
//      LDG, B300_MICROARCH.md) -- that, not DRAM, bounded the pass at 10 ms.  Here one CTA owns the block: x[u*D .. (u+1)*D)
//      is brought into shared memory by ONE bulk copy, the gathers become LDS.128 (a quarter-warp per wavefront, bank
//      conflicts only), and the matrix stream keeps the register-fed path with many loads in flight.
//
//  (3) sjds_cross_slices_kernel -- the packed cross part of a species handle with fp64 vectors: one whole 32-row slice per
//      warp item, register-fed, no ring; most slices are uniform (all rows of the same length) and pay no votes.
//
// All three keep the arithmetic of sjds.cu: same entries, same order of accumulation per row (two alternating accumulators over
// the jagged diagonals), so products are bit-identical to spmv_sjds_kernel.
#include "internal.hpp"
#include <cstdlib>
#include <type_traits>

namespace qb {

constexpr uint32_t kLenMaskB = 0xFFFFFFu;

// ---------------------------------------------------------------------------------------------- PTX helpers (sm_100a)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{ asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{ asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory"); }
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// (a bulk copy that never completes would otherwise hang the device: after ~2^26 failed probes -- seconds -- trap instead)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    unsigned spins = 0;
    while (!mbar_try_wait(bar, parity)) { if (++spins > (1u << 26)) __trap(); }
}
// generic-proxy accesses to shared memory before this point are ordered before later async-proxy (bulk copy) writes
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// global -> shared bulk copy (dst, src and bytes multiples of 16), completing `bytes` on the mbarrier; L2 evict-first hint
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint64_t pol)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
__device__ __forceinline__ void bulk_g2s_plain(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ uint64_t pol_evict_first() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ uint64_t pol_evict_last()  { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p; }

__device__ __forceinline__ double ldx_hint(const double *p, uint64_t pol)
{ double v; asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol)); return v; }
__device__ __forceinline__ double2 ldx_hint(const double2 *p, uint64_t pol)
{ double2 v; asm volatile("ld.global.nc.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol)); return v; }

// streaming loads of the matrix arrays for the register-fed path of kernel (2)
__device__ __forceinline__ int lds_i32(const int *p, uint64_t pol)
{ int v; asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol)); return v; }
__device__ __forceinline__ double lds_val(const double *p, uint64_t pol)
{ double v; asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol)); return v; }
__device__ __forceinline__ double2 lds_val(const double2 *p, uint64_t pol)
{ double2 v; asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol)); return v; }

// ------------------------------------------------------------------------------------------ (1) bulk-streamed product
// Stage layout (per warp, per stage; every area 16-byte aligned):
//   hdr[8]  int32 : [0..1] first entry of the segment (int64), [2] entries, [3] first diagonal k0, [4] slice index (< 2^31)
//   info[32] uint32: rowinfo of the slice
//   col  int32[CAP + 8], val ValT[CAP + VPAD]: the copies start at the entry rounded DOWN to a 16-byte boundary
//   (packed words, ValT = uint32_t: the col area holds col | code << cbits and there is no val area)
template <typename ValT, int KSEG> struct BulkStage {
    static constexpr bool PACKED = std::is_same<ValT, uint32_t>::value;
    static constexpr int CAP = 32 * KSEG;
    static constexpr int VALIGN = 16 / (int)sizeof(ValT) > 0 ? 16 / (int)sizeof(ValT) : 1;   // entries per 16 bytes of val
    static constexpr int VPAD = 2 * VALIGN;
    static constexpr int HDR_BYTES = 32 + 128;
    static constexpr int COL_BYTES = (CAP + 8) * 4;
    static constexpr int VAL_BYTES = PACKED ? 0 : ((CAP + VPAD) * (int)sizeof(ValT) + 15) / 16 * 16;
    static constexpr int BYTES = HDR_BYTES + COL_BYTES + VAL_BYTES;
};
// the mbarriers of one warp's ring (8 bytes per stage) come before all rings, in whole 64-byte blocks per warp
constexpr int bulk_bar_bytes(int nst) { return (8 * nst + 63) / 64 * 64; }

// What the consumer keeps of a segment between its two phases (gathers issued / products accumulated)
template <typename VecT> struct SegState {
    uint32_t info;        // rowinfo of this lane's rank in the segment's slice
    int k0;               // first jagged diagonal of the segment
    int cnt;              // entries (0: nothing was copied, nothing to wait for)
    bool last, live, full; // last segment of its slice; this lane writes a row in the epilogue; every lane has all KSEG diagonals
    int64_t row;
    int32_t rref;         // OUT: the reference's row of this lane's row (perm_inv), requested together with the gathers
    VecT zv, xi;          // epilogue operands, requested together with the gathers
};

// Two segments are in the consumer at a time -- the gathers of segment j+1 are issued before the products of segment j
// are accumulated (ping-pong register sets), so a warp always has up to 2*KSEG gathers in flight.
__device__ __forceinline__ double real_of(double v) { return v; }
__device__ __forceinline__ double real_of(double2 v) { return v.x; }

// OUT: the way out of a species handle fused into this (closing, accumulating) pass: y_ref[perm_inv[row]] = out_alpha * (y, 0)
// instead of y[row] = y (fp64 vectors only; see FusedArgs::y_ref).  The rows of a tile that share a sector of y_ref are
// closed within microseconds of each other (neighbouring up configurations of the same tile), so L2 merges the halves.
// The 32-row slices are visited in the order given by `order` (the tiles of down indices of a cross part, so that the
// gathered columns of a tile stay in L2).
template <typename ValT, typename VecT, bool DOTS, bool KEEP, int NW, int NST, int KSEG, bool OUT = false>
__global__ void __launch_bounds__(NW * 32, 2)
spmv_sjds_bulk_kernel(int64_t nslices, int64_t nrows, int64_t row_lo, const int64_t *__restrict__ rowptr,
                      const uint32_t *__restrict__ rowinfo, const int32_t *__restrict__ col, const ValT *__restrict__ val,
                      const VecT *__restrict__ x, const VecT *z, VecT *y, double2 alpha, double2 gamma, double2 beta,
                      int scal_mode, const double *__restrict__ sc, double *dots_out, double *partials, unsigned *ticket,
                      const double *__restrict__ vdict, const int32_t *__restrict__ order, int cbits,
                      const int32_t *__restrict__ perm_inv = nullptr, double2 *y_ref = nullptr, double2 out_alpha = {1.0, 0.0})
{
    static_assert(!OUT || (sizeof(VecT) == 8 && !DOTS), "the fused way out serves the fp64 closing pass");
    using VT = VecTraits<VecT>;
    using ST = BulkStage<ValT, KSEG>;
    using Seg = SegState<VecT>;
    static_assert(KSEG % 2 == 0 && KSEG >= 2, "diagonal k accumulates into accumulator k & 1 (the order of sjds.cu)");
    static_assert(NST >= 3, "the pipelined consumer holds two stages");
    constexpr bool kPacked = ST::PACKED;
    static_assert(kPacked || sizeof(ValT) >= 8, "values are fp64, complex, or packed codes");
    using ArithT = typename std::conditional<kPacked, double, ValT>::type;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ double sdict[kPacked ? kPackedMaxTable : 1];
    if (kPacked) { for (int i = threadIdx.x; i < (int)kPackedMaxTable; i += NW * 32) sdict[i] = vdict[i]; __syncthreads(); }
    const uint32_t cmask = kPacked ? (1u << cbits) - 1u : ~0u;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int BARB = bulk_bar_bytes(NST);
    unsigned char *wbase = smem_raw + BARB * NW + (size_t)warp * NST * ST::BYTES;    // [NW][NST] barriers first
    const uint32_t bar0 = smem_u32(smem_raw + BARB * warp);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < NST; s++) mbar_init(bar0 + 8 * s, 1);
        mbar_fence_init();
    }
    __syncwarp();
    const uint64_t pol_s = pol_evict_first(), pol_x = pol_evict_last();
    // the scalars of the epilogue live in shared memory (they are needed once per slice; as registers they would stay live
    // across the whole pipeline): [0] alpha, [1] gamma, [2] beta, [3].x the scale of the running dots
    __shared__ double2 s_scal[4];
    if (threadIdx.x == 0) {
        double dot_scale = 1.0;
        if (scal_mode != 0) {                              // Lanczos step a: 1 = first column block, 2 = a later one (sjds.cu)
            const double sx = sc[0], sz = sc[1], bprev = sc[2];
            alpha = make_double2(sx, 0.0);
            gamma = make_double2(0.0, 0.0);
            beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
            dot_scale = sx;
        }
        s_scal[0] = alpha; s_scal[1] = gamma; s_scal[2] = beta; s_scal[3] = make_double2(dot_scale, 0.0);
    }
    __syncthreads();
    const bool use_gamma = (s_scal[1].x != 0.0 || s_scal[1].y != 0.0);
    const bool use_beta = (s_scal[2].x != 0.0 || s_scal[2].y != 0.0);
    double d[3] = {0.0, 0.0, 0.0};

    // ---- producer cursor: slice `ps` (iteration p_it of this warp), next diagonal pk, entries of the slice before pk
    const int stride = (int)gridDim.x * NW;                // (slice counts are < 2^31: rows < 2^31 by the int32 columns)
    const int nsl = (int)nslices;
    int p_it = (int)blockIdx.x * NW + warp;
    auto slice_of = [&](int it) -> uint32_t { return it < nsl ? (uint32_t)order[it] : 0u; };      // traversal item -> slice
    auto info_of = [&](uint32_t sl) -> uint32_t { return rowinfo[(int64_t)sl * 32 + lane]; };
    bool p_more = p_it < nsl;
    const uint32_t pd = slice_of(p_it);
    int ps = (int)pd;
    uint32_t pinfo = p_more ? info_of(pd) : 0u;
    int64_t pbase = p_more ? rowptr[(int64_t)ps * 32] : 0;
    int pk = 0, poff = 0;
    // one slice ahead: requested when the producer enters a slice, consumed when it enters the next (no exposed latency)
    int n_it = p_it + stride;
    const uint32_t nd0 = slice_of(n_it);
    int ns = (int)nd0;
    uint32_t ninfo = n_it < nsl ? info_of(nd0) : 0u;
    int64_t nbase = n_it < nsl ? rowptr[(int64_t)ns * 32] : 0;
    uint32_t nn_d = slice_of(n_it + stride);                                         // the slice after that (a dependent load)

    uint32_t phases = 0;                                   // bit s = parity the consumer waits for on stage s
    int n_issued = 0;                                      // segments issued so far; segment i lives in stage i % NST

    auto issue = [&]() {
        const int st = n_issued % NST;
        n_issued++;
        // (all lanes) entries of diagonals [pk, pk + KSEG) of the producer's slice
        const int len = (int)(pinfo & kLenMaskB);
        const int maxlen = __shfl_sync(0xffffffffu, len, 0);
        const int hi = min(len, pk + KSEG), lo = min(len, pk);
        const int cnt = (int)__reduce_add_sync(0xffffffffu, (unsigned)(hi - lo));
        unsigned char *sb = wbase + (size_t)st * ST::BYTES;
        __syncwarp();
        ((uint32_t *)(sb + 32))[lane] = pinfo;
        if (lane == 0) {
            const int64_t beg = pbase + poff;
            int *hdr = (int *)sb;
            *(int64_t *)hdr = beg; hdr[2] = cnt; hdr[3] = pk; hdr[4] = ps;
            if (cnt > 0) {
                fence_proxy_async_smem();
                const int64_t c0 = beg & ~3LL, c1 = (beg + cnt + 3) & ~3LL;                       // 16-byte aligned col range
                const int64_t v0 = beg & ~(int64_t)(ST::VALIGN - 1), v1 = (beg + cnt + ST::VALIGN - 1) & ~(int64_t)(ST::VALIGN - 1);
                const uint32_t cb = (uint32_t)(c1 - c0) * 4u, vb = kPacked ? 0u : (uint32_t)((v1 - v0) * (int64_t)sizeof(ValT));
                const uint32_t bar = bar0 + 8 * st;
                mbar_expect_tx(bar, cb + vb);
                bulk_g2s(smem_u32(sb + ST::HDR_BYTES), col + c0, cb, bar, pol_s);
                if constexpr (!kPacked) bulk_g2s(smem_u32(sb + ST::HDR_BYTES + ST::COL_BYTES), val + v0, vb, bar, pol_s);
            }
        }
        __syncwarp();
        poff += cnt;
        pk += KSEG;
        if (pk >= maxlen) {                                // slice finished (also: an empty slice is one empty segment)
            p_it += stride;
            p_more = p_it < nsl;
            ps = ns; pinfo = ninfo; pbase = nbase; pk = 0; poff = 0;
            n_it += stride;
            ns = (int)nn_d;
            const bool nv = n_it < nsl;
            ninfo = nv ? info_of(nn_d) : 0u;
            nbase = nv ? rowptr[(int64_t)ns * 32] : 0;
            nn_d = slice_of(n_it + stride);
        }
    };

    VecT acc0 = VT::zero(), acc1 = VT::zero();

    // phase 1 of segment `seg`: wait for its copies, read the columns, issue the gathers (and the epilogue's operands).
    // FULL segment (every lane has all KSEG diagonals: the shortest row of the slice, rank 31, reaches k0 + KSEG): entry
    // (u, lane) sits at u*32 + lane -- constant offsets, no votes, no predicates.  Ragged segments: predicated per lane.
    auto gather = [&](int seg, Seg &g, VecT (&xv)[KSEG]) {
        const int st = seg % NST;
        unsigned char *sb = wbase + (size_t)st * ST::BYTES;
        const int4 h = *(const int4 *)sb;                  // beg (lo, hi), cnt, k0
        const int s = ((const int *)sb)[4];
        g.cnt = h.z; g.k0 = h.w;
        g.info = ((const uint32_t *)(sb + 32))[lane];
        const int len = (int)(g.info & kLenMaskB);
        const int maxlen = __shfl_sync(0xffffffffu, len, 0);
        const int minlen = __shfl_sync(0xffffffffu, len, 31);
        g.last = g.k0 + KSEG >= maxlen;
        g.full = g.k0 + KSEG <= minlen;
        g.row = (int64_t)s * 32 + (g.info >> 24);
        g.live = g.last && g.row < nrows && !(KEEP && !OUT && len == 0);      // padding ranks of the last slice point past the last row
        if (g.cnt > 0) {
            mbar_wait(bar0 + 8 * st, (phases >> st) & 1u);
            phases ^= 1u << st;
            const uint32_t *scol = (const uint32_t *)(sb + ST::HDR_BYTES) + (h.x & 3) + lane;
            if (g.full) {
#pragma unroll
                for (int u = 0; u < KSEG; u++) xv[u] = ldx_hint(x + (scol[u * 32] & cmask), pol_x);
            } else {
                int off = 0;
#pragma unroll
                for (int u = 0; u < KSEG; u++) {
                    const bool a = g.k0 + u < len;
                    if (a) xv[u] = ldx_hint(x + (scol[off] & cmask), pol_x);
                    off += __popc(__ballot_sync(0xffffffffu, a));
                }
            }
        }
        if (g.live) {
            if (use_beta) g.zv = z[g.row];
            if (use_gamma || DOTS) g.xi = x[row_lo + g.row];
            if constexpr (OUT) g.rref = perm_inv[row_lo + g.row];
        }
    };

    // phase 2: accumulate, and close the slice after its last segment (the epilogue of sjds.cu)
    auto fma_phase = [&](int seg, const Seg &g, VecT (&xv)[KSEG]) {
        const int st = seg % NST;
        unsigned char *sb = wbase + (size_t)st * ST::BYTES;
        if (g.k0 == 0) { acc0 = VT::zero(); acc1 = VT::zero(); }
        if (g.cnt > 0) {
            const int begl = *(const int *)sb;
            const ValT *sval = (const ValT *)(sb + ST::HDR_BYTES + ST::COL_BYTES) + (begl & (ST::VALIGN - 1)) + lane;
            const uint32_t *sword = (const uint32_t *)(sb + ST::HDR_BYTES) + (begl & 3) + lane;
            // diagonal k0 + u goes to accumulator (k0 + u) & 1 == u & 1 (KSEG is even): the order of sjds.cu
            if (g.full) {
#pragma unroll
                for (int u = 0; u < KSEG; u++) {
                    ArithT w;
                    if constexpr (kPacked) w = sdict[sword[u * 32] >> cbits]; else w = sval[u * 32];
                    if (u & 1) mac(acc1, w, xv[u]); else mac(acc0, w, xv[u]);
                }
            } else {
                const int len = (int)(g.info & kLenMaskB);
                int off = 0;
#pragma unroll
                for (int u = 0; u < KSEG; u++) {
                    const bool a = g.k0 + u < len;
                    if (a) {
                        ArithT w;
                        if constexpr (kPacked) w = sdict[sword[off] >> cbits]; else w = sval[off];
                        if (u & 1) mac(acc1, w, xv[u]); else mac(acc0, w, xv[u]);
                    }
                    off += __popc(__ballot_sync(0xffffffffu, a));
                }
            }
        }
        if (g.live) {
            const VecT acc = VT::add(acc0, acc1);
            VecT out = VT::scale(s_scal[0], acc);
            if (use_gamma) out = VT::add(out, VT::scale(s_scal[1], g.xi));
            if (use_beta) out = VT::add(out, VT::scale(s_scal[2], g.zv));
            if constexpr (OUT) {
                const double re = real_of(out);
                y_ref[g.rref] = make_double2(out_alpha.x * re, out_alpha.y * re);
            } else y[g.row] = out;
            if (DOTS) {
                const double2 p = VT::conj_mul(g.xi, out);
                d[0] += p.x; d[1] += p.y; d[2] += VT::abs2(out);
            }
        }
        __syncwarp();                                      // every lane is done with the stage before it is refilled
    };

    // prologue: fill the ring
#pragma unroll 1
    for (int s = 0; s < NST && p_more; s++) issue();
    int n_gathered = 0;
    Seg ga, gb;
    VecT xa[KSEG], xb[KSEG];
    if (n_gathered < n_issued) {
        gather(n_gathered, ga, xa); n_gathered++;
#pragma unroll 1
        while (true) {
            const bool hb = n_gathered < n_issued;
            if (hb) { gather(n_gathered, gb, xb); n_gathered++; }
            fma_phase(n_gathered - (hb ? 2 : 1), ga, xa);
            if (p_more) issue();
            if (!hb) break;
            const bool ha = n_gathered < n_issued;
            if (ha) { gather(n_gathered, ga, xa); n_gathered++; }
            fma_phase(n_gathered - (ha ? 2 : 1), gb, xb);
            if (p_more) issue();
            if (!ha) break;
        }
    }
    if (DOTS) {
        d[0] *= s_scal[3].x; d[1] *= s_scal[3].x;
        block_reduce_finalize<3, NW * 32>(d, partials, ticket, dots_out);
    }
}

// may the closing pass over this (cross) part write the reference-order result itself?
bool sjds_bulk_out_fusable(const qbgpu_matrix *A)
{
    return A && A->format == QBGPU_FORMAT_SELL && A->slice_order && A->ring_world <= 1;
}

template <typename ValT, typename VecT, bool DOTS, bool KEEP, int NW, int NST, int KSEG, bool OUT = false>
static int launch_bulk_cfg(const qbgpu_matrix *A, const FusedArgs &a)
{
    Context &c = ctx();
    using ST = BulkStage<ValT, KSEG>;
    auto kern = spmv_sjds_bulk_kernel<ValT, VecT, DOTS, KEEP, NW, NST, KSEG, OUT>;
    constexpr size_t smem = (size_t)bulk_bar_bytes(NST) * NW + (size_t)NW * NST * ST::BYTES;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        QB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, NW * 32, smem));
        if (blocks_per_sm < 1) return fail(QBGPU_ERR_STATE, "bulk-streamed product: the stage ring does not fit in shared memory");
        if (getenv("QBGPU_VERBOSE")) fprintf(stderr, "[qbgpu] bulk kernel NW=%d NST=%d KSEG=%d: %d CTAs/SM, %zu B smem\n", NW, NST, KSEG, blocks_per_sm, smem);
    }
    const int64_t nrows = A->nrows();
    if (nrows == 0) return QBGPU_OK;
    const int64_t nslices = (nrows + 31) / 32;
    int64_t want = (nslices + NW - 1) / NW;
    int64_t cap = (int64_t)c.num_sms * blocks_per_sm;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    const int grid = (int)(want < cap ? want : cap);
    kern<<<grid, NW * 32, smem, c.stream>>>(nslices, nrows, A->row_lo, A->rowptr, A->rowinfo, A->col, (const ValT *)A->val,
                                            (const VecT *)a.x, (const VecT *)a.z, (VecT *)a.y, a.alpha, a.gamma, a.beta,
                                            a.scal_mode, a.sc, a.dots, c.partials, c.ticket, A->vdict, A->slice_order, A->cbits,
                                            OUT ? a.perm_inv : nullptr, OUT ? (double2 *)a.y_ref : nullptr, a.out_alpha);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

// (warps per CTA, stages per warp, diagonals per segment).  What the stage rings take from the SM's 256 KB of SRAM is lost
// to L1, and L1 lines are what gathers in flight are tracked in: with fp64 vectors a fat ring (106 KB per CTA, two CTAs)
// is best; with complex vectors (twice the lines per gather) a leaner one (profiles/r02_bulk_sweep_*.txt: 8,4,8 is 2x
// slower than 8,3,6 there).  Packed words (4 bytes per entry, one bulk copy per segment) keep the segment length and with it
// the gathers in flight, and take more, smaller stages.  Packed parts with fp64 vectors take kernel (3) instead.
template <typename ValT, typename VecT> struct BulkRing {
    static constexpr bool kPacked = std::is_same<ValT, uint32_t>::value, kCplx = sizeof(VecT) == 16;
    static_assert(!kPacked || kCplx, "packed parts with fp64 vectors take sjds_cross_slices_kernel");
    static constexpr int NW = 8;
    static constexpr int NST = kPacked ? 6 : (kCplx ? 3 : 4);
    static constexpr int KSEG = kCplx ? 6 : 8;
};

template <typename ValT, typename VecT, bool DOTS, bool KEEP>
static int launch_bulk_ring(const qbgpu_matrix *A, const FusedArgs &a)
{
    using R = BulkRing<ValT, VecT>;
    return launch_bulk_cfg<ValT, VecT, DOTS, KEEP, R::NW, R::NST, R::KSEG>(A, a);
}

template <typename ValT, typename VecT>
static int launch_bulk_typed(const qbgpu_matrix *A, const FusedArgs &a)
{
    const bool dots = a.dots != nullptr;
    const bool keep = !dots && a.scal_mode == 0 && a.z == a.y && a.beta.x == 1.0 && a.beta.y == 0.0 && a.gamma.x == 0.0 && a.gamma.y == 0.0;
    if (a.y_ref) {                                          // the closing pass of a species product writes the reference's order
        if constexpr (sizeof(VecT) == 8) {
            using R = BulkRing<ValT, VecT>;
            if (keep && a.perm_inv) return launch_bulk_cfg<ValT, VecT, false, true, R::NW, R::NST, R::KSEG, true>(A, a);
        }
        return fail(QBGPU_ERR_STATE, "fused way out: not the closing pass of a species handle (internal)");
    }
    if (keep) return launch_bulk_ring<ValT, VecT, false, true>(A, a);
    return dots ? launch_bulk_ring<ValT, VecT, true, false>(A, a) : launch_bulk_ring<ValT, VecT, false, false>(A, a);
}

// ------------------------------------------------------------------- (3) slice-granular product of a packed cross part
// The cross part of a species handle (hops of the up electrons, species.cu) has rows whose length is the up-hop count of
// the row's up configuration: every 32-row slice that stays inside one block of D_dn rows is UNIFORM -- all 32 ranks have
// the same length L, and entry (k, rank) sits at rowptr[32 s] + 32 k + rank.  Only slices that straddle two blocks (one in
// about 400 on BASELINE config 3), the last partial slice and slices with empty rows are ragged.  So one warp takes one
// traversal item of `order` -- a whole slice, in tile order as kernel (1) visits them -- and per trip of kXTrip diagonals
// requests all the trip's entry words, then all its gathers of x, then accumulates.  A uniform slice pays no votes, no
// per-segment headers and no shared-memory ring: its offsets are constants.  A ragged slice takes the same trips with a
// per-lane predicate and the offsets of its diagonals counted by ballots (the layout of sjds.cu).
// Same entries, same order of accumulation (diagonal k into accumulator k & 1, ascending k), same epilogue as kernel (1):
// products, the fused way out and the running dots are bit-identical to it.
//
// Registers bound the trip: a word and a gathered double per diagonal in flight.  With a two-entry value table (the cross
// part of a Hubbard model: +-t) the value is a select between two registers, and a trip keeps its codes as one bit each.
constexpr int kXWarps = 8;              // warps per CTA: the block of the running dots' reduction tree, as in kernel (1)
constexpr int kXTrip = 12;              // diagonals per trip (even: diagonal k + u accumulates into u & 1)
constexpr int kXMinBlocks = 4;          // CTAs per SM the register budget is set for (64 registers a thread)
// (BASELINE config 3, closing pass, one B200 at 1000 W: 12 diagonals at 4 CTAs per SM 6.08 ms, 16 at 3 CTAs 6.23 ms; an L2 bulk
// prefetch of the next slice's words made both slower, 6.14 and 6.71 ms)
// The order of the running dots depends on the grid (block_reduce_finalize): the DOTS pass keeps the grid of kernel (1)
// with packed words -- two CTAs of 8 warps per SM -- so that Lanczos coefficients stay bit-identical.
constexpr int kXDotsBlocksPerSm = 2;

template <bool DOTS, bool KEEP, bool OUT, bool TWO>
__global__ void __launch_bounds__(kXWarps * 32, DOTS ? kXDotsBlocksPerSm : kXMinBlocks)
sjds_cross_slices_kernel(int64_t nslices, int64_t nrows, int64_t row_lo, const int64_t *__restrict__ rowptr,
                         const uint32_t *__restrict__ rowinfo, const int32_t *__restrict__ words, const double *__restrict__ x,
                         const double *z, double *y, double2 alpha, double2 gamma, double2 beta, int scal_mode,
                         const double *__restrict__ sc, double *dots_out, double *partials, unsigned *ticket,
                         const double *__restrict__ vdict, const int32_t *__restrict__ order, int cbits,
                         const int32_t *__restrict__ perm_inv, double2 *y_ref, double2 out_alpha)
{
    static_assert(!OUT || !DOTS, "the fused way out serves the closing pass without dots");
    using VT = VecTraits<double>;
    __shared__ double sdict[TWO ? 1 : kPackedMaxTable];
    if (!TWO) for (int i = threadIdx.x; i < (int)kPackedMaxTable; i += kXWarps * 32) sdict[i] = vdict[i];
    __shared__ double2 s_scal[4];                          // [0] alpha, [1] gamma, [2] beta, [3].x the scale of the running dots
    if (threadIdx.x == 0) {
        double dot_scale = 1.0;
        if (scal_mode != 0) {                              // Lanczos step a: 1 = first column block, 2 = a later one (sjds.cu)
            const double sx = sc[0], sz = sc[1], bprev = sc[2];
            alpha = make_double2(sx, 0.0);
            gamma = make_double2(0.0, 0.0);
            beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
            dot_scale = sx;
        }
        s_scal[0] = alpha; s_scal[1] = gamma; s_scal[2] = beta; s_scal[3] = make_double2(dot_scale, 0.0);
    }
    __syncthreads();
    const bool use_gamma = (s_scal[1].x != 0.0 || s_scal[1].y != 0.0);
    const bool use_beta = (s_scal[2].x != 0.0 || s_scal[2].y != 0.0);
    const double v0 = TWO ? vdict[0] : 0.0, v1 = TWO ? vdict[1] : 0.0;
    const uint32_t cmask = (1u << cbits) - 1u;
    const uint64_t pol_s = pol_evict_first(), pol_x = pol_evict_last();
    const int lane = threadIdx.x & 31;
    double d[3] = {0.0, 0.0, 0.0};

    // item `it` of this warp; the metadata of the next item and the slice of the one after are requested one item ahead
    const int stride = (int)gridDim.x * kXWarps;           // (slice counts are < 2^31: rows < 2^31 by the int32 columns)
    const int nsl = (int)nslices;
    int it = (int)blockIdx.x * kXWarps + (int)(threadIdx.x >> 5);
    auto slice_of = [&](int i) -> int { return i < nsl ? order[i] : 0; };
    int s = slice_of(it);
    uint32_t info = it < nsl ? rowinfo[(int64_t)s * 32 + lane] : 0u;
    int64_t base = it < nsl ? rowptr[(int64_t)s * 32] : 0;
    int s_next = slice_of(it + stride);

#pragma unroll 1
    for (; it < nsl; it += stride) {
        const bool more = it + stride < nsl;
        const uint32_t info_n = more ? rowinfo[(int64_t)s_next * 32 + lane] : 0u;
        const int64_t base_n = more ? rowptr[(int64_t)s_next * 32] : 0;
        const int s_after = slice_of(it + 2 * stride);

        const int len = (int)(info & kLenMaskB);
        const int maxlen = __shfl_sync(0xffffffffu, len, 0);
        const int minlen = __shfl_sync(0xffffffffu, len, 31);
        const int64_t row = (int64_t)s * 32 + (info >> 24);
        const bool live = row < nrows && !(KEEP && !OUT && len == 0);      // padding ranks of the last slice point past the last row
        double zv = 0.0, xi = 0.0;
        int32_t rref = 0;
        if (live) {                                        // the epilogue's operands, requested before the entries
            if (use_beta) zv = z[row];
            if (use_gamma || DOTS) xi = x[row_lo + row];
            if constexpr (OUT) rref = perm_inv[row_lo + row];
        }
        double acc0 = 0.0, acc1 = 0.0;
        const int32_t *wb = words + base + lane;
        // diagonals [k, k + kXTrip): a uniform trip has the first `rem` of them on every lane at 32 (k + u) + lane; a ragged
        // one has diagonal k + u where k + u < len, at the entries of the slice before it (`off`, counted by ballots) + lane
        auto trip = [&](auto ragged, int k, int rem, int &off) {
            constexpr bool RG = decltype(ragged)::value;
            uint32_t w[kXTrip];                            // (set on every path: a value left over from the previous trip
#pragma unroll                                         //  would stay live across it)
            for (int u = 0; u < kXTrip; u++) {
                bool a;
                int o;
                if constexpr (RG) { a = k + u < len; o = off; off += __popc(__ballot_sync(0xffffffffu, a)); }
                else { a = u < rem; o = (k + u) * 32; }
                w[u] = a ? (uint32_t)lds_i32(wb + o, pol_s) : 0u;
            }
            double xv[kXTrip];
            uint32_t codes = 0;
#pragma unroll
            for (int u = 0; u < kXTrip; u++) {
                xv[u] = 0.0;
                if (RG ? k + u < len : u < rem) {
                    xv[u] = ldx_hint(x + (w[u] & cmask), pol_x);
                    if (TWO) codes |= (w[u] >> cbits) << u;
                }
            }
#pragma unroll
            for (int u = 0; u < kXTrip; u++) {
                if (RG ? k + u < len : u < rem) {
                    const double v = TWO ? (((codes >> u) & 1u) ? v1 : v0) : sdict[w[u] >> cbits];
                    if (u & 1) mac(acc1, v, xv[u]); else mac(acc0, v, xv[u]);
                }
            }
        };
        int off = 0;
        if (maxlen == minlen) {
#pragma unroll 1
            for (int k = 0; k < len; k += kXTrip) trip(std::false_type{}, k, min(kXTrip, len - k), off);
        } else {
#pragma unroll 1
            for (int k = 0; k < maxlen; k += kXTrip) trip(std::true_type{}, k, 0, off);
        }
        if (live) {
            const double acc = VT::add(acc0, acc1);
            double out = VT::scale(s_scal[0], acc);
            if (use_gamma) out = VT::add(out, VT::scale(s_scal[1], xi));
            if (use_beta) out = VT::add(out, VT::scale(s_scal[2], zv));
            if constexpr (OUT) y_ref[rref] = make_double2(out_alpha.x * out, out_alpha.y * out);
            else y[row] = out;
            if (DOTS) {
                const double2 p = VT::conj_mul(xi, out);
                d[0] += p.x; d[1] += p.y; d[2] += VT::abs2(out);
            }
        }
        s = s_next; info = info_n; base = base_n; s_next = s_after;
    }
    if (DOTS) {
        d[0] *= s_scal[3].x; d[1] *= s_scal[3].x;
        block_reduce_finalize<3, kXWarps * 32>(d, partials, ticket, dots_out);
    }
}

template <bool DOTS, bool KEEP, bool OUT, bool TWO>
static int launch_cross_slices_cfg(const qbgpu_matrix *A, const FusedArgs &a)
{
    Context &c = ctx();
    auto kern = sjds_cross_slices_kernel<DOTS, KEEP, OUT, TWO>;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern, kXWarps * 32, 0));
        if (blocks_per_sm < 1) return fail(QBGPU_ERR_STATE, "slice-granular cross pass: no CTA fits on an SM");
        if (DOTS && blocks_per_sm > kXDotsBlocksPerSm) blocks_per_sm = kXDotsBlocksPerSm;
    }
    const int64_t nrows = A->nrows();
    if (nrows == 0) return QBGPU_OK;
    const int64_t nslices = (nrows + 31) / 32;
    const int64_t want = (nslices + kXWarps - 1) / kXWarps;
    int64_t cap = (int64_t)c.num_sms * blocks_per_sm;
    if (cap > kMaxPartialBlocks) cap = kMaxPartialBlocks;
    const int grid = (int)(want < cap ? want : cap);
    kern<<<grid, kXWarps * 32, 0, c.stream>>>(nslices, nrows, A->row_lo, A->rowptr, A->rowinfo, A->col, (const double *)a.x,
                                              (const double *)a.z, (double *)a.y, a.alpha, a.gamma, a.beta, a.scal_mode, a.sc,
                                              a.dots, c.partials, c.ticket, A->vdict, A->slice_order, A->cbits,
                                              OUT ? a.perm_inv : nullptr, OUT ? (double2 *)a.y_ref : nullptr, a.out_alpha);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

template <bool TWO>
static int launch_cross_slices_typed(const qbgpu_matrix *A, const FusedArgs &a)
{
    const bool dots = a.dots != nullptr;
    const bool keep = !dots && a.scal_mode == 0 && a.z == a.y && a.beta.x == 1.0 && a.beta.y == 0.0 && a.gamma.x == 0.0 && a.gamma.y == 0.0;
    if (a.y_ref) {                                          // the closing pass of a species product writes the reference's order
        if (keep && a.perm_inv) return launch_cross_slices_cfg<false, true, true, TWO>(A, a);
        return fail(QBGPU_ERR_STATE, "fused way out: not the closing pass of a species handle (internal)");
    }
    if (keep) return launch_cross_slices_cfg<false, true, false, TWO>(A, a);
    return dots ? launch_cross_slices_cfg<true, false, false, TWO>(A, a) : launch_cross_slices_cfg<false, false, false, TWO>(A, a);
}

// entry: tile-ordered sliced-jagged handle (slice_order set), not a ring view.  The bulk copies may read up to 15 bytes
// before/after a slice's range inside col[] / val[]: always inside the arrays except at their very ends, where the
// allocations keep 64 bytes of slack.  Packed parts with fp64 vectors take the slice-granular kernel (3).
int launch_spmv_sjds_bulk(const qbgpu_matrix *A, const FusedArgs &a)
{
    if (A->cbits && !A->api_complex) return A->ndict == 2 ? launch_cross_slices_typed<true>(A, a) : launch_cross_slices_typed<false>(A, a);
    if (A->cbits) return launch_bulk_typed<uint32_t, double2>(A, a);
    if (A->ndict) return fail(QBGPU_ERR_STATE, "bulk-streamed product: 1-byte dictionary codes are not supported (internal)");
    if (!A->api_complex) return launch_bulk_typed<double, double>(A, a);
    if (A->val_real) return launch_bulk_typed<double, double2>(A, a);
    return launch_bulk_typed<double2, double2>(A, a);
}

// ------------------------------------------------------------------------------- (2) block-local product, x in smem
// Rows [u*D - row_lo, (u+1)*D - row_lo) of the handle reference only columns [u*D, (u+1)*D).  One CTA per block u (persistent,
// blocks handed out round-robin); slices that straddle two blocks are visited by both CTAs, each handling its own rows.
template <typename ValT, typename VecT, int NT, int U, int MINB>
__global__ void __launch_bounds__(NT, MINB)
sjds_block_smem_kernel(int64_t nrows, int64_t row_lo, int64_t D, int64_t u_lo, int64_t u_cnt, const int64_t *__restrict__ rowptr,
                       const uint32_t *__restrict__ rowinfo, const int32_t *__restrict__ col, const ValT *__restrict__ val,
                       const VecT *__restrict__ x, const VecT *z, VecT *y, double2 alpha, double2 gamma, double2 beta,
                       int scal_mode, const double *__restrict__ sc, const double *__restrict__ vdict, int cbits, int use_bulk,
                       int64_t P, int64_t EP)
{
    using VT = VecTraits<VecT>;
    constexpr bool kPacked = std::is_same<ValT, uint32_t>::value;     // packed words col | code << cbits, no val array
    static_assert(kPacked || sizeof(ValT) >= 8, "values are fp64, complex, or packed codes");
    using ArithT = typename std::conditional<kPacked, double, ValT>::type;
    constexpr int NWARP = NT / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ double sdict[kPacked ? kPackedMaxTable : 1];
    __shared__ __align__(8) unsigned long long xbar_storage;
    VecT *xs = (VecT *)smem_raw;
    const uint32_t xbar = smem_u32(&xbar_storage);
    const uint32_t cmask = kPacked ? (1u << cbits) - 1u : ~0u;
    if (kPacked) { for (int i = threadIdx.x; i < (int)kPackedMaxTable; i += NT) sdict[i] = vdict[i]; }
    if (threadIdx.x == 0) { mbar_init(xbar, 1); mbar_fence_init(); }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t pol_s = pol_evict_first();
    if (scal_mode != 0) {
        const double sx = sc[0], sz = sc[1], bprev = sc[2];
        alpha = make_double2(sx, 0.0);
        gamma = make_double2(0.0, 0.0);
        beta = scal_mode == 1 ? make_double2(-bprev * sz, 0.0) : make_double2(1.0, 0.0);
    }
    const bool use_gamma = (gamma.x != 0.0 || gamma.y != 0.0);
    const bool use_beta = (beta.x != 0.0 || beta.y != 0.0);
    uint32_t xphase = 0;

    // the rowinfo / rowptr of a warp's NEXT slice are requested one slice ahead (also across the block switch), so the
    // dependent chain of a slice is only: column/value loads -> shared-memory gathers
    auto first_slice = [&](int64_t ub) -> int64_t { return (((u_lo + ub) * D - row_lo) >> 5) + warp; };
    auto last_slice = [&](int64_t ub) -> int64_t { return ((u_lo + ub + 1) * D - row_lo - 1) >> 5; };
    uint32_t info_n = 0;
    int64_t base_n = 0, pref_s = -1;                        // pref_s: the slice info_n / base_n belong to
    // periodic row metadata (qbgpu_matrix::period_slices): FULL slices read the entries of the first period, which stay in L2
    // (0.8 MB on BASELINE config 3) instead of streaming 0.8 GB of rowinfo / rowptr per product; the last, partial slice is its own
    const int64_t nfull = P > 0 ? (nrows >> 5) : 0;
    auto ld_info = [&](int64_t s) -> uint32_t { const int64_t q = (P > 0 && s < nfull) ? s % P : s; return rowinfo[q * 32 + lane]; };
    auto ld_base = [&](int64_t s) -> int64_t {
        if (P > 0 && s < nfull) { const int64_t k = s / P; return rowptr[(s - k * P) * 32] + k * EP; }
        return rowptr[s * 32];
    };

    for (int64_t ub = blockIdx.x; ub < u_cnt; ub += gridDim.x) {
        const int64_t c0 = (u_lo + ub) * D;                 // first column (= first global row) of the block
        const int64_t r0 = c0 - row_lo, r1 = r0 + D;        // local rows of the block
        __syncthreads();                                    // every warp has finished reading the previous block from xs
        bool x_ready = true;
        if (use_bulk) {
            if (threadIdx.x == 0) {
                fence_proxy_async_smem();
                const uint32_t bytes = (uint32_t)(D * (int64_t)sizeof(VecT));
                mbar_expect_tx(xbar, bytes);
                bulk_g2s_plain(smem_u32(xs), x + c0, bytes, xbar);
            }
            x_ready = false;
        } else {
            for (int64_t j = threadIdx.x; j < D; j += NT) xs[j] = x[c0 + j];
            __syncthreads();
        }
        const int64_t s_last = last_slice(ub);
        for (int64_t s = first_slice(ub); s <= s_last; s += NWARP) {
            if (pref_s != s) { info_n = ld_info(s); base_n = ld_base(s); }                      // (first slice of the kernel, or a skipped block)
            const uint32_t info = info_n;
            const int64_t base = base_n;
            {   // request the next slice of this warp: in this block, or the first one of its next block
                int64_t sn = s + NWARP;
                bool have = sn <= s_last;
                if (!have && ub + gridDim.x < u_cnt) { sn = first_slice(ub + gridDim.x); have = sn <= last_slice(ub + gridDim.x); }
                if (have) { info_n = ld_info(sn); base_n = ld_base(sn); pref_s = sn; }
            }
            const int len = (int)(info & kLenMaskB);
            const int64_t row = s * 32 + (info >> 24);
            const bool mine = row >= r0 && row < r1;        // (row < nrows follows: r1 <= nrows)
            const int maxlen = __shfl_sync(0xffffffffu, len, 0);
            const int minlen = __shfl_sync(0xffffffffu, len, 31);
            const int32_t *cb = col + base + lane;
            const ValT *vb = val + base + lane;
            VecT zv = VT::zero();
            if (mine && use_beta) zv = z[row];              // requested now, used after the last trip
            VecT acc0 = VT::zero(), acc1 = VT::zero();
            int k = 0;
            // trips in which every lane has all U diagonals (the shortest row, rank 31, reaches k + U): entry (u, lane) of
            // the trip sits at (k + u)*32 + lane -- no votes, no predicates
            for (; k + U <= minlen; k += U) {
                int c[U];
                ValT v[U];
#pragma unroll
                for (int u = 0; u < U; u++) c[u] = lds_i32(cb + (k + u) * 32, pol_s);
                if constexpr (!kPacked) {
#pragma unroll
                    for (int u = 0; u < U; u++) v[u] = lds_val(vb + (k + u) * 32, pol_s);
                }
                if (!x_ready) { mbar_wait(xbar, xphase); xphase ^= 1u; x_ready = true; }
                if (mine) {
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        const VecT xv = xs[(int)((int64_t)(int32_t)((uint32_t)c[u] & cmask) - c0)];
                        ArithT w;
                        if constexpr (kPacked) w = sdict[(uint32_t)c[u] >> cbits]; else w = v[u];
                        if (u & 1) mac(acc1, w, xv); else mac(acc0, w, xv);      // U is even: diagonal k + u -> accumulator u & 1
                    }
                }
            }
            int off = k * 32;                               // entries of the slice before diagonal k (all rows were full so far)
            for (; k < maxlen; k += U) {                    // ragged trips
                unsigned am = 0;
                int c[U];
                ValT v[U];
                int o[U];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const bool a = k + u < len;
                    am |= (a ? 1u : 0u) << u;
                    o[u] = off;
                    off += __popc(__ballot_sync(0xffffffffu, a));
                }
#pragma unroll
                for (int u = 0; u < U; u++) if ((am >> u) & 1u) { c[u] = lds_i32(cb + o[u], pol_s); if constexpr (!kPacked) v[u] = lds_val(vb + o[u], pol_s); }
                if (!x_ready) { mbar_wait(xbar, xphase); xphase ^= 1u; x_ready = true; }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    if (((am >> u) & 1u) && mine) {
                        const VecT xv = xs[(int)((int64_t)(int32_t)((uint32_t)c[u] & cmask) - c0)];
                        ArithT w;
                        if constexpr (kPacked) w = sdict[(uint32_t)c[u] >> cbits]; else w = v[u];
                        if (u & 1) mac(acc1, w, xv); else mac(acc0, w, xv);
                    }
                }
            }
            if (!x_ready) { mbar_wait(xbar, xphase); xphase ^= 1u; x_ready = true; }      // (a warp whose slices are all empty)
            if (mine) {
                const VecT acc = VT::add(acc0, acc1);
                VecT out = VT::scale(alpha, acc);
                if (use_gamma) out = VT::add(out, VT::scale(gamma, xs[row - r0]));
                if (use_beta) out = VT::add(out, VT::scale(beta, zv));
                y[row] = out;
            }
        }
        if (!x_ready) { mbar_wait(xbar, xphase); xphase ^= 1u; }                           // (a warp without any slice in this block)
    }
}

template <typename ValT, typename VecT, int NT, int U, int MINB>
static int launch_block_smem_cfg(const qbgpu_matrix *A, const FusedArgs &a, int64_t D)
{
    Context &c = ctx();
    auto kern = sjds_block_smem_kernel<ValT, VecT, NT, U, MINB>;
    const size_t smem = ((size_t)D * sizeof(VecT) + 127) / 128 * 128;
    static size_t smem_set = 0;
    if (smem_set < smem) { QB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); smem_set = smem; }
    static int bps = 0;
    static size_t bps_smem = 0;
    if (bps == 0 || bps_smem != smem) {                     // (per instantiation; the block size of a handle never changes)
        QB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, NT, smem));
        bps_smem = smem;
    }
    if (bps < 1) return fail(QBGPU_ERR_STATE, "block-local product: the block does not fit in shared memory");
    const int64_t u_lo = A->row_lo / D, u_cnt = A->nrows() / D;
    if (u_cnt == 0) return QBGPU_OK;
    const int64_t cap = (int64_t)c.num_sms * bps;
    const int grid = (int)(u_cnt < cap ? u_cnt : cap);
    // cp.async.bulk needs a 16-byte-aligned source: every block of x starts at x + u*D, so D*sizeof(VecT) and x itself must be
    // multiples of 16 (an fp64 x passed to the internal-order entry points may be only 8-byte aligned, e.g. a window of a
    // larger vector); otherwise the threads copy the block
    const int use_bulk = ((D * (int64_t)sizeof(VecT)) % 16 == 0 && D * (int64_t)sizeof(VecT) < (1 << 20) && ((uintptr_t)a.x & 15) == 0) ? 1 : 0;
    kern<<<grid, NT, smem, c.stream>>>(A->nrows(), A->row_lo, D, u_lo, u_cnt, A->rowptr, A->rowinfo, A->col, (const ValT *)A->val,
                                       (const VecT *)a.x, (const VecT *)a.z, (VecT *)a.y, a.alpha, a.gamma, a.beta, a.scal_mode, a.sc,
                                       A->vdict, A->cbits, use_bulk, A->period_slices, A->period_entries);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

// Can the block-local kernel serve this handle?  (sliced-jagged layout, rows = whole blocks of D, block fits in shared memory)
// Blocks up to 112 KB (two CTAs per SM, or one with half of the SRAM left as L1: the matrix stream is register-fed and its
// loads in flight are tracked in L1 lines).  A 206 KB block (BASELINE config 3 with complex vectors) leaves 28 KB of L1 and
// the stream then stalls at 3.2 TB/s (profiles/r02_ncu_species_stored_first_bulk_kernels_hubbard4x4.csv): 13.6 ms against
// 10.1 ms for the plain kernel, so such blocks take the plain kernel.
bool block_smem_applicable(const qbgpu_matrix *A, int64_t D)
{
    constexpr size_t kMaxBlockBytes = 112 * 1024;
    if (A->format != QBGPU_FORMAT_SELL || D <= 0 || A->row_lo % D != 0 || A->nrows() % D != 0) return false;
    return (size_t)D * A->vec_bytes() <= kMaxBlockBytes;
}

int launch_spmv_block_smem(const qbgpu_matrix *A, const FusedArgs &a, int64_t D)
{
    if (a.dots) return fail(QBGPU_ERR_ARG, "block-local product: the running dots belong to the closing pass");
    // packed words: a third of the bytes per entry, and a trip takes 8 diagonals instead of 4.  Diagonal k still accumulates
    // into k & 1, so the products stay bit-identical.  On BASELINE config 3 (fp64 vectors, one B200 at 1000 W) the pass no
    // longer follows the bytes in flight: 8 and 10 diagonals per trip measured 5.57 and 5.67 ms (12 spill at 64 registers a
    // thread).  Complex vectors take 6 (10 spill).
    if (A->cbits) return A->api_complex ? launch_block_smem_cfg<uint32_t, double2, 1024, 6, 1>(A, a, D) : launch_block_smem_cfg<uint32_t, double, 1024, 8, 1>(A, a, D);
    if (A->ndict) return fail(QBGPU_ERR_STATE, "block-local product: 1-byte dictionary codes are not supported (internal)");
    if (!A->api_complex) return launch_block_smem_cfg<double, double, 1024, 4, 1>(A, a, D);
    if (A->val_real) return launch_block_smem_cfg<double, double2, 1024, 4, 1>(A, a, D);
    return launch_block_smem_cfg<double2, double2, 1024, 4, 1>(A, a, D);
}

}  // namespace qb
