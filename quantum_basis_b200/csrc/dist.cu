// quantum_basis_b200/csrc/dist.cu -- the multi-GPU Krylov drivers behind the C ABI: one process per GPU, no MPI/NCCL inside.
//
// The reference is one C++ process (model<T>::locate_E0_lanczos, src/model.cc:1124-1316) and has no distributed mode; SURVEY
// section 8(e) asks for row shards with the Krylov vector exchanged over NVLink and the Lanczos / CG / KPM scalars reduced
// across the GPUs.  Everything a rank needs from its peers travels through PEER MEMORY (CUDA IPC mappings over NVLink /
// NVSwitch), so a C or C++ host can drive the eight GPUs of a box with nothing but this library and any way of its own to
// hand 64-byte handles around (files, pipes, MPI, torch.distributed -- INTEGRATION.md):
//
//   * vectors: every rank owns ONE allocation holding two full-length vector buffers X[0], X[1] (ping-pong; its own rows
//     are the authoritative slice), a scalar mailbox and a flag array.  Before a product the slices of the peers are PULLED
//     by copy engines (peer.cu) while the part of the product that needs no remote data runs (the "local" part of a
//     species-order shard, species.cu); the rest follows the arrival.
//   * scalars: dist_allreduce_kernel -- every rank PUSHES its partial sums into each peer's mailbox with plain stores over
//     NVLink, fences, raises an epoch flag in the peer's memory, waits for the flags of all peers in its own memory and adds
//     the mailbox in rank order: a deterministic all-reduce (every rank gets bit-identical sums, so all of them take the
//     same stop-rule decision) that is also the barrier which makes the freshly written slices visible.  One 32-thread
//     kernel, a few microseconds; no host involvement, no collective library.
//
// Loops: lanczos (reference src/lanczos.cc:134-266, purposes sr_val0 / dnmcs / sr_val1, with the stop rule of :228-248
// evaluated on every rank from the identical reduced (a, b); sr_val1 re-orthogonalises against phi0 on the device, see
// dist_lanczos_loop), eigenvec_CG (:281-341), energy_scale (src/kpm.cc:45-88), Chebyshev moments, the plain product, and the
// four stages of model<T>::locate_E0_lanczos (src/model.cc:1124-1316: E0, phi0, E1, phi1) in one call.  The local arithmetic
// is the single-GPU kernels'; only the reductions differ (a sum of per-rank sums), so E0 agrees with the single-GPU run to
// round-off of the reductions (~1e-15 relative).
#include "internal.hpp"
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace qb {

constexpr int kMaxRanks = 16;
constexpr int kMailDoubles = 8;           // doubles per all-reduce call
constexpr double kLanczosPrecisionD = 2e-12;

// smallest eigenvalue / full QL of the tridiagonal (krylov.cu)
double tridiag_smallest(const double *hess, int64_t maxit, int64_t m);
int hess_eigen_host(const double *hess, int64_t maxit, int64_t m, double *ritz, double *s, double *s_last0);

struct DistPeers { char *base[kMaxRanks]; };

}  // namespace qb

struct qbgpu_dist {
    int rank = 0, world = 1;
    int64_t n = 0;
    std::vector<int64_t> bounds;
    bool cplx = true;
    size_t esize = 16;
    char *base = nullptr;                 // own allocation: X[0] | X[1] | mailbox | flags
    size_t off_x[2] = {0, 0}, off_mail = 0, off_flags = 0, total = 0;
    qb::DistPeers peers{};                // peers.base[rank] == base
    bool connected = false;
    unsigned epoch = 0;
    int *timeout_flag = nullptr;          // device: a waiter gave up
    double *scal = nullptr;               // device scratch (64 doubles)
    // optional refinement of a shard (qbgpu_dist_set_parts): parts that need no remote data run while the slices travel
    // (`early`: the local part, and the cross entries whose columns lie in the rank's own rows), the others after the arrival
    std::vector<qbgpu_matrix_t> early, late;
    // optional pull plan (qbgpu_dist_set_pull_plan): only these row ranges of the peers' slices are fetched
    struct Seg { int owner; int64_t first, rows; };
    std::vector<Seg> plan;
    bool has_plan = false;
    int lanes = 1;
    // optional wait points (qbgpu_dist_set_wait_points): late part j starts once the first wait_after[j] plan segments arrived
    std::vector<int> wait_after;
    cudaEvent_t wait_ev[8] = {};
    bool row_views = false;               // some part covers only a sub-range of the rank's rows: dots are taken in a pass of their own
    int64_t lo() const { return bounds[rank]; }
    int64_t hi() const { return bounds[rank + 1]; }
    int64_t nloc() const { return hi() - lo(); }
    void *X(int b) const { return base + off_x[b]; }
    void *own(int b) const { return base + off_x[b] + esize * (size_t)lo(); }
};

namespace qb {

__device__ __forceinline__ unsigned ld_acquire_sys_u32(const unsigned *p)
{ unsigned v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void st_release_sys_u32(unsigned *p, unsigned v)
{ asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ void st_relaxed_sys_f64(double *p, double v)
{ asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory"); }
__device__ __forceinline__ double ld_relaxed_sys_f64(const double *p)
{ double v; asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory"); return v; }

// vals[0..count) <- sum over ranks, in rank order; count == 0: a barrier.  mailbox layout in EVERY rank's memory:
// mail[slot = epoch & 1][writer rank][kMailDoubles]; flags[writer rank] = last epoch that writer has published here.
__global__ void __launch_bounds__(32) dist_allreduce_kernel(DistPeers P, int rank, int world, size_t off_mail, size_t off_flags,
                                                            unsigned epoch, double *vals, int count, int *timeout_flag)
{
    const int t = threadIdx.x;
    const unsigned slot = epoch & 1u;
    if (t < world) {                                        // push my partials into rank t's mailbox, then raise my flag there
        double *dst = (double *)(P.base[t] + off_mail) + ((size_t)slot * kMaxRanks + rank) * kMailDoubles;
        for (int i = 0; i < count; i++) st_relaxed_sys_f64(dst + i, vals[i]);
        __threadfence_system();
        st_release_sys_u32((unsigned *)(P.base[t] + off_flags) + rank, epoch);
    }
    __syncwarp();
    if (t < world) {                                        // wait for writer t's flag in MY memory
        const unsigned *f = (const unsigned *)(P.base[rank] + off_flags) + t;
        long long spins = 0;
        while ((int)(ld_acquire_sys_u32(f) - epoch) < 0) {
            if (++spins > (1LL << 24)) { *timeout_flag = 1; break; }      // seconds: never hang the device
            __nanosleep(64);
        }
    }
    __syncwarp();
    __threadfence_system();
    if (t < count) {
        const double *mail = (const double *)(P.base[rank] + off_mail) + (size_t)slot * kMaxRanks * kMailDoubles;
        double s = 0.0;
        for (int p = 0; p < world; p++) s += ld_relaxed_sys_f64(mail + (size_t)p * kMailDoubles + t);
        vals[t] = s;
    }
}

static int dist_allreduce(qbgpu_dist *D, double *dev, int count)
{
    if (count < 0 || count > kMailDoubles) return fail(QBGPU_ERR_ARG, "dist_allreduce: at most 8 doubles per call");
    if (D->world == 1) return QBGPU_OK;
    if (!D->connected) return fail(QBGPU_ERR_STATE, "dist: not connected (qbgpu_dist_connect)");
    Context &c = ctx();
    D->epoch++;
    dist_allreduce_kernel<<<1, 32, 0, c.stream>>>(D->peers, D->rank, D->world, D->off_mail, D->off_flags, D->epoch, dev, count, D->timeout_flag);
    QB_LAUNCH_COUNT();
    QB_CUDA(cudaGetLastError());
    return QBGPU_OK;
}

static int dist_allreduce_array(qbgpu_dist *D, double *dev, int64_t count)
{
    for (int64_t o = 0; o < count; o += kMailDoubles) QB_TRY(dist_allreduce(D, dev + o, (int)std::min<int64_t>(kMailDoubles, count - o)));
    return QBGPU_OK;
}

// pulls of the peers' slices of X[b] -- all of them, or the row ranges of the pull plan -- in ring order (at distance d every
// GPU serves one reader); `lanes` copy streams (pulls on one lane run back to back).  The pulls are ordered after the point of
// the compute stream marked by dist_pull_mark(): the caller marks, launches what needs no remote data, and only then spends
// the host time of enqueueing the transfers.
static int dist_pull_mark(qbgpu_dist *D) { return D->world > 1 ? peer_mark_fence() : QBGPU_OK; }
static int dist_pull(qbgpu_dist *D, int b)
{
    if (D->has_plan) {
        const bool wp = !D->wait_after.empty();            // wait points: everything on lane 0, which completes in order
        int k = 0;
        auto mark = [&](int done) -> int {
            for (size_t j = 0; j < D->wait_after.size(); j++) if (D->wait_after[j] == done) QB_TRY(peer_record_on_lane(0, D->wait_ev[j]));
            return QBGPU_OK;
        };
        if (wp) QB_TRY(mark(0));
        for (const auto &sg : D->plan) {
            const size_t off = D->off_x[b] + D->esize * (size_t)sg.first;
            const size_t nb = D->esize * (size_t)sg.rows;
            if (nb) QB_TRY(peer_pull_fenced(wp ? 0 : sg.owner % D->lanes, sg.owner, D->base + off, D->peers.base[sg.owner] + off, nb));   // one lane per owner: its last event covers all its segments
            k++;
            if (wp) QB_TRY(mark(k));
        }
        return QBGPU_OK;
    }
    for (int d = 1; d < D->world; d++) {
        const int p = (D->rank + d) % D->world;
        const size_t off = D->off_x[b] + D->esize * (size_t)D->bounds[p];
        const size_t nb = D->esize * (size_t)(D->bounds[p + 1] - D->bounds[p]);
        if (nb) QB_TRY(peer_pull_fenced(p % D->lanes, p, D->base + off, D->peers.base[p] + off, nb));
    }
    return QBGPU_OK;
}
// order the compute stream behind every pull: the LAST pull recorded per owner slot (a slot's event is re-recorded by
// every pull from that owner, and pulls on one lane complete in order; with several lanes every owner's last event is waited for)
static int dist_wait(qbgpu_dist *D)
{
    bool seen[kMaxRanks] = {};
    if (D->has_plan) { for (const auto &sg : D->plan) if (sg.rows) seen[sg.owner] = true; }
    else for (int p = 0; p < D->world; p++) seen[p] = p != D->rank && D->bounds[p + 1] > D->bounds[p];
    for (int d = 1; d < D->world; d++) {
        const int p = (D->rank + d) % D->world;
        if (seen[p]) QB_TRY(qbgpu_peer_wait(p));
    }
    return QBGPU_OK;
}

// y_local = alpha*(H x)_local + gamma*x_local + beta*z_local (+ partial dots) with x = X[b], whose slices are final on every
// rank (the caller's previous all-reduce was the barrier).  local_part may be null (an ordinary row shard: one product
// after the arrival); with a species shard the local part opens the product while the slices travel.
static void dist_sequence(qbgpu_dist *D, const qbgpu_matrix *local_part, const qbgpu_matrix *rest, std::vector<const qbgpu_matrix *> &seq, size_t &n_early)
{
    seq.clear(); n_early = 0;
    if (!D->early.empty() || !D->late.empty()) {
        for (auto h : D->early) seq.push_back(h);
        n_early = seq.size();
        for (auto h : D->late) seq.push_back(h);
    } else {
        if (local_part) { seq.push_back(local_part); n_early = 1; }
        seq.push_back(rest);
    }
}

// y / z pointer of a part: a row view addresses the rows it covers
static inline void *part_rows(const qbgpu_dist *D, const qbgpu_matrix *P, void *base)
{ return base ? (char *)base + D->esize * (size_t)(P->row_lo - D->lo()) : nullptr; }

// order the compute stream behind the arrival of what late part j needs
static int dist_wait_for_late(qbgpu_dist *D, size_t j, bool &waited_all)
{
    if (!D->wait_after.empty() && j < D->wait_after.size()) {
        if (D->wait_after[j] > 0 || true) QB_CUDA(cudaStreamWaitEvent(ctx().stream, D->wait_ev[j], 0));
        return QBGPU_OK;
    }
    if (!waited_all) { QB_TRY(dist_wait(D)); waited_all = true; }
    return QBGPU_OK;
}

// pulls_issued: the caller has already enqueued the pulls of X[b] (the Lanczos loop does, one step ahead)
static int dist_product(qbgpu_dist *D, const qbgpu_matrix *local_part, const qbgpu_matrix *rest, int b, const FusedArgs &args, bool pulls_issued = false)
{
    if (!pulls_issued) QB_TRY(dist_pull_mark(D));
    FusedArgs a = args;
    a.x = D->X(b);
    // the parts in execution order: [early ...] wait [late ...]; the first opens the product (alpha, gamma, beta*z), the
    // others accumulate into the same y, the last carries the running dots (or, with row views, a pass of its own does)
    std::vector<const qbgpu_matrix *> seq;
    size_t n_early = 0;
    dist_sequence(D, local_part, rest, seq, n_early);
    const bool sep_dots = D->row_views && a.dots;
    bool pulled = pulls_issued, waited = false;
    for (size_t i = 0; i < seq.size(); i++) {
        if (i >= n_early) {
            if (!pulled) { QB_TRY(dist_pull(D, b)); pulled = true; }
            QB_TRY(dist_wait_for_late(D, i - n_early, waited));
        }
        const bool first = i == 0, last = i + 1 == seq.size();
        FusedArgs ai;
        if (first) { ai = a; }
        else {
            ai.x = a.x; ai.y = a.y; ai.z = a.y;
            ai.beta = make_double2(1.0, 0.0);
            if (a.scal_mode != 0) { ai.scal_mode = 2; ai.sc = a.sc; } else ai.alpha = a.alpha;
        }
        ai.y = part_rows(D, seq[i], ai.y);
        ai.z = part_rows(D, seq[i], const_cast<void *>(ai.z));
        ai.dots = (last && !sep_dots) ? a.dots : nullptr;
        QB_TRY(launch_spmv(seq[i], ai));
        if (i + 1 == n_early && !pulled) { QB_TRY(dist_pull(D, b)); pulled = true; }      // enqueue the transfers while the early parts run
    }
    if (!pulled) QB_TRY(dist_pull(D, b));
    if (!waited) QB_TRY(dist_wait(D));
    if (sep_dots) {                                         // dots[0..1] = <x_own, y>, dots[2] = |y|^2 over the rank's rows
        const int64_t nl = D->nloc();
        if (nl) { QB_TRY(vec_dotc(nl, D->cplx, D->own(b), a.y, a.dots)); QB_TRY(vec_nrm2sq(nl, D->cplx, a.y, a.dots + 2)); }
        else QB_CUDA(cudaMemsetAsync(a.dots, 0, sizeof(double) * 3, ctx().stream));
    }
    return QBGPU_OK;
}

// Lanczos step a over the same sequence of parts (first: w = sx*H*ux - b*sz*uz; others accumulate; last: the partial <v, w>).
// `w`: where the product goes -- uz itself (in place) or a scratch vector of the rank's rows.  With a scratch vector the EARLY
// parts (they need no remote data) can be launched before the host knows whether there is a next step: a step that does not
// happen leaves the exchange buffers untouched.  phase 0: the whole step; 1: only the early parts (no pulls, no waits);
// 2: the rest of a step whose early parts and pulls have been issued.
static int dist_lanczos_step_a(qbgpu_dist *D, const qbgpu_matrix *local_part, const qbgpu_matrix *rest, int bx, void *uz, void *w, double *state,
                               bool pulls_issued, int phase = 0)
{
    if (!pulls_issued && phase != 1) QB_TRY(dist_pull_mark(D));
    std::vector<const qbgpu_matrix *> seq;
    size_t n_early = 0;
    dist_sequence(D, local_part, rest, seq, n_early);
    void *w_out = (w && w != uz) ? w : nullptr;
    bool pulled = pulls_issued, waited = false;
    for (size_t i = (phase == 2 ? n_early : 0); i < (phase == 1 ? n_early : seq.size()); i++) {
        if (i >= n_early) {
            if (!pulled) { QB_TRY(dist_pull(D, bx)); pulled = true; }
            QB_TRY(dist_wait_for_late(D, i - n_early, waited));
        }
        const bool last = i + 1 == seq.size() && !D->row_views;
        QB_TRY(lanczos_step_a(seq[i], D->X(bx), part_rows(D, seq[i], uz), state, i == 0, last, w_out ? part_rows(D, seq[i], w_out) : nullptr));
        if (phase == 0 && i + 1 == n_early && !pulled) { QB_TRY(dist_pull(D, bx)); pulled = true; }
    }
    if (phase == 1) return QBGPU_OK;
    if (!pulled) QB_TRY(dist_pull(D, bx));
    if (!waited) QB_TRY(dist_wait(D));
    if (D->row_views) {                                     // state[3] = sx * Re <ux_own, w> over the rank's rows, in a pass of its own
        const int64_t nl = D->nloc();
        if (nl) QB_TRY(vec_dotc_scaled(nl, D->cplx, D->own(bx), w_out ? w_out : uz, state + 3, state + 0));
        else QB_CUDA(cudaMemsetAsync(state + 3, 0, sizeof(double), ctx().stream));
    }
    return QBGPU_OK;
}

static int dist_check(const qbgpu_dist *D, const qbgpu_matrix *local_part, const qbgpu_matrix *rest)
{
    if (!D || !rest) return fail(QBGPU_ERR_ARG, "dist: null argument");
    if (D->world > 1 && !D->connected) return fail(QBGPU_ERR_STATE, "dist: not connected (qbgpu_dist_connect)");
    if (rest->n != D->n || rest->row_lo != D->lo() || rest->row_hi != D->hi()) return fail(QBGPU_ERR_ARG, "dist: the shard does not cover this rank's rows");
    if (rest->api_complex != D->cplx) return fail(QBGPU_ERR_ARG, "dist: vector type of the handle and of the context differ");
    if (local_part && (local_part->row_lo != D->lo() || local_part->row_hi != D->hi() || local_part->api_complex != D->cplx))
        return fail(QBGPU_ERR_ARG, "dist: the local part does not match the shard");
    return QBGPU_OK;
}

static int dist_timed_out(qbgpu_dist *D, const char *what)
{
    int h = 0;
    QB_CUDA(cudaMemcpyAsync(&h, D->timeout_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx().stream));
    QB_CUDA(cudaStreamSynchronize(ctx().stream));
    if (h) return fail(QBGPU_ERR_STATE, std::string(what) + ": a rank waited in vain for its peers (all-reduce time-out)");
    return QBGPU_OK;
}

// slice [lo, hi) of the reference's vec_randomize sequence (src/miscellaneous.cc:371-388), unnormalised: element j of the
// reference's order, j = idx ? idx[k] : lo + k (idx: the reference's row of every local entry, for internal orders)
template <typename VecT>
__global__ void __launch_bounds__(256) dist_randomize_kernel(int64_t nloc, int64_t lo, const int32_t *__restrict__ idx, VecT *x, uint32_t seed)
{
    const uint64_t p = 2147483647ull;
    uint64_t s0 = seed % p;
    if (s0 == 0) s0 = 1;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nloc; k += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t j = idx ? (uint64_t)idx[k] : (uint64_t)(lo + k);
        uint64_t r = 1, base = 16807ull, e = j + 1;                        // s_j = seed * 16807^(j+1) mod p
        while (e) { if (e & 1) r = (r * base) % p; base = (base * base) % p; e >>= 1; }
        const uint64_t s = (s0 * r) % p;
        const double v = (double)s * (1.0 / 2147483647.0) - 0.5;
        if constexpr (sizeof(VecT) == 16) x[k] = make_double2(v, 0.0); else x[k] = v;
    }
}

// x <- (x - <phi0, x> phi0) / |x - <phi0, x> phi0| over the shards (x, phi0: this rank's rows): the cblas dot, axpy, nrm2 and
// scal of src/model.cc:1240-1252 and :1302-1311, each sum reduced across the ranks.  The caller passes a barrier before x is pulled.
static int dist_orthonormalize(qbgpu_dist *D, const void *phi0, void *x)
{
    Context &c = ctx();
    const int64_t nloc = D->nloc();
    double *t = D->scal + 32;                               // [0], [1] = <phi0, x>, [2] = |x|^2
    if (nloc) QB_TRY(vec_dotc(nloc, D->cplx, phi0, x, t)); else QB_CUDA(cudaMemsetAsync(t, 0, sizeof(double) * 2, c.stream));
    QB_TRY(dist_allreduce(D, t, 2));
    double h[2];
    QB_TRY(read_scalars(t, h, 2));
    if (nloc) QB_TRY(vec_axpy(nloc, D->cplx, make_double2(-h[0], D->cplx ? -h[1] : 0.0), phi0, x));
    if (nloc) QB_TRY(vec_nrm2sq(nloc, D->cplx, x, t + 2)); else QB_CUDA(cudaMemsetAsync(t + 2, 0, sizeof(double), c.stream));
    QB_TRY(dist_allreduce(D, t + 2, 1));
    double nn;
    QB_TRY(read_scalars(t + 2, &nn, 1));
    if (nloc) QB_TRY(vec_scal(nloc, D->cplx, make_double2(1.0 / sqrt(nn), 0.0), x));
    return QBGPU_OK;
}

}  // namespace qb

using namespace qb;

extern "C" {

int qbgpu_dist_create(qbgpu_dist_t *out, int rank, int world, int64_t n, const int64_t *bounds, int vec_complex)
{
    QB_TRY(ensure_init());
    if (!out || !bounds || world < 1 || world > kMaxRanks || rank < 0 || rank >= world || n <= 0) return fail(QBGPU_ERR_ARG, "dist_create: bad argument (1..16 ranks)");
    if (bounds[0] != 0 || bounds[world] != n) return fail(QBGPU_ERR_ARG, "dist_create: bounds must run from 0 to n");
    for (int p = 0; p < world; p++) if (bounds[p + 1] < bounds[p]) return fail(QBGPU_ERR_ARG, "dist_create: bounds must be non-decreasing");
    auto *D = new qbgpu_dist;
    D->rank = rank; D->world = world; D->n = n; D->bounds.assign(bounds, bounds + world + 1);
    D->cplx = vec_complex != 0; D->esize = D->cplx ? 16 : 8;
    const size_t vbytes = (D->esize * (size_t)n + 255) / 256 * 256;
    D->off_x[0] = 0; D->off_x[1] = vbytes;
    D->off_mail = 2 * vbytes;
    D->off_flags = D->off_mail + sizeof(double) * 2 * kMaxRanks * kMailDoubles;
    D->total = D->off_flags + 256;
    cudaError_t e = cudaMalloc(&D->base, D->total);
    if (e != cudaSuccess) { delete D; return cuda_fail(e, "cudaMalloc(dist buffers)", __FILE__, __LINE__); }
    QB_CUDA(cudaMemset(D->base, 0, D->total));
    QB_CUDA(cudaMalloc(&D->timeout_flag, sizeof(int)));
    QB_CUDA(cudaMemset(D->timeout_flag, 0, sizeof(int)));
    QB_CUDA(cudaMalloc(&D->scal, sizeof(double) * 64));
    QB_CUDA(cudaMemset(D->scal, 0, sizeof(double) * 64));
    for (int p = 0; p < kMaxRanks; p++) D->peers.base[p] = nullptr;
    D->peers.base[rank] = D->base;
    D->connected = world == 1;
    *out = D;
    return QBGPU_OK;
}

int qbgpu_dist_export(qbgpu_dist_t D, void *handle64)
{
    if (!D || !handle64) return fail(QBGPU_ERR_ARG, "null argument");
    return qbgpu_ipc_export(D->base, handle64);
}

int qbgpu_dist_connect(qbgpu_dist_t D, const void *handles)
{
    if (!D || !handles) return fail(QBGPU_ERR_ARG, "null argument");
    if (D->connected) return QBGPU_OK;
    for (int p = 0; p < D->world; p++) {
        if (p == D->rank) continue;
        void *ptr = nullptr;
        QB_TRY(qbgpu_ipc_open((const char *)handles + 64 * p, &ptr));
        D->peers.base[p] = (char *)ptr;
    }
    D->connected = true;
    return QBGPU_OK;
}

int qbgpu_dist_destroy(qbgpu_dist_t D)
{
    if (!D) return QBGPU_OK;
    cudaDeviceSynchronize();
    for (int p = 0; p < D->world; p++) if (p != D->rank && D->peers.base[p]) cudaIpcCloseMemHandle(D->peers.base[p]);
    cudaFree(D->base); cudaFree(D->timeout_flag); cudaFree(D->scal);
    for (auto &e : D->wait_ev) if (e) cudaEventDestroy(e);
    delete D;
    return QBGPU_OK;
}

/* Refine the shard: `early` parts need no remote data (the local part; the cross entries whose columns are the rank's own rows)
 * and run while the slices travel, `late` parts follow the arrival.  Together they must hold exactly the shard's entries (the
 * loops then ignore the decomposition passed per call).  n_early = n_late = 0 clears the refinement. */
int qbgpu_dist_set_parts(qbgpu_dist_t D, int n_early, const qbgpu_matrix_t *early, int n_late, const qbgpu_matrix_t *late)
{
    if (!D || n_early < 0 || n_late < 0 || (n_early && !early) || (n_late && !late)) return fail(QBGPU_ERR_ARG, "dist_set_parts: bad argument");
    D->early.clear(); D->late.clear();
    for (int i = 0; i < n_early + n_late; i++) {
        qbgpu_matrix_t h = i < n_early ? early[i] : late[i - n_early];
        if (!h || h->n != D->n || h->row_lo < D->lo() || h->row_hi > D->hi() || h->row_lo > h->row_hi || h->api_complex != D->cplx)
        { D->early.clear(); D->late.clear(); D->row_views = false; return fail(QBGPU_ERR_ARG, "dist_set_parts: a part does not match this rank's rows / vector type"); }
        if (i == 0 && (h->row_lo != D->lo() || h->row_hi != D->hi()))
        { D->early.clear(); D->late.clear(); D->row_views = false; return fail(QBGPU_ERR_ARG, "dist_set_parts: the first part opens the product and must cover all of the rank's rows"); }
        (i < n_early ? D->early : D->late).push_back(h);
    }
    D->row_views = false;
    for (auto h : D->early) D->row_views = D->row_views || h->row_lo != D->lo() || h->row_hi != D->hi();
    for (auto h : D->late) D->row_views = D->row_views || h->row_lo != D->lo() || h->row_hi != D->hi();
    D->wait_after.clear();
    return QBGPU_OK;
}

/* Fetch only these row ranges of the peers' slices (rows [first[k], first[k] + rows[k]) lie inside owner[k]'s rows): what the
 * late parts actually reference.  nseg = 0 with a null list restores "every slice, whole".  lanes: copy streams in use (1..8). */
int qbgpu_dist_set_pull_plan(qbgpu_dist_t D, int nseg, const int32_t *owner, const int64_t *first, const int64_t *rows, int lanes)
{
    if (!D || nseg < 0 || (nseg && (!owner || !first || !rows))) return fail(QBGPU_ERR_ARG, "dist_set_pull_plan: bad argument");
    D->plan.clear();
    D->has_plan = owner != nullptr;
    D->lanes = lanes < 1 ? 1 : (lanes > 8 ? 8 : lanes);
    for (int k = 0; k < nseg; k++) {
        const int p = owner[k];
        if (p < 0 || p >= D->world || p == D->rank || first[k] < D->bounds[p] || rows[k] < 0 || first[k] + rows[k] > D->bounds[p + 1])
        { D->plan.clear(); D->has_plan = false; return fail(QBGPU_ERR_ARG, "dist_set_pull_plan: a segment does not lie inside its owner's rows"); }
        D->plan.push_back({p, first[k], rows[k]});
    }
    return QBGPU_OK;
}

/* Late part j may start as soon as the first wait_after[j] segments of the pull plan have arrived (non-decreasing, the last one
 * = the number of segments).  Needs a pull plan; the transfers then all use one copy lane (they complete in order). */
int qbgpu_dist_set_wait_points(qbgpu_dist_t D, int n_late, const int32_t *wait_after)
{
    if (!D || n_late < 0 || (n_late && !wait_after)) return fail(QBGPU_ERR_ARG, "dist_set_wait_points: bad argument");
    D->wait_after.clear();
    if (n_late == 0) return QBGPU_OK;
    if (!D->has_plan || n_late != (int)D->late.size() || n_late > 8) return fail(QBGPU_ERR_STATE, "dist_set_wait_points: needs a pull plan and one entry per late part (at most 8)");
    for (int j = 0; j < n_late; j++) {
        if (wait_after[j] < 0 || wait_after[j] > (int)D->plan.size() || (j && wait_after[j] < wait_after[j - 1])) return fail(QBGPU_ERR_ARG, "dist_set_wait_points: must be non-decreasing and within the plan");
        if (!D->wait_ev[j]) QB_CUDA(cudaEventCreateWithFlags(&D->wait_ev[j], cudaEventDisableTiming));
    }
    if (wait_after[n_late - 1] != (int)D->plan.size()) return fail(QBGPU_ERR_ARG, "dist_set_wait_points: the last late part must wait for the whole plan");
    D->wait_after.assign(wait_after, wait_after + n_late);
    return QBGPU_OK;
}

int qbgpu_dist_own(qbgpu_dist_t D, int b, void **ptr, int64_t *nloc)
{
    if (!D || !ptr || (b != 0 && b != 1)) return fail(QBGPU_ERR_ARG, "dist_own: bad argument");
    *ptr = D->own(b);
    if (nloc) *nloc = D->nloc();
    return QBGPU_OK;
}

int qbgpu_dist_full(qbgpu_dist_t D, int b, void **ptr)
{
    if (!D || !ptr || (b != 0 && b != 1)) return fail(QBGPU_ERR_ARG, "dist_full: bad argument");
    *ptr = D->X(b);
    return QBGPU_OK;
}

int qbgpu_dist_barrier(qbgpu_dist_t D)
{
    QB_TRY(ensure_init());
    if (!D) return fail(QBGPU_ERR_ARG, "null argument");
    return dist_allreduce(D, D->scal, 0);
}

int qbgpu_dist_allreduce(qbgpu_dist_t D, double *dev, int count)
{
    QB_TRY(ensure_init());
    if (!D || (!dev && count)) return fail(QBGPU_ERR_ARG, "null argument");
    return dist_allreduce(D, dev, count);
}

/* own slice of X[b] <- this rank's rows of vec_randomize(n, seed), normalised over ALL ranks (src/miscellaneous.cc:371-388).
 * ref_row (device, nloc int32, or NULL): the reference's row of every local entry when the shard's vectors are in an
 * internal order (species shards: qbgpu_species_shard_ref_rows); NULL: the shard's rows are the reference's rows. */
int qbgpu_dist_randomize(qbgpu_dist_t D, int b, uint32_t seed, const int32_t *ref_row)
{
    QB_TRY(ensure_init());
    if (!D || (b != 0 && b != 1)) return fail(QBGPU_ERR_ARG, "dist_randomize: bad argument");
    Context &c = ctx();
    const int64_t nloc = D->nloc();
    if (seed == 0) return fail(QBGPU_ERR_ARG, "dist_randomize: seed 0 (the constant vector) is not a shard case");
    // opening barrier: a peer may still be pulling this rank's slice of X[b] for a product the caller issued before (a rank's
    // own product is done as soon as ITS pulls are; nothing tells it about its readers) -- the slice is first written
    // unnormalised and then scaled in place, so a reader caught in between would multiply by a half-scaled vector
    QB_TRY(dist_allreduce(D, D->scal, 0));
    if (nloc) {
        const int grid = (int)std::min<int64_t>((nloc + 255) / 256, 148 * 16);
        if (D->cplx) dist_randomize_kernel<double2><<<grid, 256, 0, c.stream>>>(nloc, D->lo(), ref_row, (double2 *)D->own(b), seed);
        else         dist_randomize_kernel<double><<<grid, 256, 0, c.stream>>>(nloc, D->lo(), ref_row, (double *)D->own(b), seed);
        QB_LAUNCH_COUNT();
        QB_CUDA(cudaGetLastError());
    }
    double *nn = D->scal + 40;
    if (nloc) QB_TRY(vec_nrm2sq(nloc, D->cplx, D->own(b), nn)); else QB_CUDA(cudaMemsetAsync(nn, 0, sizeof(double), c.stream));
    QB_TRY(dist_allreduce(D, nn, 1));
    double h = 0.0;
    QB_TRY(read_scalars(nn, &h, 1));
    if (nloc) QB_TRY(vec_scal(nloc, D->cplx, make_double2(1.0 / sqrt(h), 0.0), D->own(b)));
    QB_TRY(dist_allreduce(D, D->scal, 0));                 // barrier: every slice is final before anybody pulls
    return dist_timed_out(D, "dist_randomize");
}

/* y_local = H x: x = X[b] (own slice written by the caller), y_local: this rank's rows.  barrier bit 0 (1): pass a barrier
 * first -- the peers' slices are final before they are pulled (needed unless the caller's last call on this context was
 * already an all-reduce after x was written).  barrier bit 1 (2): pass a barrier after the product as well -- every rank's
 * pulls of X[b] are complete, so the caller may overwrite its own slice of X[b] as soon as the call's work is done on the
 * stream (without it, write the next x into the OTHER buffer, like the Krylov loops here do, or call qbgpu_dist_barrier). */
int qbgpu_dist_mv(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, int b, void *y_local, int barrier)
{
    QB_TRY(ensure_init());
    QB_TRY(dist_check(D, local_part, rest));
    if (!y_local || (b != 0 && b != 1)) return fail(QBGPU_ERR_ARG, "dist_mv: bad argument");
    if (barrier & 1) QB_TRY(dist_allreduce(D, D->scal, 0));
    FusedArgs a;
    a.y = y_local;
    QB_TRY(dist_product(D, local_part, rest, b, a));
    if (barrier & 2) QB_TRY(dist_allreduce(D, D->scal, 0));
    return QBGPU_OK;
}

// the loop of qbgpu_dist_lanczos / qbgpu_dist_lanczos_val1; phi (this rank's rows of phi0, or null): sr_val1.  Without phi no
// kernel of the re-orthogonalisation is launched.
static int dist_lanczos_loop(qbgpu_dist *D, const qbgpu_matrix *local_part, const qbgpu_matrix *rest, int64_t np, int64_t maxit, int64_t *m_out,
                             double *hess, bool is_val, const void *phi, int stop_on_breakdown)
{
    *m_out = 0;
    for (int64_t j = 0; j < 2 * maxit; j++) hess[j] = 0.0;
    if (np == 0) return QBGPU_OK;
    Context &c = ctx();
    const bool cplx = D->cplx;
    const int64_t nloc = D->nloc();
    double *state = D->scal;                                // 8 doubles (lanczos_step_*), then scratch
    double *p1 = D->scal + 24;                              // sr_val1: the projection's 8 doubles (vecops.cu: lanczos_step_b_phi)
    double *ab_dev = nullptr;
    QB_CUDA(cudaMalloc(&ab_dev, sizeof(double) * 2 * maxit));
    double *b_dev = ab_dev, *a_dev = ab_dev + maxit;
    auto done = [&](int rc) { cudaFree(ab_dev); return rc; };
    const double init[8] = {1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (cudaMemcpyAsync(state, init, sizeof init, cudaMemcpyHostToDevice, c.stream) != cudaSuccess) return done(fail(QBGPU_ERR_CUDA, "dist_lanczos: state upload"));
    cudaMemsetAsync(ab_dev, 0, sizeof(double) * 2 * maxit, c.stream);
    cudaStreamSynchronize(c.stream);
    std::vector<double> ritz(np + 2);
    int cnt_accuE0 = 0;
    double theta0_prev = 0.0;
    int64_t m = 0;
    // Speculation (QBGPU_DIST_SPECULATE=0: off): the product of a step goes to a scratch vector w, step b writes uz = w - a v.
    // The early parts of step m+1 (they read only the rank's own rows of the new vector) are then launched BEFORE the host has
    // read (a_m, b_{m+1}) back and evaluated the stop rule: the device works through the read-back, the O(m) Ritz solve and
    // the enqueueing of the next step's transfers (0.4 ms of 2.9 per step on eight GPUs: profiles/r02_dist_lanczos_phases_n8.txt)
    // instead of idling.  A step that does not happen only wrote w.
    const bool speculate = !(getenv("QBGPU_DIST_SPECULATE") && atoi(getenv("QBGPU_DIST_SPECULATE")) == 0);
    void *w = nullptr;
    cudaEvent_t ev_ab = nullptr;
    if (speculate && nloc) {
        if (cudaMalloc(&w, D->esize * (size_t)nloc) != cudaSuccess) return done(cuda_fail(cudaGetLastError(), "dist_lanczos: scratch vector", __FILE__, __LINE__));
        if (cudaEventCreateWithFlags(&ev_ab, cudaEventDisableTiming) != cudaSuccess) { cudaFree(w); return done(cuda_fail(cudaGetLastError(), "dist_lanczos: event", __FILE__, __LINE__)); }
    }
    auto done2 = [&](int rc) { if (ev_ab) { cudaStreamSynchronize(c.stream); cudaEventDestroy(ev_ab); } cudaFree(w); return done(rc); };
    bool early_issued = false;                              // the early parts of the coming step are already in the stream
    // QBGPU_VERBOSE: device time of the phases of a step (events on the compute stream) and host time between the steps
    const bool prof = getenv("QBGPU_VERBOSE") != nullptr;
    cudaEvent_t pe[7] = {};
    double tph[6] = {0, 0, 0, 0, 0, 0};
    if (prof) for (auto &e : pe) cudaEventCreate(&e);
    auto rec = [&](int i) { if (prof) cudaEventRecord(pe[i], c.stream); };
    while (m < np) {
        m++;
        const int bx = (int)((m - 1) % 2), bz = (int)(m % 2);
        void *uz = D->own(bz);
        // step a: w = sx*H*ux - b*sz*uz (into the scratch vector, or over uz); state[3] = partial <v, w>
        rec(0);
        if (int rc = dist_lanczos_step_a(D, local_part, rest, bx, uz, w, state, /*pulls_issued=*/m > 1, early_issued ? 2 : 0)) return done2(rc);
        early_issued = false;
        rec(1);
        if (int rc = dist_allreduce(D, state + 3, 1)) return done2(rc);
        rec(2);
        if (!phi) {
            if (int rc = lanczos_step_b(nloc, cplx, D->own(bx), uz, state, w)) return done2(rc);
            rec(3);
            if (int rc = dist_allreduce(D, state + 6, 1)) return done2(rc);      // also the barrier that makes X[bz] final everywhere
            rec(4);
            if (int rc = lanczos_step_c(state, a_dev, b_dev, m)) return done2(rc);
        } else {                                            // step b with the partials |U|^2, <phi0, U>: one all-reduce of 3
            if (int rc = lanczos_step_b_phi(nloc, cplx, D->own(bx), uz, phi, state, p1, w)) return done2(rc);
            rec(3);
            if (int rc = dist_allreduce(D, p1, 3)) return done2(rc);
            rec(4);
            if (int rc = lanczos_step_c_phi(state, p1, a_dev, b_dev, m)) return done2(rc);
        }
        cudaMemcpyAsync(c.scal_host, a_dev + (m - 1), sizeof(double), cudaMemcpyDeviceToHost, c.stream);
        cudaMemcpyAsync(c.scal_host + 1, b_dev + m, sizeof(double), cudaMemcpyDeviceToHost, c.stream);
        if (ev_ab) cudaEventRecord(ev_ab, c.stream);
        rec(5);
        if (phi) {
            // re-orthogonalisation (src/lanczos.cc:218-226), decided by step c from the reduced sums -- bit-identical on every
            // rank, so every rank takes the same branch: U -= h phi0 and the partial |U|^2 (a pass that does nothing when the
            // flag is off), the all-reduce (unconditional: also the barrier that makes the projected X[bz] final everywhere),
            // sx = 1/|U|.  All of it is in the stream before the next step's pulls and early parts below.
            if (int rc = lanczos_project(nloc, cplx, phi, uz, p1)) return done2(rc);
            if (int rc = dist_allreduce(D, p1 + 6, 1)) return done2(rc);
            if (int rc = lanczos_project_finalize(state, p1)) return done2(rc);
        }
        rec(6);
        // the slices of the NEXT step's vector (unnormalised: its scale travels as a scalar) are final now: start fetching
        // them -- and, with the scratch vector, multiplying by the early parts -- before the host reads the coefficients back
        // and decides whether there is a next step (if not: harmless)
        if (m < np) {
            if (int rc = dist_pull_mark(D)) return done2(rc);
            if (w) { if (int rc = dist_lanczos_step_a(D, local_part, rest, bz, D->own(bx), w, state, true, 1)) return done2(rc); early_issued = true; }
            if (int rc = dist_pull(D, bz)) return done2(rc);
        }
        if ((ev_ab ? cudaEventSynchronize(ev_ab) : cudaStreamSynchronize(c.stream)) != cudaSuccess) return done2(cuda_fail(cudaGetLastError(), "dist_lanczos: step", __FILE__, __LINE__));
        hess[maxit + m - 1] = c.scal_host[0];
        hess[m] = c.scal_host[1];
        if (prof) {
            cudaEventSynchronize(pe[6]);
            for (int i = 0; i < 6; i++) { float f = 0; cudaEventElapsedTime(&f, pe[i], pe[i + 1]); tph[i] += f; }
        }
        if (m == 1) continue;
        if (stop_on_breakdown && fabs(hess[m]) < kLanczosPrecisionD) break;                        // src/lanczos.cc:216
        if (is_val) {                                                                              // :228-248
            const double theta0 = tridiag_smallest(hess, maxit, m);
            if (m > 3) {
                const double accu_E0 = fabs((theta0 - theta0_prev) / theta0);
                if (accu_E0 < kLanczosPrecisionD) cnt_accuE0++; else cnt_accuE0 = 0;
                if (cnt_accuE0 > 15) {
                    double s_last = 0.0;
                    if (hess_eigen_host(hess, maxit, m, ritz.data(), nullptr, &s_last)) return done2(fail(QBGPU_ERR_NUMERIC, "hess_eigen: QL did not converge"));
                    if (fabs(hess[m] * s_last) < kLanczosPrecisionD) break;
                }
            }
            theta0_prev = theta0;
        }
    }
    *m_out = m;
    if (prof) {
        if (D->rank == 0) fprintf(stderr, "[qbgpu dist_lanczos%s] %lld steps on %d ranks, device ms per step: product %.3f | all-reduce %.3f | update pass %.3f | all-reduce %.3f | scalars+readback %.3f%s\n",
                                  phi ? " sr_val1" : "", (long long)m, D->world, tph[0] / m, tph[1] / m, tph[2] / m, tph[3] / m, tph[4] / m,
                                  phi ? (" | projection+all-reduce " + std::to_string(tph[5] / m)).c_str() : "");
        for (auto &e : pe) cudaEventDestroy(e);
    }
    if (int rc = dist_wait(D)) return done2(rc);             // (a fetch started for a step that did not happen)
    // hand the two live vectors back normalised (their scales live in state[0], state[1])
    if (nloc) {
        if (int rc = scale_copy(nloc, cplx, state + 0, 1.0, D->own((int)(m % 2)), D->own((int)(m % 2)))) return done2(rc);
        if (int rc = scale_copy(nloc, cplx, state + 1, 1.0, D->own((int)((m - 1) % 2)), D->own((int)((m - 1) % 2)))) return done2(rc);
    }
    if (int rc = dist_allreduce(D, D->scal + 8, 0)) return done2(rc);
    return done2(dist_timed_out(D, "dist_lanczos"));
}

/* lanczos(0, np, maxit, m, dim, H, v, hessenberg, purpose) of src/lanczos.cc:134-266 on the shards.  Start: the normalised
 * start vector's slice in the own part of X[0], visible to the peers (qbgpu_dist_randomize, or write it and call
 * qbgpu_dist_barrier).  purpose: "sr_val0" (stop rule of :228-248; every rank takes the same decision from the identical
 * reduced coefficients) or "dnmcs" (np steps unless b_m < 2e-12).  hess[2*maxit]: b in [0,maxit), a in [maxit, 2 maxit), on
 * every rank.  On return the normalised v_m is the own slice of X[m % 2], v_{m-1} of X[(m-1) % 2]. */
int qbgpu_dist_lanczos(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, int64_t np, int64_t maxit, int64_t *m_out,
                       double *hess, const char *purpose, int stop_on_breakdown)
{
    QB_TRY(ensure_init());
    QB_TRY(dist_check(D, local_part, rest));
    if (!m_out || !hess || !purpose) return fail(QBGPU_ERR_ARG, "dist_lanczos: null argument");
    const bool is_val = strcmp(purpose, "sr_val0") == 0, is_dn = strcmp(purpose, "dnmcs") == 0;
    if (!is_val && !is_dn) return fail(QBGPU_ERR_ARG, "dist_lanczos: purpose must be sr_val0 or dnmcs");
    if (!(np >= 0 && np < maxit)) return fail(QBGPU_ERR_ARG, "dist_lanczos: need 0 <= np < maxit");
    return dist_lanczos_loop(D, local_part, rest, np, maxit, m_out, hess, is_val, nullptr, stop_on_breakdown);
}

/* lanczos(0, np, maxit, ..., "sr_val1") of src/lanczos.cc:134-266 on the shards: the loop above (stop rule of sr_val0) with the
 * re-orthogonalisation against phi0 of :218-226 in every step after the first, decided and applied on the device. */
int qbgpu_dist_lanczos_val1(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, const void *phi0_local, int64_t np, int64_t maxit,
                            int64_t *m_out, double *hess, int stop_on_breakdown)
{
    QB_TRY(ensure_init());
    QB_TRY(dist_check(D, local_part, rest));
    if (!m_out || !hess || !phi0_local) return fail(QBGPU_ERR_ARG, "dist_lanczos_val1: null argument (phi0_local, m or hess)");
    if (!(np >= 0 && np < maxit)) return fail(QBGPU_ERR_ARG, "dist_lanczos_val1: need 0 <= np < maxit");
    return dist_lanczos_loop(D, local_part, rest, np, maxit, m_out, hess, true, phi0_local, stop_on_breakdown);
}


/* energy_scale of src/kpm.cc:45-88 on the shards: iters-1 Lanczos steps from vec_randomize(seed 1), bounds widened by extend. */
int qbgpu_dist_energy_scale(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, const int32_t *ref_row, double *lo, double *hi,
                            double extend, int64_t iters)
{
    if (!lo || !hi || iters < 3) return fail(QBGPU_ERR_ARG, "dist_energy_scale: bad argument");
    QB_TRY(qbgpu_dist_randomize(D, 0, 1, ref_row));
    const int64_t mm = iters - 1;
    std::vector<double> hess(2 * iters, 0.0), ritz(mm);
    int64_t m = 0;
    QB_TRY(qbgpu_dist_lanczos(D, local_part, rest, mm, iters, &m, hess.data(), "dnmcs", 0));
    if (hess_eigen_host(hess.data(), iters, mm, ritz.data(), nullptr, nullptr)) return fail(QBGPU_ERR_NUMERIC, "hess_eigen: QL did not converge");
    const double l = ritz[0], h = ritz[mm - 1], slack = extend * (h - l);
    *lo = l - slack; *hi = h + slack;
    return QBGPU_OK;
}

/* Chebyshev moments mu_k = <phi|T_k((H-c)/s)|phi>, k < nmom, with phi = the own slices of X[0] (visible to the peers).  Two
 * moments per product through the doubling identities (krylov.cu: kpm_impl); the partial inner products of all steps are
 * reduced across the ranks once, at the end. */
int qbgpu_dist_kpm_moments(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, double lo, double hi, int64_t nmom, double *mu)
{
    QB_TRY(ensure_init());
    QB_TRY(dist_check(D, local_part, rest));
    if (!mu || nmom < 1 || !(hi > lo)) return fail(QBGPU_ERR_ARG, "dist_kpm_moments: bad argument");
    Context &c = ctx();
    const bool cplx = D->cplx;
    const int64_t nloc = D->nloc();
    const double cc = 0.5 * (hi + lo), ss = 0.5 * (hi - lo);
    const int64_t nprod = nmom / 2 + 1;
    double *dots = nullptr;
    QB_CUDA(cudaMalloc(&dots, sizeof(double) * 4 * (nprod + 1)));
    auto done = [&](int rc) { cudaFree(dots); return rc; };
    cudaMemsetAsync(dots, 0, sizeof(double) * 4 * (nprod + 1), c.stream);
    if (nloc) { if (int rc = vec_nrm2sq(nloc, cplx, D->own(0), dots)) return done(rc); }
    // T_0 = phi in X[0]; T_{k+1} = 2 Ht T_k - T_{k-1} written over T_{k-1}: X[(k+1) % 2]
    for (int64_t k = 0; k < nprod; k++) {
        const int bx = (int)(k % 2), by = (int)((k + 1) % 2);
        FusedArgs fa;
        fa.y = D->own(by); fa.dots = dots + 4 * (k + 1);
        if (k == 0) { fa.alpha = make_double2(1.0 / ss, 0.0); fa.gamma = make_double2(-cc / ss, 0.0); }
        else { fa.alpha = make_double2(2.0 / ss, 0.0); fa.gamma = make_double2(-2.0 * cc / ss, 0.0); fa.beta = make_double2(-1.0, 0.0); fa.z = D->own(by); }
        if (int rc = dist_product(D, local_part, rest, bx, fa)) return done(rc);
        if (int rc = dist_allreduce(D, D->scal + 8, 0)) return done(rc);      // barrier: X[by] final before the next pulls
    }
    if (int rc = dist_allreduce_array(D, dots, 4 * (nprod + 1))) return done(rc);
    std::vector<double> h(4 * (nprod + 1));
    cudaMemcpyAsync(h.data(), dots, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, c.stream);
    if (cudaStreamSynchronize(c.stream) != cudaSuccess) return done(cuda_fail(cudaGetLastError(), "dist_kpm", __FILE__, __LINE__));
    // dots[4(k+1)] = Re <T_k, T_{k+1}>, dots[4(k+1)+2] = |T_{k+1}|^2 ; mu_0 = dots[0]
    const double mu0 = h[0];
    const double mu1 = h[4];
    for (int64_t j = 0; j < nmom; j++) {
        if (j == 0) mu[j] = mu0;
        else if (j == 1) mu[j] = mu1;
        else if (j % 2 == 0) { const int64_t k = j / 2 - 1; mu[j] = 2.0 * h[4 * (k + 1) + 2] - mu0; }     // mu_{2k+2} = 2|T_{k+1}|^2 - mu_0
        else { const int64_t k = (j - 1) / 2; mu[j] = 2.0 * h[4 * (k + 1)] - mu1; }                       // mu_{2k+1} = 2<T_k,T_{k+1}> - mu_1
    }
    return done(dist_timed_out(D, "dist_kpm_moments"));
}

/* eigenvec_CG of src/lanczos.cc:281-341 on the shards.  v (in/out): this rank's rows of the start / ground-state vector;
 * r, p, pp: work vectors of nloc entries, all device pointers.  Uses X[0] as the exchange buffer of every product. */
int qbgpu_dist_eigenvec_cg(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, int64_t maxit, int64_t *m_io, const double E0[2],
                           double *accu_out, void *v, void *r, void *p, void *pp)
{
    QB_TRY(ensure_init());
    QB_TRY(dist_check(D, local_part, rest));
    if (!m_io || !accu_out || !E0 || !v || !r || !p || !pp) return fail(QBGPU_ERR_ARG, "dist_eigenvec_cg: null argument");
    if (maxit <= 0 || *m_io != 0) return fail(QBGPU_ERR_ARG, "dist_eigenvec_cg: starts at m = 0");
    Context &c = ctx();
    const bool cplx = D->cplx;
    const int64_t nloc = D->nloc();
    const size_t vb = D->esize;
    double *sc = D->scal + 16;                              // [0]=gamma [1,2]=delta [3]=|pp|^2 [4]=|r|^2 [5]=gamma_next [6] scratch
    QB_CUDA(cudaMemsetAsync(sc, 0, sizeof(double) * 8, c.stream));
    const double2 e0 = make_double2(E0[0], E0[1]);
    // a product on `src` (nloc entries): copy it into the own slice of X[0], barrier, pull + multiply
    auto product = [&](const void *src, FusedArgs fa) -> int {
        if (nloc) QB_CUDA(cudaMemcpyAsync(D->own(0), src, vb * (size_t)nloc, cudaMemcpyDeviceToDevice, c.stream));
        QB_TRY(dist_allreduce(D, D->scal + 8, 0));
        return dist_product(D, local_part, rest, 0, fa);
    };
    int64_t m = 0;
    double accu = 0.0;
    while (m < maxit) {
        if (accu < kLanczosPrecisionD) {                    // src/lanczos.cc:295
            double nn;
            if (nloc) QB_TRY(vec_nrm2sq(nloc, cplx, v, sc + 6)); else QB_CUDA(cudaMemsetAsync(sc + 6, 0, sizeof(double), c.stream));
            QB_TRY(dist_allreduce(D, sc + 6, 1));
            QB_TRY(read_scalars(sc + 6, &nn, 1));
            const double rnorm = sqrt(nn);
            if (m == 0 || fabs(rnorm - 1.0) > kLanczosPrecisionD) {       // :297 re-normalise and restart
                if (nloc) QB_TRY(vec_scal(nloc, cplx, make_double2(1.0 / rnorm, 0.0), v));
                FusedArgs fa;                               // r = (E0 - H) v ; |r|^2 from the epilogue
                fa.y = r; fa.alpha = make_double2(-1.0, 0.0); fa.gamma = e0; fa.dots = sc + 1;
                QB_TRY(product(v, fa));
                QB_TRY(dist_allreduce(D, sc + 1, 3));
                if (nloc) QB_CUDA(cudaMemcpyAsync(p, r, vb * (size_t)nloc, cudaMemcpyDeviceToDevice, c.stream));
                double h[3];
                QB_TRY(read_scalars(sc + 1, h, 3));
                accu = sqrt(h[2]);
                QB_CUDA(cudaMemcpyAsync(sc, &accu, sizeof(double), cudaMemcpyHostToDevice, c.stream));
                QB_CUDA(cudaStreamSynchronize(c.stream));
                m++;
                if (accu < kLanczosPrecisionD) break;       // :315
            } else {
                break;                                      // :317
            }
        } else {
            FusedArgs fa;                                   // pp = (H - E0 + eps) p ; delta = <p,pp>   (:320-323)
            fa.y = pp; fa.alpha = make_double2(1.0, 0.0);
            fa.gamma = make_double2(DBL_EPSILON - e0.x, -e0.y); fa.dots = sc + 1;
            QB_TRY(product(p, fa));
            QB_TRY(dist_allreduce(D, sc + 1, 3));
            if (nloc) QB_TRY(cg_update_vr(nloc, cplx, sc, v, r, p, pp)); else QB_CUDA(cudaMemsetAsync(sc + 4, 0, sizeof(double), c.stream));
            QB_TRY(dist_allreduce(D, sc + 4, 1));
            if (nloc) QB_TRY(cg_update_p(nloc, cplx, sc, r, p));
            else { double g[5]; QB_TRY(read_scalars(sc, g, 5)); const double gn = sqrt(g[4]); QB_CUDA(cudaMemcpyAsync(sc + 5, &gn, sizeof(double), cudaMemcpyHostToDevice, c.stream)); QB_CUDA(cudaStreamSynchronize(c.stream)); }
            QB_CUDA(cudaMemcpyAsync(sc, sc + 5, sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
            QB_TRY(read_scalars(sc, &accu, 1));
            m++;
        }
    }
    *m_io = m;
    *accu_out = accu;
    return dist_timed_out(D, "dist_eigenvec_cg");
}


/* model<T>::locate_E0_lanczos(nev, ncv, maxit) of src/model.cc:1124-1316 on the shards, stage by stage as csr.locate_E0_lanczos
 * runs it on one GPU (same seeds, same order): E0 by sr_val0 Lanczos from vec_randomize(1); phi0 by eigenvec_CG from
 * vec_randomize(1); E1 by sr_val1 Lanczos from vec_randomize(1) projected off phi0; phi1 by eigenvec_CG at E1 from
 * vec_randomize(8), orthonormalised against phi0 when the gap is below 2e-12 (:1302-1311).  Uses X[0] and X[1]. */
int qbgpu_dist_locate_e0_lanczos(qbgpu_dist_t D, qbgpu_matrix_t local_part, qbgpu_matrix_t rest, const int32_t *ref_row, int nev, int ncv,
                                 int64_t maxit, double *eigenvals, void *phi_local, int64_t *steps, double *accuracies)
{
    QB_TRY(ensure_init());
    QB_TRY(dist_check(D, local_part, rest));
    if (!(nev > 0 && nev <= 2 && nev - 1 <= ncv && ncv <= nev))
        return fail(QBGPU_ERR_ARG, "dist_locate_e0_lanczos: need 0 < nev <= 2 and nev-1 <= ncv <= nev (src/model.cc:1141)");
    if (!eigenvals || !steps || !accuracies || (ncv > 0 && !phi_local)) return fail(QBGPU_ERR_ARG, "dist_locate_e0_lanczos: null argument (eigenvals, steps, accuracies, or phi_local with ncv > 0)");
    if (maxit < 2) return fail(QBGPU_ERR_ARG, "dist_locate_e0_lanczos: need maxit >= 2");
    for (int i = 0; i < 4; i++) { steps[i] = 0; accuracies[i] = 0.0; }
    Context &c = ctx();
    const int64_t nloc = D->nloc();
    const size_t vb = D->esize * (size_t)nloc;
    std::vector<double> hess(2 * maxit), ritz(maxit);
    // the lowest Ritz value of a finished run and its residual estimate |b_m s_{m-1}|
    auto lowest = [&](int64_t m, double *E, double *accu) -> int {
        double s_last = 0.0;
        if (hess_eigen_host(hess.data(), maxit, m, ritz.data(), nullptr, &s_last)) return fail(QBGPU_ERR_NUMERIC, "hess_eigen: QL did not converge");
        *E = ritz[0];
        *accu = fabs(hess[m] * s_last);
        return QBGPU_OK;
    };
    // stage 1 (:1165-1196): E0
    QB_TRY(qbgpu_dist_randomize(D, 0, 1, ref_row));
    int64_t m = 0;
    QB_TRY(dist_lanczos_loop(D, local_part, rest, maxit - 1, maxit, &m, hess.data(), true, nullptr, 1));
    double E0 = 0.0;
    QB_TRY(lowest(m, &E0, &accuracies[0]));
    eigenvals[0] = E0;
    steps[0] = m;
    if (ncv == 0) return QBGPU_OK;
    // stage 2 (:1205-1231): phi0 = eigenvec_CG(E0) from vec_randomize(1)
    char *phi0 = (char *)phi_local, *phi1 = ncv == 2 ? phi0 + vb : nullptr;
    DevBufGuard r, p, pp;                                   // CG work vectors, freed on every way out
    QB_CUDA(r.alloc(vb)); QB_CUDA(p.alloc(vb)); QB_CUDA(pp.alloc(vb));
    auto seeded = [&](void *dst, uint32_t seed) -> int {    // dst <- this rank's rows of vec_randomize(seed), via X[0]
        QB_TRY(qbgpu_dist_randomize(D, 0, seed, ref_row));
        if (nloc) QB_CUDA(cudaMemcpyAsync(dst, D->own(0), vb, cudaMemcpyDeviceToDevice, c.stream));
        return QBGPU_OK;
    };
    QB_TRY(seeded(phi0, 1));
    const double e0[2] = {E0, 0.0};
    QB_TRY(qbgpu_dist_eigenvec_cg(D, local_part, rest, maxit, &steps[1], e0, &accuracies[1], phi0, r.p, p.p, pp.p));
    double gap = 0.0;
    if (nev == 2) {
        // stage 3 (:1233-1265): E1 by Lanczos from vec_randomize(1) projected off phi0, re-orthogonalised in every step
        QB_TRY(qbgpu_dist_randomize(D, 0, 1, ref_row));
        QB_TRY(dist_orthonormalize(D, phi0, D->own(0)));
        QB_TRY(dist_allreduce(D, D->scal + 8, 0));          // barrier: the start vector is final everywhere before the pulls
        int64_t m1 = 0;
        QB_TRY(dist_lanczos_loop(D, local_part, rest, maxit - 1, maxit, &m1, hess.data(), true, phi0, 1));
        QB_TRY(lowest(m1, &eigenvals[1], &accuracies[2]));
        steps[2] = m1;
        gap = eigenvals[1] - E0;
    }
    if (ncv == 2) {
        // stage 4 (:1275-1315): phi1 = eigenvec_CG(E1) from vec_randomize(8); a degenerate pair is orthonormalised
        QB_TRY(seeded(phi1, 8));
        const double e1[2] = {eigenvals[1], 0.0};
        QB_TRY(qbgpu_dist_eigenvec_cg(D, local_part, rest, maxit, &steps[3], e1, &accuracies[3], phi1, r.p, p.p, pp.p));
        if (gap < kLanczosPrecisionD) QB_TRY(dist_orthonormalize(D, phi0, phi1));
    }
    QB_TRY(dist_allreduce(D, D->scal + 8, 0));
    return dist_timed_out(D, "dist_locate_e0_lanczos");
}

}  // extern "C"
