// quantum_basis_b200/csrc/matrix.cu -- upload and conversion of the reference's CSR into the device layout.
//
// Input: the reference's csr_mat<T> arrays (src/qbasis.h:976-1021): zero-based 4-array CSR with int64 indices
// (MKL_INT under -DMKL_ILP64), `sym` = only the upper triangle (col >= row) is stored, every diagonal present
// (src/sparse.cc:44-54).  This is the point where the reference creates its MKL handle (src/sparse.cc:129,258).
// Output: the expanded Hermitian CSR of internal.hpp (int32 columns, int64 row offsets, rows sorted by column,
// values demoted to fp64 when every imaginary part is exactly zero).
//
// The conversion runs on the device:
//   1. count   per output row: stored upper entries + transposed entries landing in it   (one thread per input row)
//   2. scan    exclusive prefix sum -> rowptr (cub::DeviceScan)
//   3. fill    upper entries go to their final slot directly (they follow the transposed ones, which all have
//              col < row); transposed entries claim a slot with an atomic cursor
//   4. sort    each row's transposed segment by column (insertion sort per row; segments are short) so the
//              layout -- and therefore every floating-point sum -- is deterministic
#include "internal.hpp"
#include <cub/device/device_scan.cuh>
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <vector>

namespace qb {

static double wall() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

constexpr int kCBlock = 256;

// error flag bits written by the conversion kernels
constexpr int kErrColRange = 1;
constexpr int kErrColOrder = 2;   // a row whose referenced columns are not strictly ascending

template <typename T> struct ValOps;
template <> struct ValOps<double>  { __device__ static double conj(double v) { return v; }  __device__ static double imag_abs(double) { return 0.0; } };
template <> struct ValOps<double2> { __device__ static double2 conj(double2 v) { return make_double2(v.x, -v.y); } __device__ static double imag_abs(double2 v) { return fabs(v.y); } };

// counts for rows in [lo,hi): cnt_u[i-lo] = kept stored entries of row i, cnt_t[j-lo] = transposed entries landing in row j
__global__ void __launch_bounds__(kCBlock) count_kernel(int64_t n, int64_t base, const int64_t *__restrict__ rs, const int64_t *__restrict__ re,
                                                        const int64_t *__restrict__ col, int sym, int64_t lo, int64_t hi,
                                                        int *cnt_u, int *cnt_t, int *err)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int cu = 0;
        int64_t prev = -1;
        for (int64_t p = rs[i] - base; p < re[i] - base; p++) {
            const int64_t j = col[p];
            if (j < 0 || j >= n) { atomicOr(err, kErrColRange); continue; }
            if (sym && j < i) continue;                     // FILL_UPPER: the lower part is not referenced
            // the device layout keeps the referenced entries of a row in input order and every later stage (column
            // blocks of the multi-GPU exchanges, the ring order) relies on ascending columns -- what the reference's
            // csr_mat(lil_mat&) always produces (sorted forward_list, src/sparse.cc:202-233); anything else is refused
            if (j <= prev) atomicOr(err, kErrColOrder);
            prev = j;
            if (sym) {
                cu++;
                if (j != i && j >= lo && j < hi) atomicAdd(&cnt_t[j - lo], 1);
            } else {
                cu++;
            }
        }
        if (i >= lo && i < hi) cnt_u[i - lo] = cu;
    }
}

__global__ void __launch_bounds__(kCBlock) add_counts_kernel(int64_t nloc, const int *cnt_u, const int *cnt_t, int64_t *len)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= nloc; i += (int64_t)gridDim.x * blockDim.x)
        len[i] = (i < nloc) ? (int64_t)cnt_u[i] + (int64_t)cnt_t[i] : 0;
}

template <typename TIn, typename TOut>
__device__ __forceinline__ TOut cast_val(TIn v);
template <> __device__ __forceinline__ double  cast_val<double, double>(double v) { return v; }
template <> __device__ __forceinline__ double2 cast_val<double2, double2>(double2 v) { return v; }

template <typename T>
__global__ void __launch_bounds__(kCBlock) fill_rows_kernel(int64_t n, int64_t base, const int64_t *__restrict__ rs, const int64_t *__restrict__ re,
                                                       const int64_t *__restrict__ col, const T *__restrict__ val, int sym,
                                                       int64_t lo, int64_t hi, const int64_t *__restrict__ rowptr,
                                                       const int *__restrict__ cnt_t, int *cursor, int32_t *ocol, T *oval, double *max_imag)
{
    double mi = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const bool mine = (i >= lo && i < hi);
        int64_t up = mine ? rowptr[i - lo] + cnt_t[i - lo] : 0;   // first slot of the stored (upper) run of row i
        for (int64_t p = rs[i] - base; p < re[i] - base; p++) {
            const int64_t j = col[p];
            if (j < 0 || j >= n) continue;
            if (sym && j < i) continue;
            const T v = val[p];
            if (mine) { ocol[up] = (int32_t)j; oval[up] = v; up++; mi = fmax(mi, ValOps<T>::imag_abs(v)); }
            if (sym && j != i && j >= lo && j < hi) {
                const int slot = atomicAdd(&cursor[j - lo], 1);
                const int64_t q = rowptr[j - lo] + slot;
                ocol[q] = (int32_t)i; oval[q] = ValOps<T>::conj(v);
                mi = fmax(mi, ValOps<T>::imag_abs(v));
            }
        }
    }
    // max |imag| over everything this block wrote (non-negative doubles order like their bit patterns)
    for (int o = 16; o > 0; o >>= 1) mi = fmax(mi, __shfl_xor_sync(0xffffffffu, mi, o));
    if ((threadIdx.x & 31) == 0 && mi > 0.0) atomicMax((unsigned long long *)max_imag, (unsigned long long)__double_as_longlong(mi));
}

template <typename T>
__global__ void __launch_bounds__(kCBlock) sort_transposed_kernel(int64_t nloc, const int64_t *__restrict__ rowptr, const int *__restrict__ cnt_t,
                                                                  int32_t *ocol, T *oval)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nloc; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t s = rowptr[i];
        const int len = cnt_t[i];
        for (int a = 1; a < len; a++) {
            const int32_t c = ocol[s + a];
            const T v = oval[s + a];
            int b = a - 1;
            while (b >= 0 && ocol[s + b] > c) { ocol[s + b + 1] = ocol[s + b]; oval[s + b + 1] = oval[s + b]; b--; }
            ocol[s + b + 1] = c; oval[s + b + 1] = v;
        }
    }
}

__global__ void __launch_bounds__(kCBlock) demote_kernel(int64_t nnz, const double2 *__restrict__ in, double *out)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) out[i] = in[i].x;
}

static int grid_for(int64_t n) { int64_t g = (n + kCBlock - 1) / kCBlock; if (g < 1) g = 1; if (g > 148 * 32) g = 148 * 32; return (int)g; }

// Expansion of a DEVICE-resident reference-format CSR (int64 row_start/row_end/col, base-relative offsets, values T)
// into the handle's layout.  Shared by the host entry points (after their upload) and by the on-device sector
// assembler (sectors.cu), whose upper triangle never leaves HBM.  Does not free its inputs.
template <typename T>   // T = double or double2 (input scalar type)
static int convert_device(qbgpu_matrix *A, int64_t n, int64_t base, const int64_t *d_rs, const int64_t *d_re, const int64_t *d_col,
                          const T *d_val, int sym, int flags, int64_t lo, int64_t hi)
{
    Context &c = ctx();
    const int64_t nloc = hi - lo;
    const double t1 = wall();
    int64_t *d_len = nullptr;
    int *d_cnt_u = nullptr, *d_cnt_t = nullptr, *d_cursor = nullptr, *d_err = nullptr;
    double *d_maximag = nullptr;
    void *d_tmp = nullptr;
    auto cleanup = [&]() {
        cudaFree(d_len); cudaFree(d_cnt_u); cudaFree(d_cnt_t); cudaFree(d_cursor); cudaFree(d_err); cudaFree(d_maximag); cudaFree(d_tmp);
    };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&d_cnt_u, sizeof(int) * (nloc + 1)));
    QB_CU(cudaMalloc(&d_cnt_t, sizeof(int) * (nloc + 1)));
    QB_CU(cudaMalloc(&d_cursor, sizeof(int) * (nloc + 1)));
    QB_CU(cudaMalloc(&d_len, sizeof(int64_t) * (nloc + 1)));
    QB_CU(cudaMalloc(&d_err, sizeof(int)));
    QB_CU(cudaMalloc(&d_maximag, sizeof(double)));
    QB_CU(cudaMemsetAsync(d_cnt_u, 0, sizeof(int) * (nloc + 1), c.stream));
    QB_CU(cudaMemsetAsync(d_cnt_t, 0, sizeof(int) * (nloc + 1), c.stream));
    QB_CU(cudaMemsetAsync(d_cursor, 0, sizeof(int) * (nloc + 1), c.stream));
    QB_CU(cudaMemsetAsync(d_err, 0, sizeof(int), c.stream));
    QB_CU(cudaMemsetAsync(d_maximag, 0, sizeof(double), c.stream));
    count_kernel<<<grid_for(n), kCBlock, 0, c.stream>>>(n, base, d_rs, d_re, d_col, sym, lo, hi, d_cnt_u, d_cnt_t, d_err);
    QB_LAUNCH_COUNT();
    add_counts_kernel<<<grid_for(nloc + 1), kCBlock, 0, c.stream>>>(nloc, d_cnt_u, d_cnt_t, d_len);
    QB_LAUNCH_COUNT();
    QB_CU(cudaMalloc(&A->rowptr, sizeof(int64_t) * (nloc + 1)));
    size_t tmp_bytes = 0;
    QB_CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_len, A->rowptr, nloc + 1, c.stream));
    QB_CU(cudaMalloc(&d_tmp, tmp_bytes ? tmp_bytes : 1));
    QB_CU(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_len, A->rowptr, nloc + 1, c.stream));
    int64_t nnz = 0;
    int herr = 0;
    QB_CU(cudaMemcpyAsync(&nnz, A->rowptr + nloc, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaMemcpyAsync(&herr, d_err, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    if (herr & kErrColRange) { cleanup(); return fail(QBGPU_ERR_ARG, "create_csr: column index out of range"); }
    if (herr & kErrColOrder) { cleanup(); return fail(QBGPU_ERR_ARG, "create_csr: the columns of a row must be strictly ascending (as csr_mat(lil_mat&) stores them, reference src/sparse.cc:202-233)"); }
    A->nnz = nnz;
    T *oval = nullptr;
    QB_CU(cudaMalloc(&A->col, sizeof(int32_t) * (nnz ? nnz : 1) + 64));
    QB_CU(cudaMalloc(&oval, sizeof(T) * (nnz ? nnz : 1) + 64));
    A->val = oval;
    A->val_real = (sizeof(T) == sizeof(double));
    fill_rows_kernel<T><<<grid_for(n), kCBlock, 0, c.stream>>>(n, base, d_rs, d_re, d_col, d_val, sym, lo, hi, A->rowptr, d_cnt_t, d_cursor,
                                                          A->col, oval, d_maximag);
    QB_LAUNCH_COUNT();
    if (sym) {
        sort_transposed_kernel<T><<<grid_for(nloc), kCBlock, 0, c.stream>>>(nloc, A->rowptr, d_cnt_t, A->col, oval);
        QB_LAUNCH_COUNT();
    }
    double maximag = 0.0;
    QB_CU(cudaMemcpyAsync(&maximag, d_maximag, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
    if (sizeof(T) == 16 && maximag == 0.0 && !(flags & QBGPU_KEEP_COMPLEX)) {
        // every imaginary part is exactly zero (always the case for the reference's model<complex> with real
        // couplings, SURVEY F3): store fp64 values, 12 instead of 20 bytes per entry
        double *rv = nullptr;
        QB_CU(cudaMalloc(&rv, sizeof(double) * (nnz ? nnz : 1) + 64));
        demote_kernel<<<grid_for(nnz), kCBlock, 0, c.stream>>>(nnz, (const double2 *)oval, rv);
        QB_LAUNCH_COUNT();
        QB_CU(cudaStreamSynchronize(c.stream));
        cudaFree(oval);
        A->val = rv;
        A->val_real = true;
    }
    cleanup();
#undef QB_CU
    A->convert_s = wall() - t1;
    return QBGPU_OK;
}

int create_from_device_csr(qbgpu_matrix_t *out, int64_t n, const int64_t *d_rs, const int64_t *d_re, const int64_t *d_col,
                           const void *d_val, bool val_complex, int64_t nnz_input, int sym, int flags, bool api_complex)
{
    if (!out) return fail(QBGPU_ERR_ARG, "null handle pointer");
    *out = nullptr;
    if (n <= 0 || n > 2147483647LL) return fail(QBGPU_ERR_ARG, "device csr: bad dimension");
    auto *A = new qbgpu_matrix;
    A->n = n; A->row_lo = 0; A->row_hi = n; A->api_complex = api_complex; A->nnz_input = nnz_input;
    int rc = val_complex ? convert_device<double2>(A, n, 0, d_rs, d_re, d_col, (const double2 *)d_val, sym, flags, 0, n)
                         : convert_device<double>(A, n, 0, d_rs, d_re, d_col, (const double *)d_val, sym, flags, 0, n);
    if (rc == QBGPU_OK) rc = autotune(A, flags);
    if (rc) { qbgpu_destroy(A); return rc; }
    *out = A;
    return QBGPU_OK;
}

template <typename T>   // T = double or double2 (input scalar type)
static int create_from_host(qbgpu_matrix_t *out, int64_t n, const int64_t *rs, const int64_t *re, const int64_t *col,
                            const void *val, int sym, int flags, int64_t lo, int64_t hi, bool api_complex)
{
    QB_TRY(ensure_init());
    Context &c = ctx();
    if (!out) return fail(QBGPU_ERR_ARG, "null handle pointer");
    *out = nullptr;
    if (n <= 0 || !rs || !re || !col || !val) return fail(QBGPU_ERR_ARG, "create_csr: null array or n <= 0");
    if (n > 2147483647LL) return fail(QBGPU_ERR_ARG, "create_csr: n exceeds the int32 column range of the device layout");
    if (hi < 0) hi = n;
    if (lo < 0 || lo > hi || hi > n) return fail(QBGPU_ERR_ARG, "create_csr: bad row shard");
    int64_t base = rs[0], top = re[0];
    for (int64_t i = 0; i < n; i++) {
        if (re[i] < rs[i]) return fail(QBGPU_ERR_ARG, "create_csr: row_end < row_start");
        if (rs[i] < base) base = rs[i];
        if (re[i] > top) top = re[i];
    }
    const int64_t span = top - base;                        // entries of col/val that are referenced
    auto *A = new qbgpu_matrix;
    A->n = n; A->row_lo = lo; A->row_hi = hi; A->api_complex = api_complex; A->nnz_input = span;

    const double t0 = wall();
    int64_t *d_rs = nullptr, *d_re = nullptr, *d_col = nullptr;
    T *d_val = nullptr;
    auto cleanup = [&]() { cudaFree(d_rs); cudaFree(d_re); cudaFree(d_col); cudaFree(d_val); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); qbgpu_destroy(A); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&d_rs, sizeof(int64_t) * n));
    QB_CU(cudaMalloc(&d_re, sizeof(int64_t) * n));
    QB_CU(cudaMalloc(&d_col, sizeof(int64_t) * (span ? span : 1)));
    QB_CU(cudaMalloc(&d_val, sizeof(T) * (span ? span : 1)));
    QB_CU(cudaMemcpyAsync(d_rs, rs, sizeof(int64_t) * n, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_re, re, sizeof(int64_t) * n, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_col, col + base, sizeof(int64_t) * span, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_val, (const T *)val + base, sizeof(T) * span, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
#undef QB_CU
    A->upload_s = wall() - t0;
    int rc = convert_device<T>(A, n, base, d_rs, d_re, d_col, d_val, sym, flags, lo, hi);
    cleanup();
    if (rc == QBGPU_OK) rc = autotune(A, flags);
    if (rc) { qbgpu_destroy(A); return rc; }
    *out = A;
    return QBGPU_OK;
}


// ------------------------------------------------------------------------------------------ value dictionary
// Exact-diagonalisation Hamiltonians carry very few distinct matrix elements (Heisenberg: J/2 and multiples of J/4;
// Hubbard: +-t and multiples of U), so the 8-byte value stream can be replaced by 1-byte codes into a table of the
// distinct fp64 bit patterns (QBGPU_VALUE_DICT).  Lossless: the product decodes the identical doubles.
constexpr int kDictSlots = 1024;                           // open-addressing hash set, at most 256 live keys
constexpr unsigned long long kEmptyKey = 0xFFFFFFFFFFFFFFFFull;   // a NaN payload no finite matrix element has

__device__ __forceinline__ unsigned dict_hash(unsigned long long k) { k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; return (unsigned)k & (kDictSlots - 1); }

__global__ void __launch_bounds__(kCBlock) dict_collect_kernel(int64_t nnz, const double *__restrict__ val, unsigned long long *slots, int *count)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) {
        if (*(volatile int *)count > 256) return;          // too many distinct values: give up early
        const unsigned long long k = (unsigned long long)__double_as_longlong(val[i]);
        unsigned h = dict_hash(k);
        for (int probe = 0; probe < kDictSlots; probe++, h = (h + 1) & (kDictSlots - 1)) {
            unsigned long long cur = slots[h];
            if (cur == k) break;
            if (cur == kEmptyKey) {
                cur = atomicCAS(&slots[h], kEmptyKey, k);
                if (cur == kEmptyKey) { atomicAdd(count, 1); break; }
                if (cur == k) break;
            }
        }
    }
}

__global__ void __launch_bounds__(kCBlock) dict_encode_kernel(int64_t nnz, const double *__restrict__ val, const unsigned long long *__restrict__ slots,
                                                              const int *__restrict__ slot_code, uint8_t *code)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long k = (unsigned long long)__double_as_longlong(val[i]);
        unsigned h = dict_hash(k);
        while (slots[h] != k) h = (h + 1) & (kDictSlots - 1);
        code[i] = (uint8_t)slot_code[h];
    }
}

int value_dict_encode(qbgpu_matrix *A, int max_entries)
{
    Context &c = ctx();
    if (!A->val_real || A->ndict || A->format != QBGPU_FORMAT_CSR || A->nnz == 0) return QBGPU_OK;
    unsigned long long *d_slots = nullptr;
    int *d_count = nullptr, *d_slot_code = nullptr;
    uint8_t *d_code = nullptr;
    double *d_dict = nullptr;
    auto cleanup = [&]() { cudaFree(d_slots); cudaFree(d_count); cudaFree(d_slot_code); };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); cudaFree(d_code); cudaFree(d_dict); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&d_slots, sizeof(unsigned long long) * kDictSlots));
    QB_CU(cudaMalloc(&d_count, sizeof(int)));
    QB_CU(cudaMemsetAsync(d_slots, 0xFF, sizeof(unsigned long long) * kDictSlots, c.stream));
    QB_CU(cudaMemsetAsync(d_count, 0, sizeof(int), c.stream));
    dict_collect_kernel<<<grid_for(A->nnz), kCBlock, 0, c.stream>>>(A->nnz, (const double *)A->val, d_slots, d_count);
    QB_LAUNCH_COUNT();
    std::vector<unsigned long long> slots(kDictSlots);
    int count = 0;
    QB_CU(cudaMemcpyAsync(slots.data(), d_slots, sizeof(unsigned long long) * kDictSlots, cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaMemcpyAsync(&count, d_count, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    QB_CU(cudaStreamSynchronize(c.stream));
    if (count > 256 || count > max_entries) { cleanup(); return QBGPU_OK; }      // not compressible: keep the fp64 values
    // order the dictionary by value so that the layout does not depend on thread timing
    std::vector<std::pair<double, int>> keys;
    for (int h = 0; h < kDictSlots; h++)
        if (slots[h] != kEmptyKey) { double v; memcpy(&v, &slots[h], 8); keys.push_back({v, h}); }
    std::sort(keys.begin(), keys.end(), [](const std::pair<double, int> &a, const std::pair<double, int> &b) { return value_table_less(a.first, b.first); });
    std::vector<int> slot_code(kDictSlots, 0);
    std::vector<double> dict(256, 0.0);
    for (size_t j = 0; j < keys.size(); j++) { dict[j] = keys[j].first; slot_code[keys[j].second] = (int)j; }
    QB_CU(cudaMalloc(&d_slot_code, sizeof(int) * kDictSlots));
    QB_CU(cudaMalloc(&d_dict, sizeof(double) * 256));
    QB_CU(cudaMalloc(&d_code, (size_t)A->nnz + 64));
    QB_CU(cudaMemcpyAsync(d_slot_code, slot_code.data(), sizeof(int) * kDictSlots, cudaMemcpyHostToDevice, c.stream));
    QB_CU(cudaMemcpyAsync(d_dict, dict.data(), sizeof(double) * 256, cudaMemcpyHostToDevice, c.stream));
    dict_encode_kernel<<<grid_for(A->nnz), kCBlock, 0, c.stream>>>(A->nnz, (const double *)A->val, d_slots, d_slot_code, d_code);
    QB_LAUNCH_COUNT();
    QB_CU(cudaStreamSynchronize(c.stream));
    QB_CU(cudaGetLastError());
    cleanup();
#undef QB_CU
    cudaFree(A->val);
    A->val = d_code;
    A->vdict = d_dict;
    A->ndict = (int)keys.size();
    return QBGPU_OK;
}

// ------------------------------------------------------------------------------------- split by column owner
// Multi-GPU pipelining (quantum_basis_b200/dist.py): a row shard is split into one block per column owner so that
// the block of rank p can be multiplied as soon as p's slice of x has arrived.  Columns are sorted inside a row, so
// every block is a contiguous sub-range of the row.
constexpr int kMaxParts = 16;
struct PartBounds { int64_t b[kMaxParts + 1]; };

__global__ void __launch_bounds__(kCBlock) split_count_kernel(int64_t nloc, const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                                                              int nparts, PartBounds pb, int64_t *len /* [nparts][nloc+1] */)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= nloc; i += (int64_t)gridDim.x * blockDim.x) {
        if (i == nloc) { for (int p = 0; p < nparts; p++) len[(int64_t)p * (nloc + 1) + i] = 0; continue; }
        int p = 0;
        int64_t cnt = 0;
        for (int64_t k = rowptr[i]; k < rowptr[i + 1]; k++) {
            const int64_t c = col[k];
            while (c >= pb.b[p + 1]) { len[(int64_t)p * (nloc + 1) + i] = cnt; cnt = 0; p++; }
            cnt++;
        }
        for (; p < nparts; p++) { len[(int64_t)p * (nloc + 1) + i] = cnt; cnt = 0; }
    }
}

template <typename ValT>
__global__ void __launch_bounds__(kCBlock) split_copy_kernel(int64_t nloc, const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                                                             const ValT *__restrict__ val, int part, int64_t lo, int64_t hi,
                                                             const int64_t *__restrict__ prow, int32_t *pcol, ValT *pval)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nloc; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t o = prow[i];
        for (int64_t k = rowptr[i]; k < rowptr[i + 1]; k++) {
            const int64_t c = col[k];
            if (c >= hi) break;
            if (c >= lo) { pcol[o] = (int32_t)c; pval[o] = val[k]; o++; }
        }
    }
}

int split_columns(qbgpu_matrix *A, int nparts, const int64_t *bounds, qbgpu_matrix_t *out, int flags)
{
    QB_TRY(ensure_init());
    Context &c = ctx();
    if (!A || !bounds || !out || nparts < 1 || nparts > kMaxParts) return fail(QBGPU_ERR_ARG, "split_columns: bad argument (1..16 parts)");
    if (bounds[0] != 0 || bounds[nparts] != A->n) return fail(QBGPU_ERR_ARG, "split_columns: bounds must run from 0 to n");
    for (int p = 0; p < nparts; p++) if (bounds[p + 1] < bounds[p]) return fail(QBGPU_ERR_ARG, "split_columns: bounds must be non-decreasing");
    if (A->ndict || A->mf || A->mf_sec) return fail(QBGPU_ERR_STATE, "split_columns: not available for dictionary-coded or matrix-free handles");
    const bool was_jagged = (A->format == QBGPU_FORMAT_SELL);
    QB_TRY(sjds_convert(A, false));                         // needs plain CSR order (restored below)
    const int64_t nloc = A->nrows();
    PartBounds pb;
    for (int p = 0; p <= nparts; p++) pb.b[p] = bounds[p];
    for (int p = nparts + 1; p <= kMaxParts; p++) pb.b[p] = A->n;
    for (int p = 0; p < nparts; p++) out[p] = nullptr;
    int64_t *d_len = nullptr;
    void *d_tmp = nullptr;
    auto cleanup = [&]() { cudaFree(d_len); cudaFree(d_tmp); };
    auto abort_all = [&]() { cleanup(); for (int p = 0; p < nparts; p++) { qbgpu_destroy(out[p]); out[p] = nullptr; } };
#define QB_CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { abort_all(); return cuda_fail(e_, #call, __FILE__, __LINE__); } } while (0)
    QB_CU(cudaMalloc(&d_len, sizeof(int64_t) * (size_t)nparts * (nloc + 1)));
    split_count_kernel<<<grid_for(nloc + 1), kCBlock, 0, c.stream>>>(nloc, A->rowptr, A->col, nparts, pb, d_len);
    QB_LAUNCH_COUNT();
    size_t tmp_bytes = 0;
    QB_CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_len, d_len, nloc + 1, c.stream));
    QB_CU(cudaMalloc(&d_tmp, tmp_bytes ? tmp_bytes : 1));
    for (int p = 0; p < nparts; p++) {
        auto *P = new qbgpu_matrix;
        out[p] = P;
        P->n = A->n; P->row_lo = A->row_lo; P->row_hi = A->row_hi; P->val_real = A->val_real; P->api_complex = A->api_complex;
        QB_CU(cudaMalloc(&P->rowptr, sizeof(int64_t) * (nloc + 1)));
        QB_CU(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_len + (int64_t)p * (nloc + 1), P->rowptr, nloc + 1, c.stream));
        int64_t nnz = 0;
        QB_CU(cudaMemcpyAsync(&nnz, P->rowptr + nloc, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
        QB_CU(cudaStreamSynchronize(c.stream));
        P->nnz = nnz; P->nnz_input = nnz;
        QB_CU(cudaMalloc(&P->col, sizeof(int32_t) * (nnz ? nnz : 1) + 64));
        QB_CU(cudaMalloc(&P->val, P->val_bytes() * (nnz ? nnz : 1) + 64));
        if (A->val_real) split_copy_kernel<double><<<grid_for(nloc), kCBlock, 0, c.stream>>>(nloc, A->rowptr, A->col, (const double *)A->val, p, bounds[p], bounds[p + 1], P->rowptr, P->col, (double *)P->val);
        else             split_copy_kernel<double2><<<grid_for(nloc), kCBlock, 0, c.stream>>>(nloc, A->rowptr, A->col, (const double2 *)A->val, p, bounds[p], bounds[p + 1], P->rowptr, P->col, (double2 *)P->val);
        QB_LAUNCH_COUNT();
        QB_CU(cudaStreamSynchronize(c.stream));
        QB_CU(cudaGetLastError());
    }
    cleanup();
#undef QB_CU
    if (was_jagged) QB_TRY(sjds_convert(A, true));
    for (int p = 0; p < nparts; p++) { int rc = autotune(out[p], flags); if (rc) { abort_all(); return rc; } }
    return QBGPU_OK;
}

}  // namespace qb

using namespace qb;

extern "C" {

int qbgpu_create_dcsr(qbgpu_matrix_t *A, int64_t n, const int64_t *rs, const int64_t *re, const int64_t *col,
                      const double *val, int sym, int flags)
{ return create_from_host<double>(A, n, rs, re, col, val, sym, flags, 0, -1, false); }

int qbgpu_create_zcsr(qbgpu_matrix_t *A, int64_t n, const int64_t *rs, const int64_t *re, const int64_t *col,
                      const void *val, int sym, int flags)
{ return create_from_host<double2>(A, n, rs, re, col, val, sym, flags, 0, -1, true); }

int qbgpu_create_dcsr_shard(qbgpu_matrix_t *A, int64_t n, const int64_t *rs, const int64_t *re, const int64_t *col,
                            const double *val, int sym, int flags, int64_t lo, int64_t hi)
{ return create_from_host<double>(A, n, rs, re, col, val, sym, flags, lo, hi, false); }

int qbgpu_create_zcsr_shard(qbgpu_matrix_t *A, int64_t n, const int64_t *rs, const int64_t *re, const int64_t *col,
                            const void *val, int sym, int flags, int64_t lo, int64_t hi)
{ return create_from_host<double2>(A, n, rs, re, col, val, sym, flags, lo, hi, true); }

int qbgpu_destroy(qbgpu_matrix_t A)
{
    if (!A) return QBGPU_OK;                               // like mkl_sparse_destroy on csr_mat's empty objects
    if (!A->borrowed) { matfree_destroy(A); sector_matfree_destroy(A); species_destroy(A); }
    if (!A->borrowed) { cudaFree(A->rowptr); cudaFree(A->col); cudaFree(A->val); cudaFree(A->rowinfo); cudaFree(A->vdict); cudaFree(A->slice_order);
                        cudaFree(A->perm_x); cudaFree(A->perm_y); }
    else if (A->owns_order) cudaFree(A->slice_order);
    delete A;
    return QBGPU_OK;
}

int qbgpu_matrix_get_info(qbgpu_matrix_t A, qbgpu_matrix_info *info)
{
    if (!A || !info) return fail(QBGPU_ERR_ARG, "null argument");
    info->n = A->n; info->row_lo = A->row_lo; info->row_hi = A->row_hi;
    info->nnz_stored = A->nnz + (A->second ? A->second->nnz : 0); info->nnz_input = A->nnz_input;
    info->val_is_real = A->val_real; info->value_dict = A->ndict; info->api_is_complex = A->api_complex;
    info->format = A->format; info->lanes = A->lanes;
    info->device_bytes = A->sp ? species_bytes(A) : A->mf ? matfree_bytes(A) : A->mf_sec ? (int64_t)sizeof(double) * 0 : (int64_t)(A->nnz * (4 + A->val_bytes()) + 8 * (A->nrows() + 1));
    info->upload_seconds = A->upload_s; info->convert_seconds = A->convert_s; info->autotune_seconds = A->autotune_s;
    return QBGPU_OK;
}

int qbgpu_download_expanded(qbgpu_matrix_t A, int64_t *rowptr, int32_t *col, void *val)
{
    QB_TRY(ensure_init());
    if (!A || !rowptr || !col || !val) return fail(QBGPU_ERR_ARG, "null argument");
    QB_TRY(no_species(A, "download_expanded"));
    if (A->mf || A->mf_sec) return fail(QBGPU_ERR_STATE, "matrix-free handle: there are no stored entries to download");
    if (A->cbits) return fail(QBGPU_ERR_STATE, "download_expanded: not available for packed entry words (a part of a species-order handle)");
    const bool jag = (A->format == QBGPU_FORMAT_SELL);      // hand back plain CSR order whatever the resident layout
    if (jag) QB_TRY(sjds_convert(A, false));
    QB_CUDA(cudaStreamSynchronize(ctx().stream));
    QB_CUDA(cudaMemcpy(rowptr, A->rowptr, sizeof(int64_t) * (A->nrows() + 1), cudaMemcpyDeviceToHost));
    QB_CUDA(cudaMemcpy(col, A->col, sizeof(int32_t) * A->nnz, cudaMemcpyDeviceToHost));
    if (A->ndict) {                                         // decode the 1-byte codes back to the fp64 values
        std::vector<uint8_t> codes(A->nnz);
        double dict[256];
        QB_CUDA(cudaMemcpy(codes.data(), A->val, (size_t)A->nnz, cudaMemcpyDeviceToHost));
        QB_CUDA(cudaMemcpy(dict, A->vdict, sizeof dict, cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < A->nnz; i++) ((double *)val)[i] = dict[codes[i]];
    } else {
        QB_CUDA(cudaMemcpy(val, A->val, A->val_bytes() * A->nnz, cudaMemcpyDeviceToHost));
    }
    if (jag) QB_TRY(sjds_convert(A, true));
    return QBGPU_OK;
}

int qbgpu_to_dense(qbgpu_matrix_t A, void *dense)
{
    // csr_mat<T>::to_dense (src/sparse.cc:299-315): res[row + col*dim]; only meant for tiny matrices (iram's
    // dim <= 30 fallback, src/lanczos.cc:508-542)
    QB_TRY(ensure_init());
    if (!A || !dense) return fail(QBGPU_ERR_ARG, "null argument");
    if (A->row_lo != 0 || A->row_hi != A->n) return fail(QBGPU_ERR_STATE, "to_dense needs an unsharded handle");
    QB_TRY(no_species(A, "to_dense"));
    const int64_t n = A->n;
    std::vector<int64_t> rp(n + 1);
    std::vector<int32_t> cc(A->nnz);
    std::vector<double> vv(A->nnz * (A->val_real ? 1 : 2));
    QB_TRY(qbgpu_download_expanded(A, rp.data(), cc.data(), vv.data()));
    const int nc = A->api_complex ? 2 : 1;
    double *D = (double *)dense;
    for (int64_t i = 0; i < n * n * nc; i++) D[i] = 0.0;
    for (int64_t r = 0; r < n; r++)
        for (int64_t p = rp[r]; p < rp[r + 1]; p++) {
            const int64_t at = (r + (int64_t)cc[p] * n) * nc;
            if (A->val_real) D[at] = vv[p]; else { D[at] = vv[2 * p]; D[at + 1] = vv[2 * p + 1]; }
        }
    return QBGPU_OK;
}

int qbgpu_real_view(qbgpu_matrix_t A, qbgpu_matrix_t *view)
{
    if (!A || !view) return fail(QBGPU_ERR_ARG, "null argument");
    if (!A->val_real) return fail(QBGPU_ERR_STATE, "real_view: the stored values are complex");
    auto *V = new qbgpu_matrix(*A);
    V->api_complex = false;
    V->borrowed = true;
    *view = V;
    return QBGPU_OK;
}

int qbgpu_split_columns(qbgpu_matrix_t A, int nparts, const int64_t *col_bounds, qbgpu_matrix_t *parts, int flags)
{
    if (A && A->sp) return species_split_columns(A, nparts, col_bounds, parts);   // matrix-free species shards: filtered views
    return split_columns(A, nparts, col_bounds, parts, flags);
}

int qbgpu_partition_rows(int64_t n, const int64_t *rs, const int64_t *re, const int64_t *col, int sym, int parts, int64_t *bounds)
{
    // host-only: expanded row lengths, then split the prefix sum into `parts` equal-nnz contiguous blocks
    if (n <= 0 || !rs || !re || !col || !bounds || parts < 1) return fail(QBGPU_ERR_ARG, "partition_rows: bad argument");
    std::vector<int64_t> len(n, 0);
    for (int64_t i = 0; i < n; i++)
        for (int64_t p = rs[i]; p < re[i]; p++) {
            const int64_t j = col[p];
            if (j < 0 || j >= n) return fail(QBGPU_ERR_ARG, "partition_rows: column index out of range");
            if (sym) { if (j < i) continue; len[i]++; if (j != i) len[j]++; } else len[i]++;
        }
    int64_t total = 0;
    for (int64_t i = 0; i < n; i++) total += len[i];
    bounds[0] = 0;
    int64_t acc = 0, i = 0;
    for (int p = 1; p < parts; p++) {
        const int64_t target = (int64_t)((__int128)total * p / parts);
        while (i < n && acc + len[i] <= target) { acc += len[i]; i++; }
        bounds[p] = i;
    }
    bounds[parts] = n;
    return QBGPU_OK;
}

}  // extern "C"
