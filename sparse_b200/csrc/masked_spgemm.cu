// masked_spgemm.cu -- K10: the masked sparse product s * (a @ b) for sparse s, a, b, without forming a @ b.
//
// Replaces the unfused `s * (a @ b)` (K4 product + K5 merge) of examples/triangles_example.py (`sum(a @ a * a)`),
// masked SpGEMM (GraphBLAS C<M> = A.B), and edge scores on graphs.  Only the entries of s are computed:
//   out[p] = (TO)s[p] * (TO)acc(i, j),   acc(i, j) = ((+0 + a[i,k1]*b[k1,j]) + a[i,k2]*b[k2,j]) + ...
// over the k where both a[i,k] and b[k,j] are stored, in ascending k (the reference's visiting order of
// _dot_csr_csr / _dot_coo_coo for operands with sorted rows); every product and every sum is rounded on its own.
//
// Dot (intersection) form: a warp owns a task of MS_TASK consecutive mask entries (tasks dealt out by a global
// ticket, so a hub row of the mask is shared by many warps), walks the mask rows the task touches, stages A[i,:]
// (indices + values) in shared memory once per row (rows longer than the stage are searched in global memory / L2)
// and, for each mask entry (i, j), intersects A[i,:] with Bt[j,:] (= column j of b): lanes take 32 entries of the
// shorter list at a time and binary-search them in the longer one.  Both lists are sorted, so the matches of a chunk
// come out in ascending k; a ballot of the matching lanes is then summed bit by bit in lane order (never a tree), which
// keeps the reference's rounding.  Integer sums wrap (exact in any order); bool is OR of ANDs, the `+=` of the
// reference's bool `sums` array.
#include <type_traits>

#include "common.cuh"

namespace b2s {

constexpr unsigned MS_FULL = 0xffffffffu;
constexpr int MS_WARPS = 4;     // warps per CTA
constexpr int MS_STAGE = 512;   // entries of A[i,:] staged per warp
constexpr int MS_TASK = 128;    // mask entries per ticket

template <typename T>
__device__ __forceinline__ T ms_mul(T a, T b) {
    if constexpr (std::is_same<T, bool>::value) return a && b;
    else return mul_rn(a, b);
}
template <typename T>
__device__ __forceinline__ T ms_add(T a, T b) {
    if constexpr (std::is_same<T, bool>::value) return a || b;
    else return add_rn(a, b);
}
template <typename T>
__device__ __forceinline__ T ms_shfl(T v, int src) {
    if constexpr (std::is_same<T, bool>::value) return __shfl_sync(MS_FULL, (int)v, src) != 0;
    else return __shfl_sync(MS_FULL, v, src);
}

// first position in y[0, n) whose value is >= k
template <typename I>
__device__ __forceinline__ int64_t ms_lower_bound(const I *y, int64_t n, I k) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (y[mid] < k) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

template <typename TA, typename TO, typename I>
__global__ void __launch_bounds__(MS_WARPS * 32)
masked_spgemm_kernel(int64_t M, const I *__restrict__ s_indptr, const I *__restrict__ s_cols,
                     const TO *__restrict__ s_vals, const I *__restrict__ a_indptr, const I *__restrict__ a_idx,
                     const TA *__restrict__ a_val, const I *__restrict__ bt_indptr, const I *__restrict__ bt_idx,
                     const TA *__restrict__ bt_val, TO *__restrict__ out, unsigned long long *__restrict__ ticket) {
    __shared__ I s_ai[MS_WARPS][MS_STAGE];
    __shared__ TA s_av[MS_WARPS][MS_STAGE];
    const int lane = threadIdx.x & 31;
    const int w = threadIdx.x >> 5;
    const int64_t nnz = (int64_t)s_indptr[M];
    const int64_t ntask = (nnz + MS_TASK - 1) / MS_TASK;
    int64_t staged = -1;  // mask row whose A row is in s_ai / s_av
    for (;;) {
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(ticket, 1ull);
        t = __shfl_sync(MS_FULL, t, 0);
        if ((int64_t)t >= ntask) break;
        const int64_t e0 = (int64_t)t * MS_TASK;
        const int64_t e1 = min(e0 + (int64_t)MS_TASK, nnz);
        // the mask row holding entry e0: s_indptr[row] <= e0 < s_indptr[row + 1]
        int64_t lo = 0, hi = M;
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if ((int64_t)s_indptr[mid] <= e0) lo = mid;
            else hi = mid;
        }
        int64_t p = e0;
        for (int64_t row = lo; p < e1; ++row) {
            const int64_t rend = min((int64_t)s_indptr[row + 1], e1);
            if (rend <= p) continue;  // empty mask row
            const int64_t as = (int64_t)a_indptr[row];
            const int64_t la = (int64_t)a_indptr[row + 1] - as;
            const I *ai = a_idx + as;
            const TA *av = a_val + as;
            if (la <= MS_STAGE) {
                if (staged != row) {
                    __syncwarp();  // every lane is done with the previous row's stage
                    for (int64_t q = lane; q < la; q += 32) {
                        s_ai[w][q] = ai[q];
                        s_av[w][q] = av[q];
                    }
                    __syncwarp();
                    staged = row;
                }
                ai = &s_ai[w][0];
                av = &s_av[w][0];
            }
            for (; p < rend; ++p) {
                const I j = s_cols[p];
                const int64_t bs = (int64_t)bt_indptr[j];
                const int64_t lb = (int64_t)bt_indptr[j + 1] - bs;
                TA acc = TA(0);
                if (la > 0 && lb > 0) {
                    // walk the shorter list, search the longer one
                    const bool walk_a = la <= lb;
                    const I *xi = walk_a ? ai : bt_idx + bs;
                    const TA *xv = walk_a ? av : bt_val + bs;
                    const int64_t lx = walk_a ? la : lb;
                    const I *yi = walk_a ? bt_idx + bs : ai;
                    const TA *yv = walk_a ? bt_val + bs : av;
                    const int64_t ly = walk_a ? lb : la;
                    for (int64_t base = 0; base < lx; base += 32) {
                        const int64_t q = base + lane;
                        bool hit = false;
                        TA prod = TA(0);
                        if (q < lx) {
                            const I k = xi[q];
                            const int64_t pos = ms_lower_bound(yi, ly, k);
                            if (pos < ly && yi[pos] == k) {
                                hit = true;
                                prod = ms_mul(xv[q], yv[pos]);
                            }
                        }
                        // ordered accumulation: the matches of this chunk in lane (= ascending k) order
                        unsigned m = __ballot_sync(MS_FULL, hit);
                        while (m) {
                            const int src = __ffs(m) - 1;
                            acc = ms_add(acc, ms_shfl(prod, src));
                            m &= m - 1;
                        }
                    }
                }
                if (lane == 0) out[p] = ms_mul(s_vals[p], (TO)acc);
            }
        }
    }
}

template <typename TA, typename TO, typename I>
static int masked_spgemm_launch(int64_t M, const void *sp, const void *sc, const void *sv, const void *ap,
                                const void *ai, const void *av, const void *bp, const void *bi, const void *bv,
                                void *out, cudaStream_t s) {
    auto kern = masked_spgemm_kernel<TA, TO, I>;
    int occ = 1;
    B2S_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, MS_WARPS * 32, 0));
    const int64_t blocks = (int64_t)num_sms() * (occ < 1 ? 1 : occ);
    unsigned long long *ticket = nullptr;
    int rc = scratch_alloc((void **)&ticket, sizeof(unsigned long long), s);
    if (rc != B2S_OK) return rc;
    B2S_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned long long), s));
    kern<<<(unsigned)blocks, MS_WARPS * 32, 0, s>>>(M, (const I *)sp, (const I *)sc, (const TO *)sv, (const I *)ap,
                                                    (const I *)ai, (const TA *)av, (const I *)bp, (const I *)bi,
                                                    (const TA *)bv, (TO *)out, ticket);
    B2S_CHECK_LAUNCH();
    return scratch_free(ticket, s);
}

}  // namespace b2s

using namespace b2s;

extern "C" {

/*
 * Masked sparse product (K10): out_vals[p] = s_vals[p] * sum_k A[i_p, k] * Bt[j_p, k] for every stored (i_p, j_p) of
 * the mask.  S (M x N), A (M x K) and Bt (N x K, b compressed by column) are CSR with sorted, duplicate-free rows.
 */
int b2s_masked_spgemm(int dtype_ab, int dtype_out, int idx_bytes, int64_t M, int64_t N, int64_t K,
                      const void *s_indptr_dev, const void *s_cols_dev, const void *s_vals_dev,
                      const void *a_indptr_dev, const void *a_indices_dev, const void *a_data_dev,
                      const void *bt_indptr_dev, const void *bt_indices_dev, const void *bt_data_dev,
                      void *out_vals_dev, void *stream) {
    B2S_REQUIRE(idx_bytes == 4 || idx_bytes == 8, B2S_ERR_INVALID, "masked_spgemm: idx_bytes");
    B2S_REQUIRE(M >= 0 && N >= 0 && K >= 0, B2S_ERR_INVALID, "masked_spgemm: negative dimension");
    if (M == 0) return B2S_OK;
    cudaStream_t s = (cudaStream_t)stream;
#define B2S_MS(TA, TO)                                                                                           \
    return idx_bytes == 4                                                                                        \
               ? masked_spgemm_launch<TA, TO, int32_t>(M, s_indptr_dev, s_cols_dev, s_vals_dev, a_indptr_dev,    \
                                                       a_indices_dev, a_data_dev, bt_indptr_dev, bt_indices_dev, \
                                                       bt_data_dev, out_vals_dev, s)                             \
               : masked_spgemm_launch<TA, TO, int64_t>(M, s_indptr_dev, s_cols_dev, s_vals_dev, a_indptr_dev,    \
                                                       a_indices_dev, a_data_dev, bt_indptr_dev, bt_indices_dev, \
                                                       bt_data_dev, out_vals_dev, s)
    // the (product, result) dtype pairs the host produces: floats as they are, integers computed in int64 (wrapping,
    // cast back on the host), bool products with any result type
    if (dtype_ab == B2S_F32 && dtype_out == B2S_F32) B2S_MS(float, float);
    if (dtype_ab == B2S_F32 && dtype_out == B2S_F64) B2S_MS(float, double);
    if (dtype_ab == B2S_F64 && dtype_out == B2S_F64) B2S_MS(double, double);
    if (dtype_ab == B2S_I64 && dtype_out == B2S_I64) B2S_MS(int64_t, int64_t);
    if (dtype_ab == B2S_I64 && dtype_out == B2S_F64) B2S_MS(int64_t, double);
    if (dtype_ab == B2S_BOOL && dtype_out == B2S_BOOL) B2S_MS(bool, bool);
    if (dtype_ab == B2S_BOOL && dtype_out == B2S_I64) B2S_MS(bool, int64_t);
    if (dtype_ab == B2S_BOOL && dtype_out == B2S_F32) B2S_MS(bool, float);
    if (dtype_ab == B2S_BOOL && dtype_out == B2S_F64) B2S_MS(bool, double);
#undef B2S_MS
    set_error("masked_spgemm: dtype pair (%d, %d) is outside the kernel's dtype matrix", dtype_ab, dtype_out);
    return B2S_ERR_UNSUPPORTED;
}

}  // extern "C"
