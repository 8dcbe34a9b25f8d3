// Distance work of the GPU builder for SPARSE (csr) HNSW indices (pecos_b200/hnsw_build.py, DESIGN §4.4).
//
// Every distance here has the reference's exact bits: FeatVecSparse{IP,L2}Simd::distance is the ordered sum (ascending
// feature index, unfused -- the library is compiled with -fmad=false -- starting from +0.0f) of the matched products, turned
// into ip = (float)(1.0 - dot) or l2 = (float)(0.0 - 2.0 * dot) (the reference's sparse l2 takes |x|^2 as the distance of x to
// itself, which is 0).  Orders are by (float distance, id).
//
//   hb_sparse_knn_kernel     exact prefix kNN: for every row q of a level, the k nearest rows c < q.  Gustavson-style SpGEMM
//                            over the level's posting lists: one warp per query walks q's features in ascending order and,
//                            per feature, adds x_q,f * x_c,f for the posting entries c < q into per-candidate accumulators.
//                            The candidates are swept in blocks of KNN_BLOCK whose accumulators live in shared memory; a
//                            per-(q, feature) cursor into the posting list advances monotonically across the blocks, so the
//                            whole posting prefix of q is read once.  Within one feature the candidates are distinct (no
//                            conflicts), features are processed in order (each (q, c) sum is the reference's ordered sum),
//                            no atomics: deterministic.  After each block the warp scans the accumulators in ascending id
//                            order into a sorted running top-k of (orderable(distance) << 32 | position) keys.
//   hb_sparse_select_kernel  the reference's neighbour-selection heuristic (hnsw.hpp:556-592), one warp per node: candidates
//                            in ascending (distance, id) order; lane t computes the distance of candidate j to kept neighbour
//                            t by an ordered merge of the two rows; j is rejected if any is < its distance to the node.
#include "../../include/pecos_b200.h"

#include <cstdint>
#include <cstdio>

#include "cuda_util.h"

namespace {

constexpr uint32_t FULL = 0xffffffffu;
constexpr uint32_t KNN_BLOCK = 2048;  // candidate accumulators per warp (8 KB of shared memory)
constexpr uint32_t KNN_WARPS = 4;     // warps (= queries) per CTA
constexpr uint32_t SEL_WARPS = 8;
constexpr unsigned long long KEY_SIGN = 1ull << 63;  // keys leave the kernel sign-flipped: signed int64 order = key order

__device__ __forceinline__ float dist_from_dot(float dot, int metric) {
    const double r = metric == 0 ? 1.0 - static_cast<double>(dot) : 0.0 - 2.0 * static_cast<double>(dot);
    return static_cast<float>(r);
}

// monotone map float -> u32 (-0.0 and +0.0 compare equal as floats, so they map to one value)
__device__ __forceinline__ uint32_t orderable(float d) {
    const uint32_t u = __float_as_uint(d == 0.0f ? 0.0f : d);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ float row_distance(uint32_t a, uint32_t b, int metric, const int64_t* __restrict__ row_ptr,
                                              const int32_t* __restrict__ col, const float* __restrict__ val) {
    int64_t i = row_ptr[a], j = row_ptr[b];
    const int64_t ie = row_ptr[a + 1], je = row_ptr[b + 1];
    float dot = 0.0f;
    while (i < ie && j < je) {
        const int32_t ca = col[i], cb = col[j];
        if (ca < cb) {
            ++i;
        } else if (cb < ca) {
            ++j;
        } else {
            const float p = val[i] * val[j];
            dot = dot + p;
            ++i;
            ++j;
        }
    }
    return dist_from_dot(dot, metric);
}

// Insert `key` (known to belong in the top-k) into the warp's ascending list lk[0..cnt) (ldot: the keys' dot products).
__device__ __forceinline__ void topk_insert(unsigned long long* lk, float* ldot, uint32_t cnt, uint32_t k, unsigned long long key,
                                            float dot, uint32_t lane) {
    uint32_t pos = 0;
    for (uint32_t j0 = 0; j0 < cnt; j0 += 32) {
        const uint32_t j = j0 + lane;
        pos += __popc(__ballot_sync(FULL, j < cnt && lk[j] < key));
    }
    const uint32_t last = cnt < k ? cnt : k - 1;  // entries [pos, last) move up by one; the k-th falls off when full
    for (int64_t top = last; top > static_cast<int64_t>(pos); top -= 32) {
        const int64_t j = top - 32 + lane;
        const bool mv = j >= static_cast<int64_t>(pos) && j < top;
        unsigned long long a = 0;
        float b = 0.0f;
        if (mv) { a = lk[j]; b = ldot[j]; }
        __syncwarp();
        if (mv) { lk[j + 1] = a; ldot[j + 1] = b; }
        __syncwarp();
    }
    if (lane == 0) { lk[pos] = key; ldot[pos] = dot; }
    __syncwarp();
}

__global__ void __launch_bounds__(KNN_WARPS * 32)
hb_sparse_knn_kernel(uint32_t n, uint32_t k, int metric, const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                     const float* __restrict__ val, const int64_t* __restrict__ post_ptr, const int2* __restrict__ post,
                     const int64_t* __restrict__ self_pos, int64_t* __restrict__ cursor, long long* __restrict__ out_keys) {
    extern __shared__ __align__(16) unsigned char smem[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * KNN_WARPS + warp;
    if (gw >= n) return;
    const uint32_t q = n - 1 - gw;  // the longest prefixes start first
    float* acc = reinterpret_cast<float*>(smem) + warp * KNN_BLOCK;
    unsigned long long* lk = reinterpret_cast<unsigned long long*>(smem + KNN_WARPS * KNN_BLOCK * 4) + warp * k;
    float* ldot = reinterpret_cast<float*>(smem + KNN_WARPS * KNN_BLOCK * 4 + KNN_WARPS * k * 8) + warp * k;

    const int64_t e0 = row_ptr[q], e1 = row_ptr[q + 1];
    for (int64_t e = e0 + lane; e < e1; e += 32) cursor[e] = post_ptr[col[e]];
    __syncwarp();

    uint32_t cnt = 0;
    float kth_dot = 0.0f;
    for (uint32_t c0 = 0; c0 < q; c0 += KNN_BLOCK) {
        const uint32_t nc = min(KNN_BLOCK, q - c0), cend = c0 + nc;
        for (uint32_t i = lane; i < nc; i += 32) acc[i] = 0.0f;
        __syncwarp();
        // products, feature by feature in ascending index order: the (q, c) sums are the reference's ordered sums
        for (int64_t e = e0; e < e1; ++e) {
            const float xq = val[e];
            const int64_t end = self_pos[e];  // q's own entry: everything before it in the list has a row < q
            int64_t s = cursor[e];
            while (s < end) {
                const int64_t p = s + lane;
                int2 ent = make_int2(0, 0);
                bool ok = false;
                if (p < end) {
                    ent = post[p];
                    ok = static_cast<uint32_t>(ent.x) < cend;
                }
                const uint32_t m = __ballot_sync(FULL, ok);  // rows ascend along the list: the hits are a prefix
                if (ok) {
                    const float prod = xq * __int_as_float(ent.y);
                    acc[ent.x - c0] = acc[ent.x - c0] + prod;
                }
                __syncwarp();
                s += __popc(m);
                if (m != FULL) break;
            }
            __syncwarp();
            if (lane == 0) cursor[e] = s;
        }
        __syncwarp();
        // selection: ascending id order, so a candidate whose distance ties the current k-th loses to it.  Distances are
        // non-increasing in the dot product, so dot <= (k-th's dot) can never enter a full list.
        for (uint32_t i0 = 0; i0 < nc; i0 += 32) {
            const uint32_t i = i0 + lane;
            float dot = 0.0f;
            bool want = false;
            if (i < nc) {
                dot = acc[i];
                want = cnt < k || dot > kth_dot;
            }
            uint32_t m = __ballot_sync(FULL, want);
            while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const float d = __shfl_sync(FULL, dot, src);
                if (cnt == k && !(d > kth_dot)) continue;
                const unsigned long long key =
                    (static_cast<unsigned long long>(orderable(dist_from_dot(d, metric))) << 32) | (c0 + i0 + src);
                if (cnt == k && key >= lk[k - 1]) continue;
                topk_insert(lk, ldot, cnt, k, key, d, lane);
                if (cnt < k) ++cnt;
                if (cnt == k) kth_dot = ldot[k - 1];
            }
        }
        __syncwarp();
    }
    long long* out = out_keys + static_cast<size_t>(q) * k;
    for (uint32_t j = lane; j < k; j += 32)
        out[j] = j < cnt ? static_cast<long long>(lk[j] ^ KEY_SIGN) : static_cast<long long>(~0ull ^ KEY_SIGN);
}

__global__ void __launch_bounds__(SEL_WARPS * 32)
hb_sparse_select_kernel(uint32_t n, uint32_t C, uint32_t cap, int metric, const int64_t* __restrict__ row_ptr,
                        const int32_t* __restrict__ col, const float* __restrict__ val, const int64_t* __restrict__ cand,
                        const float* __restrict__ cand_d, uint8_t* __restrict__ keep) {
    extern __shared__ __align__(16) unsigned char smem[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t r = blockIdx.x * SEL_WARPS + warp;
    if (r >= n) return;
    uint32_t* kept = reinterpret_cast<uint32_t*>(smem) + warp * cap;
    const int64_t* cr = cand + static_cast<size_t>(r) * C;
    const float* dr = cand_d + static_cast<size_t>(r) * C;
    uint8_t* out = keep + static_cast<size_t>(r) * C;
    uint32_t valid = 0;
    for (uint32_t j0 = 0; j0 < C; j0 += 32) valid += __popc(__ballot_sync(FULL, j0 + lane < C && cr[j0 + lane] >= 0));
    if (valid < cap) {  // fewer candidates than the capacity: all are kept (hnsw.hpp:562-565)
        for (uint32_t j = lane; j < C; j += 32) out[j] = cr[j] >= 0;
        return;
    }
    uint32_t nk = 0;
    for (uint32_t j = 0; j < C; ++j) {
        const int64_t c = cr[j];
        bool kp = false;
        if (c >= 0 && nk < cap) {
            const float dq = dr[j];
            bool bad = false;
            for (uint32_t t = lane; t < nk; t += 32)
                bad |= row_distance(static_cast<uint32_t>(c), kept[t], metric, row_ptr, col, val) < dq;
            kp = !__any_sync(FULL, bad);
        }
        if (lane == 0) out[j] = kp;
        if (kp) {
            if (lane == 0) kept[nk] = static_cast<uint32_t>(c);
            ++nk;
            __syncwarp();
        }
    }
}

int report(const char* where, cudaError_t err) {
    if (err == cudaSuccess) return 0;
    std::fprintf(stderr, "pecos_b200: %s: %s\n", where, cudaGetErrorString(err));
    return 1;
}

}  // namespace

extern "C" {

int pb200_hnsw_build_sparse_knn(int device, void* stream, uint32_t n, uint32_t k, int metric, const void* row_ptr,
                                const void* col_idx, const void* val, const void* post_ptr, const void* post_entries,
                                const void* self_pos, void* cursor, void* out_keys) {
    if (n == 0 || k == 0) return 0;
    if (int rc = report("cudaSetDevice", cudaSetDevice(device))) return rc;
    const size_t smem = static_cast<size_t>(KNN_WARPS) * (KNN_BLOCK * 4 + static_cast<size_t>(k) * 12);
    if (int rc = report("cudaFuncSetAttribute(hb_sparse_knn_kernel)",
                        cudaFuncSetAttribute(hb_sparse_knn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(smem))))
        return rc;
    const uint32_t grid = (n + KNN_WARPS - 1) / KNN_WARPS;
    hb_sparse_knn_kernel<<<grid, KNN_WARPS * 32, smem, static_cast<cudaStream_t>(stream)>>>(
        n, k, metric, static_cast<const int64_t*>(row_ptr), static_cast<const int32_t*>(col_idx), static_cast<const float*>(val),
        static_cast<const int64_t*>(post_ptr), static_cast<const int2*>(post_entries), static_cast<const int64_t*>(self_pos),
        static_cast<int64_t*>(cursor), static_cast<long long*>(out_keys));
    return report("hb_sparse_knn_kernel launch", cudaGetLastError());
}

int pb200_hnsw_build_sparse_select(int device, void* stream, uint32_t n, uint32_t C, uint32_t cap, int metric,
                                   const void* row_ptr, const void* col_idx, const void* val, const void* cand,
                                   const void* cand_d, void* keep) {
    if (n == 0 || C == 0) return 0;
    if (int rc = report("cudaSetDevice", cudaSetDevice(device))) return rc;
    const size_t smem = static_cast<size_t>(SEL_WARPS) * cap * 4;
    if (int rc = report("cudaFuncSetAttribute(hb_sparse_select_kernel)",
                        cudaFuncSetAttribute(hb_sparse_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(smem))))
        return rc;
    const uint32_t grid = (n + SEL_WARPS - 1) / SEL_WARPS;
    hb_sparse_select_kernel<<<grid, SEL_WARPS * 32, smem, static_cast<cudaStream_t>(stream)>>>(
        n, C, cap, metric, static_cast<const int64_t*>(row_ptr), static_cast<const int32_t*>(col_idx),
        static_cast<const float*>(val), static_cast<const int64_t*>(cand), static_cast<const float*>(cand_d),
        static_cast<uint8_t*>(keep));
    return report("hb_sparse_select_kernel launch", cudaGetLastError());
}

}  // extern "C"
