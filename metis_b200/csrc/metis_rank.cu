// Ordering of the candidate records on the device (SURVEY.md 8(f)-2).
//
// metis_het_search appends its 16-byte records in completion order.  The reference's list
// `estimate_costs` (cost_het_cluster.py:44) is in (inter-stage plan, chain step) order and its ranked
// listing is `sorted(estimate_costs, key=cost)` (cost_het_cluster.py:76) - a STABLE sort, so equal costs keep
// their estimate_costs order.  Both orders are produced here by one cooperative kernel: a stable
// least-significant-digit radix sort, 8 bits per pass, over the key
//     (ordinal : 32, step : 16)                       6 passes  -> estimate_costs order
//     then the order-preserving image of the fp64 cost  8 passes  -> ranked order (ties keep position order)
// Each warp owns a contiguous chunk of the array: it counts its digits, a grid-wide scan turns the
// counts into global offsets, and the warp scatters its chunk in order (ranks inside a 32-element tile
// from __match_any_sync), which is what keeps every pass stable.  Passes whose digit is the same for all
// records (high bytes of small ordinals, steps < 256, shared exponent bytes) are detected after the
// count and skipped.  The work is byte shuffling bound by HBM/L2 bandwidth; for the 2.7e5 records of
// BASELINE configs[2] it is tens of microseconds per pass.
//
// The k first records of the ranked order (metis_select_records) come from a radix SELECT over the same key, most
// significant byte first, which reads the records a few times but orders only the k it keeps.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>

#include "../../include/metis_b200.h"
#include "metis_internal.h"

namespace cg = cooperative_groups;

namespace metis {

constexpr int kRankThreads = 256;
constexpr int kRankWarps = kRankThreads / 32;

struct RankArgs {
    uint4 *a, *b;             // records (16 B each): a = caller's array, b = scratch
    uint32_t *ia, *ib;        // original index travelling with each record
    long long n;
    unsigned int *hist;       // [256][warps]
    unsigned int *bintot;     // [256]
    int pass_begin, pass_end; // passes 0-5 sort by position, 6-13 by cost
    uint32_t *perm_out;       // optional
};

// The 112-bit ranking key of a record: hi = order-preserving image of the fp64 cost, lo = position (ordinal : 32,
// step : 16).  Unsigned comparison of (hi, lo) is the order of METIS_SORT_RANKED; both the sort and the selection
// below read records only through this function.
struct RecordKey {
    unsigned long long hi, lo;
};

__device__ __forceinline__ RecordKey key_of(const uint4 &r) {
    // r.x, r.y = cost bits (lo, hi); r.z = ordinal; r.w = step | num_repartition << 16 | num_stage << 24
    unsigned long long u = ((unsigned long long)r.y << 32) | r.x;
    u ^= (u >> 63) ? ~0ULL : 0x8000000000000000ULL;      // total order of the doubles (no NaN reaches here)
    return RecordKey{u, ((unsigned long long)r.z << 16) | (r.w & 0xFFFFu)};
}

// byte `pass` of the key, least significant first: passes 0-5 are the position, 6-13 the cost image
__device__ __forceinline__ unsigned int digit_of(const uint4 &r, int pass) {
    const RecordKey key = key_of(r);
    return (unsigned int)(pass < 6 ? key.lo >> (8 * pass) : key.hi >> (8 * (pass - 6))) & 0xFFu;
}

__global__ void __launch_bounds__(kRankThreads) rank_records_kernel(RankArgs q) {
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned int bins[kRankWarps][256];
    __shared__ unsigned int sbase[256];
    __shared__ unsigned int sscan[kRankWarps];
    __shared__ int s_skip;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long nwarps = (long long)gridDim.x * kRankWarps;
    const long long gw = (long long)blockIdx.x * kRankWarps + wib;
    const long long n = q.n;
    long long chunk = (n + nwarps - 1) / nwarps;
    chunk = (chunk + 31) / 32 * 32;
    const long long lo = gw * chunk < n ? gw * chunk : n;
    const long long hi = lo + chunk < n ? lo + chunk : n;
    const unsigned full = 0xFFFFFFFFu;
    const unsigned lt = (1u << lane) - 1u;

    for (long long i = (long long)blockIdx.x * kRankThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kRankThreads)
        q.ia[i] = (uint32_t)i;
    uint4 *src = q.a, *dst = q.b;
    uint32_t *isrc = q.ia, *idst = q.ib;
    grid.sync();

    for (int pass = q.pass_begin; pass < q.pass_end; ++pass) {
        // ---- count -------------------------------------------------------------------------------
        for (int d = lane; d < 256; d += 32) bins[wib][d] = 0;
        __syncwarp();
        for (long long t = lo; t < hi; t += 32) {
            const long long i = t + lane;
            const int d = i < hi ? (int)digit_of(src[i], pass) : -1;
            const unsigned peers = __match_any_sync(full, d);
            if (d >= 0 && lane == __ffs(peers) - 1) bins[wib][d] += __popc(peers);
            __syncwarp();
        }
        for (int d = lane; d < 256; d += 32) q.hist[(long long)d * nwarps + gw] = bins[wib][d];
        grid.sync();
        // ---- scan: rows (one digit over all warps), then the 256 digit totals -----------------------
        for (long long d = gw; d < 256; d += nwarps) {
            unsigned int *row = q.hist + d * nwarps;
            unsigned int run = 0;
            for (long long c = 0; c < nwarps; c += 32) {
                const unsigned int v = c + lane < nwarps ? row[c + lane] : 0;
                unsigned int inc = v;
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned int up = __shfl_up_sync(full, inc, o);
                    if (lane >= o) inc += up;
                }
                if (c + lane < nwarps) row[c + lane] = run + inc - v;
                run += __shfl_sync(full, inc, 31);
            }
            if (lane == 0) q.bintot[d] = run;
        }
        grid.sync();
        {
            const unsigned int v = threadIdx.x < 256 ? *(volatile unsigned int *)&q.bintot[threadIdx.x] : 0;
            if (threadIdx.x == 0) s_skip = 0;
            __syncthreads();
            if (threadIdx.x < 256 && (long long)v == n) s_skip = 1;        // every record has this digit
            unsigned int inc = v;
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int up = __shfl_up_sync(full, inc, o);
                if (lane >= o) inc += up;
            }
            if (lane == 31) sscan[wib] = inc;
            __syncthreads();
            unsigned int before = 0;
            for (int k = 0; k < wib; ++k) before += sscan[k];
            if (threadIdx.x < 256) sbase[threadIdx.x] = before + inc - v;
            __syncthreads();
        }
        if (s_skip) { __syncthreads(); continue; }              // same decision in every block: nothing to move
        // ---- scatter, chunk order preserved ----------------------------------------------------------
        for (int d = lane; d < 256; d += 32) bins[wib][d] = sbase[d] + q.hist[(long long)d * nwarps + gw];
        __syncwarp();
        for (long long t = lo; t < hi; t += 32) {
            const long long i = t + lane;
            uint4 r = make_uint4(0, 0, 0, 0);
            uint32_t id = 0;
            int d = -1;
            if (i < hi) { r = src[i]; id = isrc[i]; d = (int)digit_of(r, pass); }
            const unsigned peers = __match_any_sync(full, d);
            unsigned int base = 0;
            if (d >= 0) base = bins[wib][d];
            __syncwarp();
            if (d >= 0) {
                if (lane == __ffs(peers) - 1) bins[wib][d] = base + __popc(peers);
                const unsigned int to = base + __popc(peers & lt);
                dst[to] = r;
                idst[to] = id;
            }
            __syncwarp();
        }
        { uint4 *t = src; src = dst; dst = t; }
        { uint32_t *t = isrc; isrc = idst; idst = t; }
        grid.sync();
    }
    // ---- results into the caller's arrays ----------------------------------------------------------------
    for (long long i = (long long)blockIdx.x * kRankThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kRankThreads) {
        if (src != q.a) q.a[i] = src[i];
        if (q.perm_out) q.perm_out[i] = isrc[i];
    }
}

// ---- selection of the k smallest keys (most-significant-digit radix select) ------------------------------------
// Pass after pass, every block counts the next key byte (most significant first) of the records whose key matches
// the prefix decided so far, and merges its histogram into a global one.  After a grid-wide barrier every block
// reads the same merged histogram and takes the same decision: the byte in which the remaining rank falls extends
// the prefix.  The walk stops when that byte's bucket is taken whole, or when the key runs out (records with equal
// keys: the first ones in input order are taken, as a stable sort would).  A last pass writes the min(k, n)
// selected records in input order; metis_sort_records then ranks only those.
constexpr int kKeyDigits = 14;
static_assert(kRankThreads == 256, "one thread per digit value in the decision step");

struct SelectArgs {
    const uint4 *in;
    long long n, k;
    uint4 *out;               // min(k, n) selected records, input order
    uint32_t *idx;            // their input positions
    unsigned int *hist;       // [kKeyDigits][256]
    unsigned long long *wcount;   // [2][warps]: records below the threshold / inside its bucket, per warp
};

__global__ void __launch_bounds__(kRankThreads) select_records_kernel(SelectArgs q) {
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned int bins[256];
    __shared__ unsigned int sscan[kRankWarps];
    __shared__ unsigned long long s_phi, s_plo, s_mhi, s_mlo;   // decided prefix of (hi, lo) and its bit mask
    __shared__ unsigned long long s_rem;                        // records still to take from the prefix's bucket
    __shared__ unsigned long long s_before, s_count;
    __shared__ unsigned int s_digit;
    __shared__ int s_whole;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long nwarps = (long long)gridDim.x * kRankWarps;
    const long long gw = (long long)blockIdx.x * kRankWarps + wib;
    const long long n = q.n;
    const unsigned full = 0xFFFFFFFFu;
    const unsigned lt = (1u << lane) - 1u;

    for (long long i = (long long)blockIdx.x * kRankThreads + threadIdx.x; i < kKeyDigits * 256; i += (long long)gridDim.x * kRankThreads)
        q.hist[i] = 0;
    if (threadIdx.x == 0) {
        s_phi = s_plo = s_mhi = s_mlo = 0;
        s_rem = (unsigned long long)q.k;
        s_whole = q.k >= n;                                     // everything: the empty prefix, taken whole
    }
    grid.sync();

    for (int depth = 0; !s_whole && depth < kKeyDigits; ++depth) {
        const int pass = kKeyDigits - 1 - depth;
        const unsigned long long phi = s_phi, plo = s_plo, mhi = s_mhi, mlo = s_mlo, rem = s_rem;
        bins[threadIdx.x] = 0;
        __syncthreads();
        for (long long t = gw * 32; t < n; t += nwarps * 32) {
            const long long i = t + lane;
            int d = -1;
            if (i < n) {
                const uint4 r = q.in[i];
                const RecordKey key = key_of(r);
                if ((key.hi & mhi) == phi && (key.lo & mlo) == plo) d = (int)digit_of(r, pass);
            }
            const unsigned peers = __match_any_sync(full, d);
            if (d >= 0 && lane == __ffs(peers) - 1) atomicAdd(&bins[d], (unsigned int)__popc(peers));
        }
        __syncthreads();
        if (bins[threadIdx.x]) atomicAdd(&q.hist[pass * 256 + threadIdx.x], bins[threadIdx.x]);
        grid.sync();
        // ---- the same decision in every block: the byte in which the rem-th record of the bucket falls ----------
        const unsigned int v = __ldcg(&q.hist[pass * 256 + threadIdx.x]);
        unsigned int inc = v;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int up = __shfl_up_sync(full, inc, o);
            if (lane >= o) inc += up;
        }
        if (lane == 31) sscan[wib] = inc;
        __syncthreads();
        unsigned long long upto = inc;
        for (int w = 0; w < wib; ++w) upto += sscan[w];
        const unsigned long long before = upto - v;
        if (before < rem && rem <= upto) {
            s_digit = threadIdx.x;
            s_before = before;
            s_count = v;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned long long dg = s_digit;
            if (pass >= 6) { s_phi |= dg << (8 * (pass - 6)); s_mhi |= 0xFFULL << (8 * (pass - 6)); }
            else           { s_plo |= dg << (8 * pass);       s_mlo |= 0xFFULL << (8 * pass); }
            s_rem = rem - s_before;
            s_whole = s_rem == s_count;
        }
        __syncthreads();
    }

    // ---- compaction in input order: every record below the prefix, then the first s_rem inside its bucket -------
    const unsigned long long phi = s_phi, plo = s_plo, mhi = s_mhi, mlo = s_mlo;
    const unsigned long long limit = s_whole ? ~0ULL : s_rem;
    long long chunk = (n + nwarps - 1) / nwarps;
    chunk = (chunk + 31) / 32 * 32;
    const long long lo = gw * chunk < n ? gw * chunk : n;
    const long long hi = lo + chunk < n ? lo + chunk : n;
    auto classify = [&](long long i, uint4 &r) -> int {   // 0 below the prefix, 1 inside its bucket, 2 above
        if (i >= hi) return 2;
        r = q.in[i];
        const RecordKey key = key_of(r);
        const unsigned long long h = key.hi & mhi, l = key.lo & mlo;
        if (h != phi) return h < phi ? 0 : 2;
        if (l != plo) return l < plo ? 0 : 2;
        return 1;
    };
    unsigned long long nbelow = 0, ninside = 0;
    for (long long t = lo; t < hi; t += 32) {
        uint4 r;
        const int c = classify(t + lane, r);
        nbelow += __popc(__ballot_sync(full, c == 0));
        ninside += __popc(__ballot_sync(full, c == 1));
    }
    if (lane == 0) {
        q.wcount[gw] = nbelow;
        q.wcount[nwarps + gw] = ninside;
    }
    grid.sync();
    unsigned long long base_below = 0, base_inside = 0;
    for (long long c = 0; c < gw; c += 32) {
        if (c + lane < gw) {
            base_below += __ldcg(&q.wcount[c + lane]);
            base_inside += __ldcg(&q.wcount[nwarps + c + lane]);
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        base_below += __shfl_xor_sync(full, base_below, o);
        base_inside += __shfl_xor_sync(full, base_inside, o);
    }
    for (long long t = lo; t < hi; t += 32) {
        uint4 r;
        const long long i = t + lane;
        const int c = classify(i, r);
        const unsigned below = __ballot_sync(full, c == 0), inside = __ballot_sync(full, c == 1);
        const unsigned long long my_below = base_below + __popc(below & lt);
        const unsigned long long my_inside = base_inside + __popc(inside & lt);
        if (c == 0 || (c == 1 && my_inside < limit)) {
            const unsigned long long to = my_below + (my_inside < limit ? my_inside : limit);
            q.out[to] = r;
            q.idx[to] = (uint32_t)i;
        }
        base_below += __popc(below);
        base_inside += __popc(inside);
    }
}

__global__ void gather_index_kernel(const uint32_t *__restrict__ from, const uint32_t *__restrict__ perm, long long n,
                                    uint32_t *__restrict__ to) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        to[i] = from[perm[i]];
}

static int coop_grid(const void *kernel, const char *name, int *blocks) {
    int dev = 0, sms = 0, per_sm = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kRankThreads, 0);
    if (e != cudaSuccess) return fail_cuda(e, name);
    if (per_sm < 1) return fail_arg("cooperative record kernel does not fit on this device");
    if (per_sm > 2) per_sm = 2;                 // 2 blocks x 8 warps per SM are plenty for a bandwidth-light pass
    *blocks = sms * per_sm;
    return METIS_OK;
}

}  // namespace metis

using namespace metis;

extern "C" {

// upper bound on the warps of the cooperative grid (B200: 148 SMs x 2 blocks x 8 warps)
static const int64_t kRankMaxWarps = 8192;

int64_t metis_sort_workspace_bytes(int64_t n) {
    if (n < 0) return METIS_E_ARG;
    return 512 + n * 16 + 2 * n * 4 + 256 * kRankMaxWarps * 4 + 256 * 4 + 512;
}

int metis_sort_records(MetisRecord *records, int64_t n, int32_t mode, uint32_t *perm_out, void *workspace,
                       int64_t workspace_bytes, void *stream_) {
    if (n < 0 || (n > 0 && !records) || !workspace) return fail_arg("metis_sort_records: bad argument");
    if (mode < METIS_SORT_POSITION || mode > METIS_SORT_BY_COST_STABLE) return fail_arg("metis_sort_records: unknown mode");
    if (n >= 0xFFFFFFF0LL) return fail_arg("metis_sort_records: more than 2^32 records");
    if (workspace_bytes < metis_sort_workspace_bytes(n)) return METIS_E_CAPACITY;
    if (n == 0) return METIS_OK;
    int blocks = 0;
    const int rc = coop_grid((const void *)rank_records_kernel, "rank_records_kernel occupancy", &blocks);
    if (rc) return rc;
    if ((int64_t)blocks * kRankWarps > kRankMaxWarps) blocks = (int)(kRankMaxWarps / kRankWarps);
    uint8_t *p = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    RankArgs q;
    q.a = reinterpret_cast<uint4 *>(records);
    q.b = reinterpret_cast<uint4 *>(p);            p += n * 16;
    q.ia = reinterpret_cast<uint32_t *>(p);        p += n * 4;
    q.ib = reinterpret_cast<uint32_t *>(p);        p += n * 4;
    p = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(p) + 255) & ~(uintptr_t)255);
    q.hist = reinterpret_cast<unsigned int *>(p);  p += 256 * (int64_t)blocks * kRankWarps * 4;
    q.bintot = reinterpret_cast<unsigned int *>(p);
    q.n = n;
    q.pass_begin = mode == METIS_SORT_BY_COST_STABLE ? 6 : 0;
    q.pass_end = mode == METIS_SORT_POSITION ? 6 : 14;
    q.perm_out = perm_out;
    void *args[] = {&q};
    cudaError_t e = cudaLaunchCooperativeKernel((const void *)rank_records_kernel, dim3((unsigned)blocks), dim3(kRankThreads),
                                                args, 0, static_cast<cudaStream_t>(stream_));
    if (e != cudaSuccess) return fail_cuda(e, "rank_records_kernel");
    return METIS_OK;
}

int64_t metis_select_workspace_bytes(int64_t n, int64_t k) {
    if (n < 0 || k < 0) return METIS_E_ARG;
    const int64_t m = k < n ? k : n;
    return 256 + kKeyDigits * 256 * 4 + 2 * kRankMaxWarps * 8 + 2 * m * 4 + 256 + metis_sort_workspace_bytes(m);
}

int metis_select_records(const MetisRecord *records, int64_t n, int64_t k, MetisRecord *out, uint32_t *idx_out,
                         void *workspace, int64_t workspace_bytes, void *stream_) {
    if (n < 0 || k < 0 || (n > 0 && k > 0 && (!records || !out)) || !workspace)
        return fail_arg("metis_select_records: bad argument");
    if (n >= 0xFFFFFFF0LL) return fail_arg("metis_select_records: more than 2^32 records");
    if (workspace_bytes < metis_select_workspace_bytes(n, k)) return METIS_E_CAPACITY;
    if (n == 0 || k == 0) return METIS_OK;
    const int64_t m = k < n ? k : n;
    int blocks = 0;
    int rc = coop_grid((const void *)select_records_kernel, "select_records_kernel occupancy", &blocks);
    if (rc) return rc;
    if ((int64_t)blocks * kRankWarps > kRankMaxWarps) blocks = (int)(kRankMaxWarps / kRankWarps);
    const cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    uint8_t *p = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    SelectArgs q;
    q.in = reinterpret_cast<const uint4 *>(records);
    q.n = n;
    q.k = k;
    q.out = reinterpret_cast<uint4 *>(out);
    q.hist = reinterpret_cast<unsigned int *>(p);          p += kKeyDigits * 256 * 4;
    q.wcount = reinterpret_cast<unsigned long long *>(p);  p += 2 * kRankMaxWarps * 8;
    q.idx = reinterpret_cast<uint32_t *>(p);               p += m * 4;
    uint32_t *perm = reinterpret_cast<uint32_t *>(p);      p += m * 4;
    p = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(p) + 255) & ~(uintptr_t)255);
    const int64_t sort_bytes = workspace_bytes - (p - reinterpret_cast<uint8_t *>(workspace));
    void *args[] = {&q};
    cudaError_t e = cudaLaunchCooperativeKernel((const void *)select_records_kernel, dim3((unsigned)blocks),
                                                dim3(kRankThreads), args, 0, stream);
    if (e != cudaSuccess) return fail_cuda(e, "select_records_kernel");
    // the selected records are in input order, so the stable ranked sort also keeps equal keys in input order
    rc = metis_sort_records(out, m, METIS_SORT_RANKED, idx_out ? perm : nullptr, p, sort_bytes, stream_);
    if (rc) return rc;
    if (idx_out) {
        const int threads = 256;
        const long long grid = (m + threads - 1) / threads < 1024 ? (m + threads - 1) / threads : 1024;
        gather_index_kernel<<<(unsigned)grid, threads, 0, stream>>>(q.idx, perm, m, idx_out);
        e = cudaGetLastError();
        if (e != cudaSuccess) return fail_cuda(e, "gather_index_kernel");
    }
    return METIS_OK;
}

}  // extern "C"
