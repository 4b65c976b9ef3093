// SetConv fast path for the induced -> target direction (regular key grid, up to 128 channels).
//
// The generic kernels (setconv.cu) give every query its own sweep over its sigma-window: with ~20-50 grid rows per
// window and 128 queries per task every row of V is fetched ~7x (L2-bandwidth bound, ~6x the algorithmic bytes).
// Here one CTA owns one task and first SORTS its queries by position (rank by counting, in shared memory); a warp
// then processes 8 position-adjacent queries together over the UNION of their windows, so each V row is loaded once
// per group (one 16-byte load per lane = the whole 128-channel row per warp) and feeds 8 x 4 FMAs per lane.  The value
// gradient uses the mirrored scheme: 8 adjacent grid rows against the contiguous run of sorted queries whose windows
// touch them.  Weights are computed one row (or query) per lane and broadcast with shuffles.
//
//   mode 0: feat = sum_k softmax_k(a) V_k, dens, (max logit, sum exp)            (forward)
//   mode 1: d theta: T - G*A1 + ddens*A2 with max-shifted logits (see setconv.cu)
//   dV    : dV[k] = sum_q w_qk dF_q                                               (gather, no atomics)
#include "tc_common.cuh"

namespace npf {

constexpr float kWindowLogT = 41.6f;
constexpr int kGroup = 8;        // queries (or rows) per warp pass
constexpr int kRowBatch = 4;     // value rows loaded per batch (3 CTAs x 8 warps per SM keep >= 96 16-byte loads per lane slot in flight)
constexpr int kMaxQ = 2048;      // queries per task handled in shared memory

// logits use 1 / sigma (one division per kernel instead of one per pair; <= 1 ulp from the quotient form)
__device__ __forceinline__ float logit_t(float xq, float xk, float inv_sigma) {
    const float t = (xk - xq) * inv_sigma;
    return -(t * t);
}

// identical policy to key_window() in setconv.cu
__device__ __forceinline__ void window_t(const float* __restrict__ keys, int K, float xq, float sigma, int& lo_o, int& hi_o) {
    lo_o = 0; hi_o = K - 1;
    if (K < 3) return;
    const float x0 = __ldg(keys), x1 = __ldg(keys + K - 1);
    const float dx = (x1 - x0) / (float)(K - 1);
    if (!(dx > 0.f)) return;
    float pos = (xq - x0) / dx;
    pos = fminf(fmaxf(pos, 0.f), (float)(K - 1));
    const int n0 = (int)rintf(pos);
    const float dn = xq - __ldg(keys + n0);
    const float D = sqrtf(dn * dn + kWindowLogT * sigma * sigma);
    float lo = floorf((xq - D - x0) / dx) - 1.f;
    float hi = ceilf((xq + D - x0) / dx) + 1.f;
    if (!(lo == lo) || !(hi == hi)) return;
    lo = fminf(fmaxf(lo, 0.f), (float)(K - 1));
    hi = fminf(fmaxf(hi, 0.f), (float)(K - 1));
    lo_o = min((int)lo, n0);
    hi_o = max((int)hi, n0);
}

// Pull a contiguous range into L2 ahead of use (one prefetch per 128-byte line, spread over the CTA): the DRAM latency of
// the task's value rows then overlaps the sort / window phase instead of stalling every batch of the group pass.
__device__ __forceinline__ void prefetch_l2_range(const void* base, size_t bytes, int part, int n_parts) {
    const char* p = reinterpret_cast<const char*>(base);
    const size_t lines = (bytes + 127) >> 7;
    const size_t per = (lines + n_parts - 1) / n_parts, l0 = per * part, l1 = min(lines, l0 + per);
    for (size_t l = l0 + threadIdx.x; l < l1; l += blockDim.x) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + (l << 7)));
}

struct TileSmem {
    float* xs;    // [Q] sorted query positions
    int* ord;     // [Q] original index of the sorted query
    int* lo;      // [Q] window (in sorted order)
    int* hi;
    float* m;     // [Q] max logit
    float* invs;  // [Q] 1 / sum exp(a - m)
};

__device__ __forceinline__ TileSmem carve(float* base, int Q) {
    TileSmem t;
    t.xs = base;
    t.ord = reinterpret_cast<int*>(base + Q);
    t.lo = t.ord + Q;
    t.hi = t.lo + Q;
    t.m = reinterpret_cast<float*>(t.hi + Q);
    t.invs = t.m + Q;
    return t;
}

// sort the task's queries by position (stable: ties by index) via rank counting
__device__ __forceinline__ void sort_queries(const TileSmem& t, const float* __restrict__ qb, int Q, float* scratch /*[Q]*/) {
    for (int i = threadIdx.x; i < Q; i += blockDim.x) scratch[i] = __ldg(qb + i);
    __syncthreads();
    for (int i = threadIdx.x; i < Q; i += blockDim.x) {
        const float x = scratch[i];
        int rank = 0, j = 0;
        if ((Q & 3) == 0) {                                // scratch sits 6 Q floats into the 16-byte aligned dynamic smem: float4 reads
            for (; j < Q; j += 4) {
                const float4 y = *reinterpret_cast<const float4*>(scratch + j);
                rank += (y.x < x) + (y.y < x) + (y.z < x) + (y.w < x);
                rank += (y.x == x && j < i) + (y.y == x && j + 1 < i) + (y.z == x && j + 2 < i) + (y.w == x && j + 3 < i);
            }
        }
        for (; j < Q; ++j) {
            const float y = scratch[j];
            rank += (y < x) || (y == x && j < i);
        }
        t.xs[rank] = x;
        t.ord[rank] = i;
    }
    __syncthreads();
}

// mode 0 forward / mode 1 theta gradient
template <int MODE>
__global__ void __launch_bounds__(256, 3) setconv_grp_kernel(const float* __restrict__ keys, long key_bs, const float* __restrict__ queries,
                                                          long qry_bs, const float* __restrict__ values, const float* __restrict__ theta,
                                                          float* __restrict__ feat_o, float* __restrict__ dens_o, float* __restrict__ mstat_o,
                                                          const float* __restrict__ feat_i, const float* __restrict__ mstat_i,
                                                          const float* __restrict__ dfeat, const float* __restrict__ ddens,
                                                          float* __restrict__ dtheta, int K, int Q, int C) {
    extern __shared__ float smem[];
    __shared__ float part[8];
    const TileSmem t = carve(smem, Q);
    float* scratch = t.invs + Q;
    const int b = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float th = __ldg(theta);
    const float sigma = 1e-5f + softplus_f(th);
    const float inv_sigma = 1.f / sigma;
    const float* kb = keys + (long)b * key_bs;
    const float* vb = values + (long)b * K * C;
    prefetch_l2_range(vb, sizeof(float) * (size_t)K * C, blockIdx.y, gridDim.y);
    if (MODE == 1) {
        prefetch_l2_range(dfeat + (long)b * Q * C, sizeof(float) * (size_t)Q * C, blockIdx.y, gridDim.y);
        prefetch_l2_range(feat_i + (long)b * Q * C, sizeof(float) * (size_t)Q * C, blockIdx.y, gridDim.y);
    }
    sort_queries(t, queries + (long)b * qry_bs, Q, scratch);

    // per-query window (one thread per query).  Forward: the max logit is the one of the nearest grid row (the window code's
    // n0 or a neighbour: all three are tried); the softmax denominator is accumulated by the group pass below from the very
    // weights it applies, so no thread walks its window serially.
    for (int i = threadIdx.x; i < Q; i += blockDim.x) {
        const float xq = t.xs[i];
        int lo, hi;
        window_t(kb, K, xq, sigma, lo, hi);
        t.lo[i] = lo; t.hi[i] = hi;
        if (MODE == 0) {
            const float x0 = __ldg(kb), dx = (__ldg(kb + K - 1) - x0) / (float)(K - 1);
            int n0 = (dx > 0.f) ? (int)rintf(fminf(fmaxf((xq - x0) / dx, 0.f), (float)(K - 1))) : lo;
            n0 = min(max(n0, lo), hi);
            float m = logit_t(xq, __ldg(kb + n0), inv_sigma);
            if (n0 > lo) m = fmaxf(m, logit_t(xq, __ldg(kb + n0 - 1), inv_sigma));
            if (n0 < hi) m = fmaxf(m, logit_t(xq, __ldg(kb + n0 + 1), inv_sigma));
            if (!(dx > 0.f)) for (int k = lo; k <= hi; ++k) m = fmaxf(m, logit_t(xq, __ldg(kb + k), inv_sigma));   // degenerate grid
            t.m[i] = m;
        } else {
            const long oq = (long)b * Q + t.ord[i];
            t.m[i] = __ldg(mstat_i + oq * 2);
            t.invs[i] = 1.f / __ldg(mstat_i + oq * 2 + 1);
        }
    }
    __syncthreads();

    const int c4 = lane * 4;
    const bool ch_ok = c4 < C;
    float warp_contrib = 0.f;
    const int n_groups = (Q + kGroup - 1) / kGroup;
    for (int grp = blockIdx.y * 8 + warp; grp < n_groups; grp += 8 * gridDim.y) {
        const int t0 = grp * kGroup;
        const int nt = min(kGroup, Q - t0);
        int glo = t.lo[t0], ghi = t.hi[t0];
        for (int j = 1; j < nt; ++j) { glo = min(glo, t.lo[t0 + j]); ghi = max(ghi, t.hi[t0 + j]); }
        float4 acc[kGroup];
#pragma unroll
        for (int j = 0; j < kGroup; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        float a1[kGroup], a2[kGroup];      // forward: a1 = this lane's share of sum_k exp(a - m);  theta gradient: A1, A2
#pragma unroll
        for (int j = 0; j < kGroup; ++j) { a1[j] = 0.f; a2[j] = 0.f; }
        for (int base = glo; base <= ghi; base += 32) {
            const int row = base + lane;
            const float xk = (row <= ghi) ? __ldg(kb + row) : 0.f;
            float w[kGroup];
#pragma unroll
            for (int j = 0; j < kGroup; ++j) {
                w[j] = 0.f;
                if (j < nt && row <= ghi && row >= t.lo[t0 + j] && row <= t.hi[t0 + j]) {
                    const float a = logit_t(t.xs[t0 + j], xk, inv_sigma);
                    if (MODE == 0) {
                        w[j] = expf(a - t.m[t0 + j]);          // unnormalised: divided by the sum once per query below
                        a1[j] += w[j];
                    } else {
                        w[j] = expf(a - t.m[t0 + j]) * t.invs[t0 + j] * (a - t.m[t0 + j]);
                        a1[j] += w[j];
                        a2[j] = fmaf(expf(a), a, a2[j]);
                    }
                }
            }
            const int cnt = min(32, ghi - base + 1);
            for (int rr0 = 0; rr0 < cnt; rr0 += kRowBatch) {   // kRowBatch row loads in flight, then kRowBatch x (8 shuffles + 32 FMAs)
                float4 v[kRowBatch];
#pragma unroll
                for (int u = 0; u < kRowBatch; ++u) {
                    v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (ch_ok && rr0 + u < cnt) v[u] = __ldg(reinterpret_cast<const float4*>(vb + (long)(base + rr0 + u) * C + c4));
                }
#pragma unroll
                for (int u = 0; u < kRowBatch; ++u) {
#pragma unroll
                    for (int j = 0; j < kGroup; ++j) {
                        const float wj = __shfl_sync(0xffffffffu, w[j], rr0 + u);   // rows past the window carry weight 0
                        acc[j].x = fmaf(wj, v[u].x, acc[j].x); acc[j].y = fmaf(wj, v[u].y, acc[j].y);
                        acc[j].z = fmaf(wj, v[u].z, acc[j].z); acc[j].w = fmaf(wj, v[u].w, acc[j].w);
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < kGroup; ++j) {
            if (j >= nt) continue;
            const long oq = (long)b * Q + t.ord[t0 + j];
            if (MODE == 0) {
                const float ssum = warp_sum(a1[j]), inv = 1.f / ssum;
                if (ch_ok) *reinterpret_cast<float4*>(feat_o + oq * C + c4) = make_float4(acc[j].x * inv, acc[j].y * inv, acc[j].z * inv, acc[j].w * inv);
                if (lane == 0) {                               // dens = sum_k exp(a) = exp(m) * sum_k exp(a - m)
                    const float m = t.m[t0 + j];
                    dens_o[oq] = expf(m) * ssum;
                    mstat_o[oq * 2] = m; mstat_o[oq * 2 + 1] = ssum;
                }
            } else {
                float T = 0.f, G = 0.f;
                if (ch_ok) {
                    const float4 g = __ldg(reinterpret_cast<const float4*>(dfeat + oq * C + c4));
                    const float4 f = __ldg(reinterpret_cast<const float4*>(feat_i + oq * C + c4));
                    T = g.x * acc[j].x + g.y * acc[j].y + g.z * acc[j].z + g.w * acc[j].w;
                    G = g.x * f.x + g.y * f.y + g.z * f.z + g.w * f.w;
                }
                T = warp_sum(T); G = warp_sum(G);
                const float A1 = warp_sum(a1[j]), A2 = warp_sum(a2[j]);
                warp_contrib += T - G * A1 + __ldg(ddens + oq) * A2;
            }
        }
    }
    if (MODE == 1) {
        if (lane == 0) part[warp] = warp_contrib;
        __syncthreads();
        if (threadIdx.x == 0) {
            float tot = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) tot += part[i];
            atomicAdd(dtheta, tot * (-2.f / sigma) * sigmoid_f(th));
        }
    }
}

// dV[b,k,:] = sum_q w_qk dF[b,q,:]: a warp owns 8 adjacent key rows and walks the contiguous run of sorted queries whose
// window touches them.
__global__ void __launch_bounds__(256, 3) setconv_grp_dv_kernel(const float* __restrict__ keys, long key_bs, const float* __restrict__ queries,
                                                             long qry_bs, const float* __restrict__ theta, const float* __restrict__ mstat,
                                                             const float* __restrict__ dfeat, float* __restrict__ dvalues, int K, int Q, int C) {
    extern __shared__ float smem[];
    const TileSmem t = carve(smem, Q);
    float* scratch = t.invs + Q;
    const int b = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float sigma = 1e-5f + softplus_f(__ldg(theta));
    const float inv_sigma = 1.f / sigma;
    const float* kb = keys + (long)b * key_bs;
    prefetch_l2_range(dfeat + (long)b * Q * C, sizeof(float) * (size_t)Q * C, blockIdx.y, gridDim.y);
    sort_queries(t, queries + (long)b * qry_bs, Q, scratch);
    for (int i = threadIdx.x; i < Q; i += blockDim.x) {
        int lo, hi;
        window_t(kb, K, t.xs[i], sigma, lo, hi);
        t.lo[i] = lo; t.hi[i] = hi;
        const long oq = (long)b * Q + t.ord[i];
        t.m[i] = __ldg(mstat + oq * 2);
        t.invs[i] = 1.f / __ldg(mstat + oq * 2 + 1);
    }
    __syncthreads();
    const int c4 = lane * 4;
    const bool ch_ok = c4 < C;
    const int n_rgroups = (K + kGroup - 1) / kGroup;
    for (int rg = blockIdx.y * 8 + warp; rg < n_rgroups; rg += 8 * gridDim.y) {
        const int k0 = rg * kGroup, nr = min(kGroup, K - k0);
        // lo[] and hi[] are non-decreasing in sorted order: queries with hi >= k0 and lo <= k0+nr-1 form one run
        int ta = 0, tb = Q;
        { int l = 0, h = Q; while (l < h) { const int mid = (l + h) >> 1; if (t.hi[mid] >= k0) h = mid; else l = mid + 1; } ta = l; }
        { int l = ta, h = Q; while (l < h) { const int mid = (l + h) >> 1; if (t.lo[mid] > k0 + nr - 1) h = mid; else l = mid + 1; } tb = l; }
        float xk[kGroup];
#pragma unroll
        for (int r = 0; r < kGroup; ++r) xk[r] = (r < nr) ? __ldg(kb + k0 + r) : 0.f;
        float4 acc[kGroup];
#pragma unroll
        for (int r = 0; r < kGroup; ++r) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int base = ta; base < tb; base += 32) {
            const int ti = base + lane;
            float w[kGroup];
#pragma unroll
            for (int r = 0; r < kGroup; ++r) {
                w[r] = 0.f;
                if (ti < tb && r < nr && k0 + r >= t.lo[ti] && k0 + r <= t.hi[ti])
                    w[r] = expf(logit_t(t.xs[ti], xk[r], inv_sigma) - t.m[ti]) * t.invs[ti];
            }
            const int cnt = min(32, tb - base);
            for (int tt0 = 0; tt0 < cnt; tt0 += kRowBatch) {
                float4 g[kRowBatch];
#pragma unroll
                for (int u = 0; u < kRowBatch; ++u) {
                    g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (ch_ok && tt0 + u < cnt) g[u] = __ldg(reinterpret_cast<const float4*>(dfeat + ((long)b * Q + t.ord[base + tt0 + u]) * C + c4));
                }
#pragma unroll
                for (int u = 0; u < kRowBatch; ++u) {
#pragma unroll
                    for (int r = 0; r < kGroup; ++r) {
                        const float wr = __shfl_sync(0xffffffffu, w[r], tt0 + u);   // queries past the run carry weight 0
                        acc[r].x = fmaf(wr, g[u].x, acc[r].x); acc[r].y = fmaf(wr, g[u].y, acc[r].y);
                        acc[r].z = fmaf(wr, g[u].z, acc[r].z); acc[r].w = fmaf(wr, g[u].w, acc[r].w);
                    }
                }
            }
        }
        if (ch_ok) {
#pragma unroll
            for (int r = 0; r < kGroup; ++r)
                if (r < nr) *reinterpret_cast<float4*>(dvalues + ((long)b * K + k0 + r) * C + c4) = acc[r];
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Task-resident variant (C == 128, K * 512 B <= ~190 KB): ONE persistent CTA per SM walks the tasks; the task's whole value
// matrix V[K,128] is brought into shared memory by the TMA (cp.async.bulk, one mbarrier per 32-row chunk) while the CTA sorts
// the queries, so HBM sees every byte exactly once, fully coalesced, and the group pass reads rows with LDS.128 instead of
// waiting on batches of global loads.  A warp owns 8 position-adjacent queries; the lanes compute the 8 x 32 weights of a
// 32-row slab once (one row per lane), park them in the warp's shared-memory slab and every row step is then
// 2 broadcast LDS.128 (weights) + 1 LDS.128 (values) + 32 FFMA.  Warps start on a slab as soon as its chunk has landed.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kTaskThreads = 512;
constexpr int kTaskWarps = kTaskThreads / 32;
constexpr int kChunkRows = 32;
constexpr int kMaxChunks = 16;          // K <= 512

// rank-counting sort with every thread busy: `parts` threads share one query and split the comparison range
__device__ __forceinline__ void sort_queries_wide(const TileSmem& t, const float* __restrict__ qb, int Q, float* scratch, int* rank_acc) {
    for (int i = threadIdx.x; i < Q; i += blockDim.x) { scratch[i] = __ldg(qb + i); rank_acc[i] = 0; }
    __syncthreads();
    const int parts = (int)blockDim.x / Q >= 4 ? 4 : ((int)blockDim.x / Q >= 2 ? 2 : 1);
    const int span = (Q + parts - 1) / parts;
    for (int w = threadIdx.x; w < Q * parts; w += blockDim.x) {
        const int i = w % Q, part = w / Q;
        const float x = scratch[i];
        const int j0 = part * span, j1 = min(Q, j0 + span);
        int r0 = 0, r1 = 0;
        int j = j0;
        for (; j + 2 <= j1; j += 2) {
            const float y0 = scratch[j], y1 = scratch[j + 1];
            r0 += (y0 < x) || (y0 == x && j < i);
            r1 += (y1 < x) || (y1 == x && j + 1 < i);
        }
        if (j < j1) { const float y = scratch[j]; r0 += (y < x) || (y == x && j < i); }
        if (parts == 1) rank_acc[i] = r0 + r1; else atomicAdd(&rank_acc[i], r0 + r1);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < Q; i += blockDim.x) {
        const int rank = rank_acc[i];
        t.xs[rank] = scratch[i];
        t.ord[rank] = i;
    }
    __syncthreads();
}

// per-query constants of the task, packed for one broadcast LDS.128: (position, max logit, 1 / sum, window lo | hi << 16)
__device__ __forceinline__ float4 pack_qc(float x, float m, float invs, int lo, int hi) { return make_float4(x, m, invs, __int_as_float(lo | (hi << 16))); }

template <int MODE>
__global__ void __launch_bounds__(kTaskThreads, 1) setconv_task_kernel(const float* __restrict__ keys, long key_bs, const float* __restrict__ queries,
                                                                       long qry_bs, const float* __restrict__ values, const float* __restrict__ theta,
                                                                       float* __restrict__ feat_o, float* __restrict__ dens_o, float* __restrict__ mstat_o,
                                                                       const float* __restrict__ feat_i, const float* __restrict__ mstat_i,
                                                                       const float* __restrict__ dfeat, const float* __restrict__ ddens,
                                                                       float* __restrict__ dtheta, int B, int K, int Q) {
    constexpr int C = 128;
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t bars[kMaxChunks];
    __shared__ float part[kTaskWarps];
    const int n_chunks = (K + kChunkRows - 1) / kChunkRows;
    float* Vs = smem;                                              // [n_chunks * 32][128]
    float* wbuf_all = Vs + (size_t)n_chunks * kChunkRows * C;      // [16 warps][32 rows][8 queries]
    float4* qc = reinterpret_cast<float4*>(wbuf_all + kTaskWarps * kChunkRows * kGroup);   // [Q]
    const TileSmem t = carve(reinterpret_cast<float*>(qc + Q), Q);
    float* scratch = t.invs + Q;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* wbuf = wbuf_all + warp * (kChunkRows * kGroup);
    const float th = __ldg(theta);
    const float sigma = 1e-5f + softplus_f(th);
    const float inv_sigma = 1.f / sigma;
    if (threadIdx.x == 0) {
        for (int c = 0; c < n_chunks; ++c) mbar_init(&bars[c], 1);
    }
    __syncthreads();
    float warp_contrib = 0.f;
    uint32_t parity = 0;
    for (int b = blockIdx.x; b < B; b += gridDim.x, parity ^= 1) {
        const float* kb = keys + (long)b * key_bs;
        const float* vb = values + (long)b * K * C;
        if (threadIdx.x == 0) {
            fence_async_smem();                    // the previous task's generic reads of Vs are ordered before the new async writes
            for (int c = 0; c < n_chunks; ++c) {
                const int rows = min(kChunkRows, K - c * kChunkRows);
                const uint32_t bytes = (uint32_t)rows * C * sizeof(float);
                mbar_expect_tx(&bars[c], bytes);
                bulk_g2s(Vs + (size_t)c * kChunkRows * C, vb + (size_t)c * kChunkRows * C, bytes, &bars[c]);
            }
        }
        sort_queries_wide(t, queries + (long)b * qry_bs, Q, scratch, t.lo);
        const float x0 = __ldg(kb), dx = (__ldg(kb + K - 1) - x0) / (float)(K - 1);
        for (int i = threadIdx.x; i < Q; i += blockDim.x) {
            const float xq = t.xs[i];
            int lo, hi;
            window_t(kb, K, xq, sigma, lo, hi);
            float m, invs = 0.f;
            if (MODE == 0) {
                int n0 = (dx > 0.f) ? (int)rintf(fminf(fmaxf((xq - x0) / dx, 0.f), (float)(K - 1))) : lo;
                n0 = min(max(n0, lo), hi);
                m = logit_t(xq, __ldg(kb + n0), inv_sigma);
                if (n0 > lo) m = fmaxf(m, logit_t(xq, __ldg(kb + n0 - 1), inv_sigma));
                if (n0 < hi) m = fmaxf(m, logit_t(xq, __ldg(kb + n0 + 1), inv_sigma));
                if (!(dx > 0.f)) for (int k = lo; k <= hi; ++k) m = fmaxf(m, logit_t(xq, __ldg(kb + k), inv_sigma));
            } else {
                const long oq = (long)b * Q + t.ord[i];
                m = __ldg(mstat_i + oq * 2);
                invs = 1.f / __ldg(mstat_i + oq * 2 + 1);
            }
            qc[i] = pack_qc(xq, m, invs, lo, hi);
        }
        __syncthreads();

        const int c4 = lane * 4;
        const int n_groups = (Q + kGroup - 1) / kGroup;
        for (int grp = warp; grp < n_groups; grp += kTaskWarps) {
            const int t0 = grp * kGroup;
            const int nt = min(kGroup, Q - t0);
            // the group's 8 query records in registers (broadcast 16-byte reads), union window
            float qx[kGroup], qm[kGroup], qi[kGroup];
            int qlo[kGroup], qhi[kGroup];
            int glo = K, ghi = -1;
#pragma unroll
            for (int j = 0; j < kGroup; ++j) {
                const float4 r = qc[min(t0 + j, Q - 1)];
                const int lh = __float_as_int(r.w);
                qx[j] = r.x; qm[j] = r.y; qi[j] = r.z;
                qlo[j] = (j < nt) ? (lh & 0xFFFF) : K;              // empty window for the padding queries of the last group
                qhi[j] = (j < nt) ? (lh >> 16) : -1;
                glo = min(glo, qlo[j]); ghi = max(ghi, qhi[j]);
            }
            float4 acc[kGroup];
#pragma unroll
            for (int j = 0; j < kGroup; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            float a1[kGroup], a2[kGroup];
#pragma unroll
            for (int j = 0; j < kGroup; ++j) { a1[j] = 0.f; a2[j] = 0.f; }
            for (int base = glo; base <= ghi; base += 32) {
                const int row = base + lane;
                const float xk = __ldg(kb + min(row, K - 1));
                float w[kGroup];
#pragma unroll
                for (int j = 0; j < kGroup; ++j) {                   // branch-free: 8 independent exp chains per lane
                    const bool in = row >= qlo[j] && row <= qhi[j];
                    const float a = logit_t(qx[j], xk, inv_sigma);
                    const float e = expf(a - qm[j]);
                    if (MODE == 0) {
                        w[j] = in ? e : 0.f;
                        a1[j] += w[j];
                    } else {
                        w[j] = in ? e * qi[j] * (a - qm[j]) : 0.f;
                        a1[j] += w[j];
                        a2[j] += in ? expf(a) * a : 0.f;
                    }
                }
                __syncwarp();                                       // previous slab fully consumed
                *reinterpret_cast<float4*>(wbuf + lane * kGroup) = make_float4(w[0], w[1], w[2], w[3]);
                *reinterpret_cast<float4*>(wbuf + lane * kGroup + 4) = make_float4(w[4], w[5], w[6], w[7]);
                __syncwarp();
                const int cnt = min(32, ghi - base + 1);
                // the rows base .. base+cnt-1 live in at most two chunks
                mbar_wait(&bars[base / kChunkRows], parity);
                mbar_wait(&bars[(base + cnt - 1) / kChunkRows], parity);
                const float* vrow = Vs + (size_t)base * C + c4;
#pragma unroll 4
                for (int r = 0; r < cnt; ++r) {
                    const float4 wa = *reinterpret_cast<const float4*>(wbuf + r * kGroup);
                    const float4 wb = *reinterpret_cast<const float4*>(wbuf + r * kGroup + 4);
                    const float4 v = *reinterpret_cast<const float4*>(vrow + (size_t)r * C);
                    const float ws[kGroup] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
                    for (int j = 0; j < kGroup; ++j) {
                        acc[j].x = fmaf(ws[j], v.x, acc[j].x); acc[j].y = fmaf(ws[j], v.y, acc[j].y);
                        acc[j].z = fmaf(ws[j], v.z, acc[j].z); acc[j].w = fmaf(ws[j], v.w, acc[j].w);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < kGroup; ++j) {
                if (j >= nt) continue;
                const long oq = (long)b * Q + t.ord[t0 + j];
                if (MODE == 0) {
                    const float ssum = warp_sum(a1[j]), inv = 1.f / ssum;
                    *reinterpret_cast<float4*>(feat_o + oq * C + c4) = make_float4(acc[j].x * inv, acc[j].y * inv, acc[j].z * inv, acc[j].w * inv);
                    if (lane == 0) {
                        dens_o[oq] = expf(qm[j]) * ssum;
                        mstat_o[oq * 2] = qm[j]; mstat_o[oq * 2 + 1] = ssum;
                    }
                } else {
                    const float4 g = __ldg(reinterpret_cast<const float4*>(dfeat + oq * C + c4));
                    const float4 f = __ldg(reinterpret_cast<const float4*>(feat_i + oq * C + c4));
                    float T = g.x * acc[j].x + g.y * acc[j].y + g.z * acc[j].z + g.w * acc[j].w;
                    float G = g.x * f.x + g.y * f.y + g.z * f.z + g.w * f.w;
                    T = warp_sum(T); G = warp_sum(G);
                    const float A1 = warp_sum(a1[j]), A2 = warp_sum(a2[j]);
                    warp_contrib += T - G * A1 + __ldg(ddens + oq) * A2;
                }
            }
        }
        // every chunk must have landed before its barrier is re-armed and its rows overwritten (the last chunks may lie outside all windows)
        if (warp == 0) for (int c = lane; c < n_chunks; c += 32) mbar_wait(&bars[c], parity);
        __syncthreads();                                            // Vs, the query arrays and the slabs are reused by the next task
    }
    if (MODE == 1) {
        if (lane == 0) part[warp] = warp_contrib;
        __syncthreads();
        if (threadIdx.x == 0) {
            float tot = 0.f;
#pragma unroll
            for (int i = 0; i < kTaskWarps; ++i) tot += part[i];
            atomicAdd(dtheta, tot * (-2.f / sigma) * sigmoid_f(th));
        }
    }
}

// dV[b,k,:] = sum_q w_qk dF[b,q,:] with the task's dF[Q,128] resident in shared memory (one bulk copy).
__global__ void __launch_bounds__(kTaskThreads, 1) setconv_task_dv_kernel(const float* __restrict__ keys, long key_bs, const float* __restrict__ queries,
                                                                          long qry_bs, const float* __restrict__ theta, const float* __restrict__ mstat,
                                                                          const float* __restrict__ dfeat, float* __restrict__ dvalues, int B, int K, int Q) {
    constexpr int C = 128;
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t bar;
    float* Fs = smem;                                               // [Q][128]
    float* wbuf_all = Fs + (size_t)Q * C;                           // [16 warps][32 queries][8 rows]
    float4* qc = reinterpret_cast<float4*>(wbuf_all + kTaskWarps * kChunkRows * kGroup);
    const TileSmem t = carve(reinterpret_cast<float*>(qc + Q), Q);
    float* scratch = t.invs + Q;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* wbuf = wbuf_all + warp * (kChunkRows * kGroup);
    const float sigma = 1e-5f + softplus_f(__ldg(theta));
    const float inv_sigma = 1.f / sigma;
    if (threadIdx.x == 0) mbar_init(&bar, 1);
    __syncthreads();
    uint32_t parity = 0;
    for (int b = blockIdx.x; b < B; b += gridDim.x, parity ^= 1) {
        const float* kb = keys + (long)b * key_bs;
        if (threadIdx.x == 0) {
            fence_async_smem();
            const uint32_t bytes = (uint32_t)Q * C * sizeof(float);
            mbar_expect_tx(&bar, bytes);
            bulk_g2s(Fs, dfeat + (long)b * Q * C, bytes, &bar);
        }
        sort_queries_wide(t, queries + (long)b * qry_bs, Q, scratch, t.lo);
        for (int i = threadIdx.x; i < Q; i += blockDim.x) {
            int lo, hi;
            window_t(kb, K, t.xs[i], sigma, lo, hi);
            t.lo[i] = lo; t.hi[i] = hi;
            const long oq = (long)b * Q + t.ord[i];
            qc[i] = pack_qc(t.xs[i], __ldg(mstat + oq * 2), 1.f / __ldg(mstat + oq * 2 + 1), lo, hi);
        }
        __syncthreads();
        mbar_wait(&bar, parity);
        const int c4 = lane * 4;
        const int n_rgroups = (K + kGroup - 1) / kGroup;
        for (int rg = warp; rg < n_rgroups; rg += kTaskWarps) {
            const int k0 = rg * kGroup, nr = min(kGroup, K - k0);
            int ta = 0, tb = Q;
            { int l = 0, h = Q; while (l < h) { const int mid = (l + h) >> 1; if (t.hi[mid] >= k0) h = mid; else l = mid + 1; } ta = l; }
            { int l = ta, h = Q; while (l < h) { const int mid = (l + h) >> 1; if (t.lo[mid] > k0 + nr - 1) h = mid; else l = mid + 1; } tb = l; }
            float xk[kGroup];
#pragma unroll
            for (int r = 0; r < kGroup; ++r) xk[r] = __ldg(kb + min(k0 + r, K - 1));
            float4 acc[kGroup];
#pragma unroll
            for (int r = 0; r < kGroup; ++r) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int base = ta; base < tb; base += 32) {
                const int ti = base + lane;
                const float4 rec = qc[min(ti, Q - 1)];
                const int lh = __float_as_int(rec.w);
                const int lo = (ti < tb) ? (lh & 0xFFFF) : K, hi = (ti < tb) ? (lh >> 16) : -1;
                float w[kGroup];
#pragma unroll
                for (int r = 0; r < kGroup; ++r) {
                    const bool in = r < nr && k0 + r >= lo && k0 + r <= hi;
                    const float e = expf(logit_t(rec.x, xk[r], inv_sigma) - rec.y) * rec.z;
                    w[r] = in ? e : 0.f;
                }
                __syncwarp();
                *reinterpret_cast<float4*>(wbuf + lane * kGroup) = make_float4(w[0], w[1], w[2], w[3]);
                *reinterpret_cast<float4*>(wbuf + lane * kGroup + 4) = make_float4(w[4], w[5], w[6], w[7]);
                __syncwarp();
                const int cnt = min(32, tb - base);
                const int my_ord = t.ord[min(ti, Q - 1)];
#pragma unroll 4
                for (int q = 0; q < cnt; ++q) {
                    const float4 wa = *reinterpret_cast<const float4*>(wbuf + q * kGroup);
                    const float4 wb = *reinterpret_cast<const float4*>(wbuf + q * kGroup + 4);
                    const int o = __shfl_sync(0xffffffffu, my_ord, q);
                    const float4 g = *reinterpret_cast<const float4*>(Fs + (size_t)o * C + c4);
                    const float ws[kGroup] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
                    for (int r = 0; r < kGroup; ++r) {
                        acc[r].x = fmaf(ws[r], g.x, acc[r].x); acc[r].y = fmaf(ws[r], g.y, acc[r].y);
                        acc[r].z = fmaf(ws[r], g.z, acc[r].z); acc[r].w = fmaf(ws[r], g.w, acc[r].w);
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < kGroup; ++r)
                if (r < nr) *reinterpret_cast<float4*>(dvalues + ((long)b * K + k0 + r) * C + c4) = acc[r];
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Tensor-core forward for the induced -> target direction (C == 128, regular key grid):
//     feat[b] = diag(1 / s) . E[b] . V[b],    E[q, k] = exp(a_qk - m_q),   s_q = sum_k E[q, k]
// is a [128 queries x K keys] x [K x 128 channels] GEMM per task whose left operand is never stored: W-producer warps evaluate
// E in registers (one exp per pair, ex2.approx), split it into bf16 hi + lo and write it straight into the UMMA SWIZZLE_128B
// operand layout; V-producer warps stream the task's value rows from HBM (each byte once), split them the same way and stage
// them row-major, which the tensor core reads as the MN-major B operand; tcgen05.mma accumulates hi.hi + hi.lo + lo.hi over
// 64-key chunks (2-stage ring) into a TMEM accumulator that is double-buffered across tasks, and the epilogue scales row q by
// 1 / s_q and writes coalesced rows.  No query sort and no windows: keys outside a query's sigma-window get E = 0 by fp32
// underflow exactly as in the reference's dense softmax.  The SIMT version is bounded by the FFMA pipe (~ the HBM time
// itself); here the FMA work rides on the tensor pipe and the kernel is bounded by the V stream.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kTcKeys = 64;                 // keys per chunk (one 128-byte swizzle atom of bf16 along the reduction)
constexpr int kTcVProd = 8, kTcWProd = 8, kTcEpi = 8;
constexpr int kTcMmaWarp = kTcVProd + kTcWProd;
constexpr int kTcEpiWarp0 = kTcMmaWarp + 1;
constexpr int kTcThreads = (kTcEpiWarp0 + kTcEpi) * 32;      // 800
constexpr int kTcScratchLd = 20;

__device__ __forceinline__ uint64_t make_desc_sw128_t(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return make_desc(saddr, lbo_bytes, sbo_bytes) | (2ull << 61);
}
__device__ __forceinline__ void split_store8(const float (&v)[8], uint8_t* hi, uint8_t* lo, uint32_t off) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        h[e] = pack_bf16(v[2 * e], v[2 * e + 1]);
        l[e] = pack_bf16(v[2 * e] - __uint_as_float(h[e] << 16), v[2 * e + 1] - __uint_as_float(h[e] & 0xFFFF0000u));
    }
    *reinterpret_cast<uint4*>(hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
}

__global__ void __launch_bounds__(kTcThreads + 32, 1) setconv_tc_fwd_kernel(const float* __restrict__ keys, long key_bs, const float* __restrict__ queries,
                                                                      long qry_bs, const float* __restrict__ values, const float* __restrict__ theta,
                                                                      float* __restrict__ feat_o, float* __restrict__ dens_o, float* __restrict__ mstat_o,
                                                                      int B, int K, int Q) {
    constexpr int C = 128;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_vfull[2], bar_wfull[2], bar_empty[2], bar_tfull[2], bar_tempty[2], bar_rfull[2], bar_rempty[2];
    __shared__ uint32_t tmem_slot;
    __shared__ float s_sum[2][128];
    __shared__ __align__(16) float s_keys[kMaxChunks * kChunkRows + kTcKeys];   // shared key grid, padded with +inf to whole chunks

    constexpr uint32_t kWTile = 128u * kTcKeys * 2u;            // E chunk, one bf16 image: 16 KB
    constexpr uint32_t kVTile = kTcKeys * 128u * 2u;            // V chunk, one bf16 image: 16 KB
    constexpr uint32_t kStage = 2u * kWTile + 2u * kVTile;      // hi + lo of both: 64 KB
    float* scratch_all = reinterpret_cast<float*>(smem_raw + 2 * kStage);
    // raw fp32 V chunks (64 rows x 512 B), filled by TMA bulk copies from a loader warp two chunks ahead of the converting warps:
    // the V stream no longer waits on a global-load round trip per chunk (the register-staged version kept 32 KB in flight per SM)
    float* vraw = scratch_all + kTcEpi * 32 * kTcScratchLd;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    if (tid == 32) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_vfull[i], kTcVProd * 32);
            mbar_init(&bar_wfull[i], kTcWProd * 32);
            mbar_init(&bar_empty[i], 1);
            mbar_init(&bar_tfull[i], 1);
            mbar_init(&bar_tempty[i], kTcEpi * 32);
            mbar_init(&bar_rfull[i], 1);
            mbar_init(&bar_rempty[i], kTcVProd * 32);
        }
    }
    const float sigma = 1e-5f + softplus_f(__ldg(theta));
    const float inv_sigma = 1.f / sigma;
    const int n_chunks = (K + kTcKeys - 1) / kTcKeys;
    const int n_qt = (Q + 127) >> 7;
    const int n_units = B * n_qt;                                // (task, 128-query tile)
    pdl_trigger();
    for (int i = tid; i < n_chunks * kTcKeys; i += kTcThreads + 32) s_keys[i] = i < K ? __ldg(keys + i) : INFINITY;   // the grid is an input of the step
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    pdl_wait();

    if (warp == kTcThreads / 32) {
        // ------------------------------------------------------------------ loader: raw V chunks by TMA bulk copies, 2-deep ring
        int gr = 0;
        for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
            const float* vb = values + (long)(u / n_qt) * K * C;
            for (int c = 0; c < n_chunks; ++c, ++gr) {
                const int r = gr & 1;
                if (gr >= 2) mbar_wait(&bar_rempty[r], (uint32_t)((gr >> 1) - 1) & 1u);
                float* dst = vraw + r * (kTcKeys * C);
                const int rows = min(kTcKeys, K - c * kTcKeys);
                for (int i = lane; i < (kTcKeys - rows) * 32; i += 32) reinterpret_cast<float4*>(dst + rows * C)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                __syncwarp();
                if (lane == 0) {
                    fence_async_smem();
                    const uint32_t bytes = (uint32_t)rows * C * sizeof(float);
                    mbar_expect_tx(&bar_rfull[r], bytes);
                    bulk_g2s(dst, vb + (long)c * kTcKeys * C, bytes, &bar_rfull[r]);
                }
                __syncwarp();
            }
        }
    } else if (warp < kTcVProd) {
        // ------------------------------------------------------------------ V producers: warp w owns rows 8 w .. 8 w + 7 of a 64-key chunk
        const uint32_t vchunk = (uint32_t)(lane >> 1) & 7u;
        const uint32_t voff = (uint32_t)(lane >> 4) * 8192u + (uint32_t)(warp * 8) * 128u + (uint32_t)(lane & 1) * 8u;
        int g = 0;
        // the value rows of a unit are pulled into L2 one whole unit ahead (the register-staged loads keep only 32 KB in flight
        // per SM, far too little against ~5 us of loaded DRAM latency; an L2 hit costs ~1 k cycles)
        auto prefetch_unit = [&](int u) {
            if (u >= n_units) return;
            const char* base = reinterpret_cast<const char*>(values + (long)(u / n_qt) * K * C);
            const int lines = (K * C * 4 + 127) >> 7;
            for (int l = tid; l < lines; l += kTcVProd * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + ((long)l << 7)));
        };
        prefetch_unit(blockIdx.x);
        for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
            const int b = u / n_qt;
            const float* vb = values + (long)b * K * C;
            prefetch_unit(u + gridDim.x);
            for (int c = 0; c < n_chunks; ++c, ++g) {
                const int s = g & 1;
                float4 v[8];
                const int r = g & 1;
                mbar_wait(&bar_rfull[r], (uint32_t)(g >> 1) & 1u);
                const float* src = vraw + r * (kTcKeys * C) + (warp * 8) * C + lane * 4;
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = *reinterpret_cast<const float4*>(src + i * C);
                mbar_arrive(&bar_rempty[r]);                       // the raw chunk is in registers: the loader may refill the slot
                if (g >= 2) mbar_wait(&bar_empty[s], ((g >> 1) - 1) & 1);
                uint8_t* v_hi = smem_raw + s * kStage + 2 * kWTile;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const uint32_t off = voff + (uint32_t)i * 128u + ((vchunk ^ (uint32_t)i) << 4);
                    const uint32_t h01 = pack_bf16(v[i].x, v[i].y), h23 = pack_bf16(v[i].z, v[i].w);
                    *reinterpret_cast<uint2*>(v_hi + off) = make_uint2(h01, h23);
                    *reinterpret_cast<uint2*>(v_hi + kVTile + off) =
                        make_uint2(pack_bf16(v[i].x - __uint_as_float(h01 << 16), v[i].y - __uint_as_float(h01 & 0xFFFF0000u)),
                                   pack_bf16(v[i].z - __uint_as_float(h23 << 16), v[i].w - __uint_as_float(h23 & 0xFFFF0000u)));
                }
                fence_async_smem();
                mbar_arrive(&bar_vfull[s]);
            }
        }
    } else if (warp < kTcMmaWarp) {
        // ------------------------------------------------------------------ E producers: thread = (query, half of the chunk's keys)
        const int wt = tid - kTcVProd * 32;                       // 0..255
        const int ql = wt >> 1, half = wt & 1;                     // query row of the tile, keys [32 half, 32 half + 32) of the chunk
        const float x0 = s_keys[0], inv_dx = (float)(K - 1) / (s_keys[K - 1] - x0);
        const float is2 = inv_sigma * 1.2011224087864498f;         // exp(a - m) = exp2(-(d is2)^2 - m log2 e),  is2 = sqrt(log2 e) / sigma
        int g = 0, tcount = 0;
        // padding queries sit at +inf: every weight underflows to exactly 0 without a select in the inner loop.  The NEXT
        // unit's position is fetched a whole unit ahead (a cold load under load costs several microseconds).
        auto load_xq = [&](int u) {
            if (u >= n_units) return INFINITY;
            const int q = (u % n_qt) * 128 + ql;
            return q < Q ? __ldg(queries + (long)(u / n_qt) * qry_bs + q) : INFINITY;
        };
        float xq_next = load_xq(blockIdx.x);
        for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++tcount) {
            const int b = u / n_qt, q = (u % n_qt) * 128 + ql;
            const bool qok = q < Q;
            const float xq = xq_next;
            xq_next = load_xq(u + gridDim.x);
            // max logit: the nearest grid row (three candidates), as in the SIMT kernels
            float m = 0.f;
            if (qok) {
                const int n0 = (int)rintf(fminf(fmaxf((xq - x0) * inv_dx, 0.f), (float)(K - 1)));
                m = logit_t(xq, s_keys[n0], inv_sigma);
                if (n0 > 0) m = fmaxf(m, logit_t(xq, s_keys[n0 - 1], inv_sigma));
                if (n0 < K - 1) m = fmaxf(m, logit_t(xq, s_keys[n0 + 1], inv_sigma));
            }
            const float m2 = m * 1.4426950408889634f;
            float ssum = 0.f;
            for (int c = 0; c < n_chunks; ++c, ++g) {
                const int s = g & 1;
                if (g >= 2) mbar_wait(&bar_empty[s], ((g >> 1) - 1) & 1);
                uint8_t* w_hi = smem_raw + s * kStage;
                const float4* kp = reinterpret_cast<const float4*>(s_keys + c * kTcKeys + half * 32);     // broadcast reads; rows >= K hold +inf
#pragma unroll
                for (int j = 0; j < 4; ++j) {                     // 8 keys = one 16-byte bf16 chunk of row ql
                    const float4 ka = kp[2 * j], kb2 = kp[2 * j + 1];
                    const float kk[8] = {ka.x, ka.y, ka.z, ka.w, kb2.x, kb2.y, kb2.z, kb2.w};
                    float e[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float t = (kk[i] - xq) * is2;
                        float ev;
                        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ev) : "f"(fmaf(-t, t, -m2)));
                        e[i] = ev;
                        ssum += ev;
                    }
                    const uint32_t chunk = (uint32_t)(half * 4 + j);
                    split_store8(e, w_hi, w_hi + kWTile, (uint32_t)ql * 128u + ((chunk ^ (uint32_t)(ql & 7)) << 4));
                }
                fence_async_smem();
                if (c == n_chunks - 1) {                           // denominators of this unit, before the last chunk is released
                    const float tot = ssum + __shfl_xor_sync(0xffffffffu, ssum, 1);
                    if (half == 0) {
                        s_sum[tcount & 1][ql] = qok ? tot : 1.f;
                        if (qok) {
                            const long oq = (long)b * Q + q;
                            dens_o[oq] = expf(m) * tot;
                            mstat_o[oq * 2] = m; mstat_o[oq * 2 + 1] = tot;
                        }
                    }
                }
                mbar_arrive(&bar_wfull[s]);
            }
        }
    } else if (warp == kTcMmaWarp) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc(128, 128, 0, 1);     // A = E chunk (K-major), B = V chunk rows (MN-major view)
            int g = 0, tcount = 0;
            for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++tcount) {
                const int t = tcount & 1;
                mbar_wait(&bar_tempty[t], ((tcount >> 1) & 1) ^ 1);
                const uint32_t d = tmem + (uint32_t)t * 128u;
                for (int c = 0; c < n_chunks; ++c, ++g) {
                    const int s = g & 1;
                    const uint32_t par = (g >> 1) & 1;
                    mbar_wait(&bar_vfull[s], par);
                    mbar_wait(&bar_wfull[s], par);
                    tc_fence_after();
                    const uint32_t sw_hi = smem_u32(smem_raw + s * kStage), sw_lo = sw_hi + kWTile, sv_hi = sw_hi + 2 * kWTile, sv_lo = sv_hi + kVTile;
                    const uint64_t de_h = make_desc_sw128_t(sw_hi, 16, 1024), de_l = make_desc_sw128_t(sw_lo, 16, 1024);
                    const uint64_t dv_h = make_desc_sw128_t(sv_hi, 8192, 1024), dv_l = make_desc_sw128_t(sv_lo, 8192, 1024);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t a_h = desc_adv(de_h, ks * 32u), b_h = desc_adv(dv_h, ks * 2048u);
                        umma_bf16(d, a_h, b_h, idesc, (c | ks) ? 1u : 0u);
                        umma_bf16(d, a_h, desc_adv(dv_l, ks * 2048u), idesc, 1);
                        umma_bf16(d, desc_adv(de_l, ks * 32u), b_h, idesc, 1);
                    }
                    umma_commit(&bar_empty[s]);
                }
                umma_commit(&bar_tfull[t]);
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue: TMEM -> scale by 1 / s -> coalesced rows of feat
        const int e = warp - kTcEpiWarp0;
        const int lane_base = 32 * (warp & 3);
        const int col_base = (e >> 2) * 64;
        float* scratch = scratch_all + e * (32 * kTcScratchLd);
        const int r_in = lane >> 2, c4 = (lane & 3) * 4;
        int tcount = 0;
        for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++tcount) {
            const int t = tcount & 1;
            const int b = u / n_qt, q0 = (u % n_qt) * 128;
            mbar_wait(&bar_tfull[t], (tcount >> 1) & 1);
            tc_fence_after();
            const float inv = 1.f / s_sum[t][lane_base + lane];    // this thread's TMEM lane = query row
#pragma unroll 1
            for (int ch = 0; ch < 4; ++ch) {
                const int c0 = col_base + ch * 16;
                float v[16];
                tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(t * 128 + c0), v);
                if (ch == 3) {
                    tc_fence_before();
                    mbar_arrive(&bar_tempty[t]);
                }
#pragma unroll
                for (int j = 0; j < 16; j += 4)
                    *reinterpret_cast<float4*>(scratch + lane * kTcScratchLd + j) = make_float4(v[j] * inv, v[j + 1] * inv, v[j + 2] * inv, v[j + 3] * inv);
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int r = j * 8 + r_in;
                    const int q = q0 + lane_base + r;
                    if (q < Q)
                        *reinterpret_cast<float4*>(feat_o + ((long)b * Q + q) * C + c0 + c4) = *reinterpret_cast<const float4*>(scratch + r * kTcScratchLd + c4);
                }
                __syncwarp();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------------------------------------------------------
// Tensor-core BACKWARD for the induced -> target direction (C == 128, regular shared key grid, Q <= 128):
//     dV[b]     = P^T  . dF[b]              P[q,k]  = exp(a_qk - m_q) / s_q                       (value gradient)
//     d theta  ~= sum_{k,c} V[k,c] . dV2[k,c],   dV2 = E2^T . dF,   E2[q,k] = P[q,k] ((a_qk - m_q) - A1_q),
//                 A1_q = sum_k P[q,k] (a_qk - m_q)        (the softmax part of d theta: sum_q T_q - G_q A1_q of the SIMT kernels,
//                 with G_q = dF_q . feat_q folded in through A1 -- feat is not read at all)
//               + sum_{q,k} ddens_q exp(a_qk) a_qk        (the density part, accumulated by the threads that evaluate exp)
// Both products are [128 keys x Q queries] x [Q x 128 channels] GEMMs that share the B operand: the task's dF tile is staged
// ONCE (bf16 hi + lo, row-major = MN-major B) and the two generated left operands (P^T, E2^T: never stored anywhere) are
// written by the producer warps straight into SWIZZLE_128B K-major images, 64 queries per stage, 2-stage ring; the MMA
// warp accumulates hi.hi + hi.lo + lo.hi of both into two TMEM accumulators (double-buffered across key tiles: 512
// columns); the epilogue writes the dV tile as coalesced rows and reduces dV2 against the V rows it reads from HBM exactly
// once (V is an epilogue operand here, not an MMA operand).  HBM traffic per task: dF + V read once, dV written once
// (the SIMT pair read V + dF + feat and dF again).  Replaces setconv_task_kernel<1> + setconv_task_dv_kernel.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kBwProd = 16;                                   // producer warps (A-operand generation, dF staging)
constexpr int kBwMmaWarp = kBwProd;
constexpr int kBwEpiWarp0 = kBwProd + 1;
constexpr int kBwEpi = 8;
constexpr int kBwThreads = (kBwEpiWarp0 + kBwEpi) * 32;      // 800
constexpr uint32_t kBwImg = 128u * 64u * 2u;                  // one bf16 image of a [128 x 64] operand tile: 16 KB
constexpr uint32_t kBwStage = 4u * kBwImg;                    // P hi, P lo, E2 hi, E2 lo: 64 KB
constexpr uint32_t kBwF = 4u * kBwImg;                        // dF: (hi, lo) x 2 query chunks: 64 KB

// window_t() for a key grid that lives in SHARED memory (plain loads; __ldg is a global-space load)
__device__ __forceinline__ void window_s(const float* sk, int K, float xq, float sigma, int& lo_o, int& hi_o) {
    lo_o = 0; hi_o = K - 1;
    if (K < 3) return;
    const float x0 = sk[0], x1 = sk[K - 1];
    const float dx = (x1 - x0) / (float)(K - 1);
    if (!(dx > 0.f)) return;
    float pos = (xq - x0) / dx;
    pos = fminf(fmaxf(pos, 0.f), (float)(K - 1));
    const int n0 = (int)rintf(pos);
    const float dn = xq - sk[n0];
    const float D = sqrtf(dn * dn + kWindowLogT * sigma * sigma);
    float lo = floorf((xq - D - x0) / dx) - 1.f;
    float hi = ceilf((xq + D - x0) / dx) + 1.f;
    if (!(lo == lo) || !(hi == hi)) return;
    lo = fminf(fmaxf(lo, 0.f), (float)(K - 1));
    hi = fminf(fmaxf(hi, 0.f), (float)(K - 1));
    lo_o = min((int)lo, n0);
    hi_o = max((int)hi, n0);
}

__device__ __forceinline__ void prod_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kBwProd * 32) : "memory"); }

__global__ void __launch_bounds__(kBwThreads, 1) setconv_tc_bwd_kernel(const float* __restrict__ keys, const float* __restrict__ queries, long qry_bs,
                                                                      const float* __restrict__ values, const float* __restrict__ theta,
                                                                      const float* __restrict__ mstat, const float* __restrict__ dfeat,
                                                                      const float* __restrict__ ddens, float* __restrict__ dvalues,
                                                                      float* __restrict__ dtheta, int B, int K, int Q) {
    constexpr int C = 128;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_afull[2], bar_aempty[2], bar_ffull, bar_fempty, bar_tfull[2], bar_tempty[2];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float s_keys[kMaxChunks * kChunkRows];
    __shared__ __align__(16) float4 s_qa[128];                // (x_q, m_q log2 e, 1 / s_q, A1_q)
    __shared__ __align__(16) float2 s_qb[128];                // (ddens_q exp(m_q), m_q)
    __shared__ float s_part[kBwThreads / 32];

    uint8_t* sA = smem_raw;                                   // 2 stages x 64 KB
    uint8_t* sF = smem_raw + 2 * kBwStage;                    // dF images: [chunk][hi 16K | ...]: hi(c0) hi(c1) lo(c0) lo(c1)
    float* scratch_all = reinterpret_cast<float*>(smem_raw + 2 * kBwStage + kBwF);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    if (tid == 32) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_afull[i], kBwProd * 32);
            mbar_init(&bar_aempty[i], 1);
            mbar_init(&bar_tfull[i], 1);
            mbar_init(&bar_tempty[i], kBwEpi * 32);
        }
        mbar_init(&bar_ffull, kBwProd * 32);
        mbar_init(&bar_fempty, 1);
    }
    const float th = __ldg(theta);
    const float sigma = 1e-5f + softplus_f(th);
    const float inv_sigma = 1.f / sigma;
    const int n_kt = (K + 127) >> 7;                          // key tiles per task
    const int n_qc = (Q + 63) >> 6;                           // 64-query chunks per task (1 or 2)
    const int n_tiles = B * n_kt;
    // contiguous, balanced tile ranges: the first n_tiles % grid CTAs take one tile more
    const int per = n_tiles / (int)gridDim.x, rem = n_tiles - per * (int)gridDim.x;
    const int g0 = (int)blockIdx.x * per + min((int)blockIdx.x, rem), g1 = g0 + per + ((int)blockIdx.x < rem ? 1 : 0);
    pdl_trigger();
    for (int i = tid; i < K; i += kBwThreads) s_keys[i] = __ldg(keys + i);     // the grid is an input of the step
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    pdl_wait();

    float part = 0.f;                                         // this thread's share of the d theta sum

    if (warp < kBwProd) {
        // ------------------------------------------------------------------ producers
        const int r = tid & 127, quarter = tid >> 7;           // key row of the tile; queries [16 quarter, 16 quarter + 16) of a chunk
        const float is2 = inv_sigma * 1.2011224087864498f;     // exp(a - m) = exp2(-(d is2)^2 - m log2 e)
        const int fw = warp & 7, fc = warp >> 3;               // dF staging: rows 8 fw .. 8 fw + 7 of query chunk fc
        const uint32_t vchunk = (uint32_t)(lane >> 1) & 7u;
        const uint32_t voff = (uint32_t)fc * kBwImg + (uint32_t)(lane >> 4) * 8192u + (uint32_t)(fw * 8) * 128u + (uint32_t)(lane & 1) * 8u;
        int ga = 0, ntask = 0, cur_b = -1;
        float nq_x = 0.f, nq_m = 0.f, nq_s = 1.f, nq_d = 0.f;       // query record of the next task (threads 0..127: one query each)
        auto load_qrec = [&](int bb) {
            if (tid < 128 && tid < Q) {
                const long oq = (long)bb * Q + tid;
                nq_x = __ldg(queries + (long)bb * qry_bs + tid);
                nq_m = __ldg(mstat + oq * 2);
                nq_s = __ldg(mstat + oq * 2 + 1);
                nq_d = __ldg(ddens + oq);
            }
        };
        if (g0 < g1) load_qrec(g0 / n_kt);
        for (int g = g0; g < g1; ++g) {
            const int b = g / n_kt, kt = g - b * n_kt;
            for (int gp = (g == g0 ? g : g + 1); gp <= g + 1 && gp < g1; ++gp) {   // the value rows of the NEXT tile (epilogue operand) -> L2, one tile ahead
                const int bp = gp / n_kt, ktp = gp - bp * n_kt;
                const int rows = min(128, K - ktp * 128);
                const char* vbase = reinterpret_cast<const char*>(values + ((long)bp * K + ktp * 128) * C);
                for (int l = tid; l < rows * 4; l += kBwProd * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(vbase + ((long)l << 7)));
            }
            if (b != cur_b) {
                cur_b = b;
                prod_sync();                                   // everyone is done with the previous task's query records
                float4 f[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int q = fc * 64 + fw * 8 + i;
                    f[i] = q < Q ? __ldg(reinterpret_cast<const float4*>(dfeat + ((long)b * Q + q) * C) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                if (tid < 128) {
                    const int q = tid;
                    float xq = s_keys[0], m = 0.f, invs = 0.f, dd = 0.f;       // padding queries: every generated weight is exactly 0
                    if (q < Q) {                                                // fetched one task ahead (nq_*): no load latency here
                        xq = nq_x; m = nq_m;
                        invs = 1.f / nq_s;
                        dd = nq_d * expf(m);
                    }
                    s_qa[q] = make_float4(xq, m * 1.4426950408889634f, invs, 0.f);
                    s_qb[q] = make_float2(dd, m);
                }
                if ((b + 1) * n_kt < g1) {                                      // the NEXT task of this CTA: query records -> registers, dF rows -> L2
                    load_qrec(b + 1);
                    const char* fbase = reinterpret_cast<const char*>(dfeat + (long)(b + 1) * Q * C);
                    for (int l = tid; l < Q * 4; l += kBwProd * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(fbase + ((long)l << 7)));
                }
                prod_sync();
                {   // A1_q = sum_k P_qk (a_qk - m_q) over the query's sigma-window: 4 threads per query
                    const int q = tid >> 2, kp = tid & 3;
                    const float4 qa = s_qa[q];
                    int lo, hi;
                    window_s(s_keys, K, qa.x, sigma, lo, hi);
                    float a1 = 0.f;
                    for (int k = lo + kp; k <= hi; k += 4) {
                        const float t = (s_keys[k] - qa.x) * is2;
                        const float l2 = fmaf(-t, t, -qa.y);
                        float e;
                        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(l2));
                        a1 = fmaf(e, l2, a1);
                    }
                    a1 += __shfl_xor_sync(0xffffffffu, a1, 1);
                    a1 += __shfl_xor_sync(0xffffffffu, a1, 2);
                    if (kp == 0) s_qa[q].w = (q < Q) ? a1 * qa.z * 0.6931471805599453f : 0.f;
                }
                if (ntask >= 1) mbar_wait(&bar_fempty, (uint32_t)(ntask - 1) & 1u);      // the previous task's MMAs no longer read the dF images
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const uint32_t off = voff + (uint32_t)i * 128u + ((vchunk ^ (uint32_t)i) << 4);
                    const uint32_t h01 = pack_bf16(f[i].x, f[i].y), h23 = pack_bf16(f[i].z, f[i].w);
                    *reinterpret_cast<uint2*>(sF + off) = make_uint2(h01, h23);
                    *reinterpret_cast<uint2*>(sF + 2 * kBwImg + off) =
                        make_uint2(pack_bf16(f[i].x - __uint_as_float(h01 << 16), f[i].y - __uint_as_float(h01 & 0xFFFF0000u)),
                                   pack_bf16(f[i].z - __uint_as_float(h23 << 16), f[i].w - __uint_as_float(h23 & 0xFFFF0000u)));
                }
                fence_async_smem();
                mbar_arrive(&bar_ffull);
                ++ntask;
                prod_sync();                                   // A1 visible to every producer
            }
            const int key = kt * 128 + r;
            const bool kok = key < K;
            const float xk = s_keys[kok ? key : 0];
            for (int c = 0; c < n_qc; ++c, ++ga) {
                const int s = ga & 1;
                if (ga >= 2) mbar_wait(&bar_aempty[s], (uint32_t)((ga >> 1) - 1) & 1u);
                uint8_t* st_base = sA + (uint32_t)s * kBwStage;
#pragma unroll
                for (int jj = 0; jj < 2; ++jj) {
                    const int j = quarter * 2 + jj;            // 16-byte chunk of the row = 8 queries
                    float pv[8], ev[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int q = c * 64 + j * 8 + i;
                        const float4 qa = s_qa[q];             // broadcast: every lane of the warp reads the same query record
                        const float2 qb = s_qb[q];
                        const float t = (xk - qa.x) * is2;
                        const float l2 = fmaf(-t, t, -qa.y);
                        float e;
                        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(l2));
                        e = kok ? e : 0.f;
                        const float am = l2 * 0.6931471805599453f;     // a - m
                        const float p = e * qa.z;
                        pv[i] = p;
                        ev[i] = p * (am - qa.w);
                        part = fmaf((am + qb.y) * e, qb.x, part);      // ddens_q exp(a_qk) a_qk
                    }
                    const uint32_t off = (uint32_t)r * 128u + (((uint32_t)j ^ (uint32_t)(r & 7)) << 4);
                    split_store8(pv, st_base, st_base + kBwImg, off);
                    split_store8(ev, st_base + 2 * kBwImg, st_base + 3 * kBwImg, off);
                }
                fence_async_smem();
                mbar_arrive(&bar_afull[s]);
            }
        }
    } else if (warp == kBwMmaWarp) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc(128, 128, 0, 1);     // A = generated tile (K-major), B = dF rows (MN-major view)
            const uint32_t sf = smem_u32(sF);
            int ga = 0, tc = 0, ntask = 0, cur_b = -1;
            for (int g = g0; g < g1; ++g, ++tc) {
                const int b = g / n_kt;
                if (b != cur_b) {
                    cur_b = b;
                    mbar_wait(&bar_ffull, (uint32_t)ntask & 1u);
                    ++ntask;
                }
                const int t = tc & 1;
                mbar_wait(&bar_tempty[t], (uint32_t)((tc >> 1) & 1) ^ 1u);
                const uint32_t d_v = tmem + (uint32_t)t * 256u, d_e = d_v + 128u;
                for (int c = 0; c < n_qc; ++c, ++ga) {
                    const int s = ga & 1;
                    mbar_wait(&bar_afull[s], (uint32_t)(ga >> 1) & 1u);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(sA + (uint32_t)s * kBwStage);
                    const uint32_t f_hi = sf + (uint32_t)c * kBwImg, f_lo = f_hi + 2 * kBwImg;
                    const uint64_t db_h = make_desc_sw128_t(f_hi, 8192, 1024), db_l = make_desc_sw128_t(f_lo, 8192, 1024);
                    const uint64_t dp_h = make_desc_sw128_t(sa, 16, 1024), dp_l = make_desc_sw128_t(sa + kBwImg, 16, 1024);
                    const uint64_t de_h = make_desc_sw128_t(sa + 2 * kBwImg, 16, 1024), de_l = make_desc_sw128_t(sa + 3 * kBwImg, 16, 1024);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t b_h = desc_adv(db_h, ks * 2048u), b_l = desc_adv(db_l, ks * 2048u);
                        const uint64_t p_h = desc_adv(dp_h, ks * 32u), p_l = desc_adv(dp_l, ks * 32u);
                        const uint64_t e_h = desc_adv(de_h, ks * 32u), e_l = desc_adv(de_l, ks * 32u);
                        const uint32_t acc = (c | ks) ? 1u : 0u;
                        umma_bf16(d_v, p_h, b_h, idesc, acc);
                        umma_bf16(d_v, p_h, b_l, idesc, 1);
                        umma_bf16(d_v, p_l, b_h, idesc, 1);
                        umma_bf16(d_e, e_h, b_h, idesc, acc);
                        umma_bf16(d_e, e_h, b_l, idesc, 1);
                        umma_bf16(d_e, e_l, b_h, idesc, 1);
                    }
                    umma_commit(&bar_aempty[s]);
                }
                umma_commit(&bar_tfull[t]);
                if (g + 1 == g1 || (g + 1) / n_kt != b) umma_commit(&bar_fempty);      // last tile of the task: the dF images may be replaced
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue: dV rows out, dV2 . V reduced into d theta
        const int e = warp - kBwEpiWarp0;
        const int lane_base = 32 * (warp & 3);
        const int col_base = (e >> 2) * 64;
        float* scratch = scratch_all + e * (32 * kTcScratchLd);
        const int r_in = lane >> 2, c4 = (lane & 3) * 4;
        int tc = 0;
        // The V pieces this thread meets after the transpose are fetched FAR ahead of their use: two column chunks are always in
        // flight in registers, issued before the tile's dV half (4 TMEM drains + stores) or two dV2 chunks earlier, so an L2 /
        // DRAM round trip (~1-2.5 k cycles under load) is covered by several hundred-cycle epilogue steps instead of one.
        auto vload = [&](int g, int ch, float4 (&dst)[4]) {
            const int b = g / n_kt, kt = g - b * n_kt;
            const long row0 = (long)b * K + kt * 128 + lane_base;
            const int rows_ok = K - (kt * 128 + lane_base);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int rr = j * 8 + r_in;
                dst[j] = rr < rows_ok ? __ldg(reinterpret_cast<const float4*>(values + (row0 + rr) * C + col_base + ch * 16 + c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        float4 va[4], vb[4];
        if (g0 < g1) { vload(g0, 0, va); vload(g0, 1, vb); }
        for (int g = g0; g < g1; ++g, ++tc) {
            const int t = tc & 1;
            const int b = g / n_kt, kt = g - b * n_kt;
            const long row0 = (long)b * K + kt * 128 + lane_base;          // global row of this warp's TMEM lane 0
            const int rows_ok = K - (kt * 128 + lane_base);                // rows [0, rows_ok) of the warp's 32 exist
            mbar_wait(&bar_tfull[t], (uint32_t)(tc >> 1) & 1u);
            tc_fence_after();
            // ---- value gradient: TMEM -> per-warp transpose -> coalesced rows of dV
#pragma unroll 1
            for (int ch = 0; ch < 4; ++ch) {
                const int c0 = col_base + ch * 16;
                float v[16];
                tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(t * 256 + c0), v);
#pragma unroll
                for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(scratch + lane * kTcScratchLd + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int rr = j * 8 + r_in;
                    if (rr < rows_ok)
                        *reinterpret_cast<float4*>(dvalues + (row0 + rr) * C + c0 + c4) = *reinterpret_cast<const float4*>(scratch + rr * kTcScratchLd + c4);
                }
                __syncwarp();
            }
            // ---- d theta: sum of dV2 (.) V over the tile
            auto dot_chunk = [&](int ch, const float4 (&vv)[4], bool last) {
                float v[16];
                tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(t * 256 + 128 + col_base + ch * 16), v);
                if (last) {                                                 // both accumulators of buffer t are drained
                    tc_fence_before();
                    mbar_arrive(&bar_tempty[t]);
                }
#pragma unroll
                for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(scratch + lane * kTcScratchLd + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int rr = j * 8 + r_in;
                    const float4 d2 = *reinterpret_cast<const float4*>(scratch + rr * kTcScratchLd + c4);
                    part = fmaf(d2.x, vv[j].x, part); part = fmaf(d2.y, vv[j].y, part);
                    part = fmaf(d2.z, vv[j].z, part); part = fmaf(d2.w, vv[j].w, part);
                }
                __syncwarp();
            };
            dot_chunk(0, va, false);
            vload(g, 2, va);
            dot_chunk(1, vb, false);
            vload(g, 3, vb);
            dot_chunk(2, va, false);
            if (g + 1 < g1) vload(g + 1, 0, va);
            dot_chunk(3, vb, true);
            if (g + 1 < g1) vload(g + 1, 1, vb);
        }
    }
    part = warp_sum(part);
    if (lane == 0) s_part[warp] = part;
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
        float tot = 0.f;
        for (int i = 0; i < kBwThreads / 32; ++i) tot += s_part[i];
        atomicAdd(dtheta, tot * (-2.f / sigma) * sigmoid_f(th));
    }
    if (warp == 0) tmem_dealloc(tmem, 512);
}

static bool tc_bwd_ok(int K, int Q, int C, long key_bs) {
    return C == 128 && key_bs == 0 && K >= 3 && K <= kMaxChunks * kChunkRows && Q >= 1 && Q <= 128;
}

static bool tc_fwd_ok(int K, int Q, int C, long key_bs) {
    (void)Q;
    return C == 128 && key_bs == 0 && K <= kMaxChunks * kChunkRows && K > 2 * kTcKeys;     // >= 3 chunks: the per-unit denominators are double-buffered against the 2-stage ring
}

static size_t task_smem_fwd(int K, int Q) {
    return sizeof(float) * ((size_t)((K + kChunkRows - 1) / kChunkRows) * kChunkRows * 128 + (size_t)kTaskWarps * kChunkRows * kGroup + 11 * (size_t)Q);
}
static size_t task_smem_dv(int Q) { return sizeof(float) * ((size_t)Q * 128 + (size_t)kTaskWarps * kChunkRows * kGroup + 11 * (size_t)Q); }
constexpr size_t kTaskSmemMax = 226 * 1024;     // 227 KB per CTA minus the static barriers (K = 384 rows of V need 218.6 KB)
static bool task_ok(int K, int Q, int C) { return C == 128 && K <= kMaxChunks * kChunkRows && K < 32768 && task_smem_fwd(K, Q) <= kTaskSmemMax; }

static bool tile_ok(int K, int Q, int C, const void* values) {
    return C % 4 == 0 && C >= 8 && C <= 128 && Q >= 1 && Q <= kMaxQ && K >= 3 && (reinterpret_cast<uintptr_t>(values) & 15) == 0;
}
static size_t tile_smem(int Q) { return sizeof(float) * 7 * (size_t)Q; }
// CTAs per task: enough to give every SM ~4 CTAs, but never fewer than one 8-warp pass of groups per CTA
static unsigned split_for(int B, int n_groups) {
    long s = cdiv(4L * kNumSMs, B);
    const long max_s = cdiv(n_groups, 8);
    if (s > max_s) s = max_s;
    if (s < 1) s = 1;
    return (unsigned)s;
}

int setconv_tile_fwd(const float* keys, long key_bs, const float* queries, long qry_bs, const float* values,
                     const float* theta, float* feat, float* dens, float* mstat, int B, int K, int Q, int C,
                     cudaStream_t st) {
    if (!tile_ok(K, Q, C, values) || (reinterpret_cast<uintptr_t>(feat) & 15)) return NPF_ENOTSUP;
    if (tc_fwd_ok(K, Q, C, key_bs)) {
        static bool cattr = false;
        if (!cattr) { cudaFuncSetAttribute(setconv_tc_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024); cattr = true; }
        const int units = B * ((Q + 127) / 128);
        const size_t smem = 2 * 65536 + (size_t)kTcEpi * 32 * kTcScratchLd * sizeof(float) + 2 * (size_t)kTcKeys * 128 * sizeof(float);
        launch_pdl(setconv_tc_fwd_kernel, dim3(units < kNumSMs ? units : kNumSMs), dim3(kTcThreads + 32), smem, st, keys, key_bs, queries, qry_bs, values, theta, feat, dens,
                   mstat, B, K, Q);
        count_launch();
        return check_launch("setconv_tc_fwd_kernel");
    }
    if (task_ok(K, Q, C)) {
        static bool tattr = false;
        if (!tattr) { cudaFuncSetAttribute(setconv_task_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTaskSmemMax); tattr = true; }
        setconv_task_kernel<0><<<B < kNumSMs ? B : kNumSMs, kTaskThreads, task_smem_fwd(K, Q), st>>>(keys, key_bs, queries, qry_bs, values, theta, feat, dens, mstat,
                                                                                                     nullptr, nullptr, nullptr, nullptr, nullptr, B, K, Q);
        count_launch();
        return check_launch("setconv_task_kernel<fwd>");
    }
    const size_t smem = tile_smem(Q);
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(setconv_grp_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024); attr = true; }
    setconv_grp_kernel<0><<<dim3(B, split_for(B, (Q + kGroup - 1) / kGroup)), 256, smem, st>>>(keys, key_bs, queries, qry_bs, values, theta, feat, dens, mstat, nullptr, nullptr,
                                                nullptr, nullptr, nullptr, K, Q, C);
    count_launch();
    return check_launch("setconv_grp_kernel<fwd>");
}

int setconv_tile_bwd(const float* keys, long key_bs, const float* queries, long qry_bs, const float* values,
                     const float* theta, const float* feat, const float* mstat, const float* dfeat,
                     const float* ddens, float* dvalues, float* dtheta, int B, int K, int Q, int C, cudaStream_t st) {
    if (!tile_ok(K, Q, C, values) || (reinterpret_cast<uintptr_t>(dfeat) & 15) || (reinterpret_cast<uintptr_t>(feat) & 15) ||
        (dvalues && (reinterpret_cast<uintptr_t>(dvalues) & 15)))
        return NPF_ENOTSUP;
    if (dvalues && tc_bwd_ok(K, Q, C, key_bs)) {
        const size_t smem = 2 * kBwStage + kBwF + (size_t)kBwEpi * 32 * kTcScratchLd * sizeof(float);
        static bool battr = false;
        if (!battr) { cudaFuncSetAttribute(setconv_tc_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); battr = true; }
        const int n_tiles = B * ((K + 127) / 128);
        launch_pdl(setconv_tc_bwd_kernel, dim3(n_tiles < kNumSMs ? n_tiles : kNumSMs), dim3(kBwThreads), smem, st, keys, queries, qry_bs, values, theta, mstat, dfeat,
                   ddens, dvalues, dtheta, B, K, Q);
        count_launch();
        return check_launch("setconv_tc_bwd_kernel");
    }
    if (task_ok(K, Q, C)) {
        static bool tattr = false;
        if (!tattr) {
            cudaFuncSetAttribute(setconv_task_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTaskSmemMax);
            cudaFuncSetAttribute(setconv_task_dv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTaskSmemMax);
            tattr = true;
        }
        const int grid = B < kNumSMs ? B : kNumSMs;
        setconv_task_kernel<1><<<grid, kTaskThreads, task_smem_fwd(K, Q), st>>>(keys, key_bs, queries, qry_bs, values, theta, nullptr, nullptr, nullptr, feat, mstat,
                                                                              dfeat, ddens, dtheta, B, K, Q);
        count_launch();
        int rc = check_launch("setconv_task_kernel<dtheta>");
        if (rc != NPF_OK || !dvalues) return rc;
        if (task_smem_dv(Q) <= kTaskSmemMax) {
            setconv_task_dv_kernel<<<grid, kTaskThreads, task_smem_dv(Q), st>>>(keys, key_bs, queries, qry_bs, theta, mstat, dfeat, dvalues, B, K, Q);
            count_launch();
            return check_launch("setconv_task_dv_kernel");
        }
        static bool dattr = false;
        if (!dattr) { cudaFuncSetAttribute(setconv_grp_dv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024); dattr = true; }
        setconv_grp_dv_kernel<<<dim3(B, split_for(B, (K + kGroup - 1) / kGroup)), 256, tile_smem(Q), st>>>(keys, key_bs, queries, qry_bs, theta, mstat, dfeat, dvalues, K, Q, C);
        count_launch();
        return check_launch("setconv_grp_dv_kernel");
    }
    const size_t smem = tile_smem(Q);
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(setconv_grp_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        cudaFuncSetAttribute(setconv_grp_dv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        attr = true;
    }
    setconv_grp_kernel<1><<<dim3(B, split_for(B, (Q + kGroup - 1) / kGroup)), 256, smem, st>>>(keys, key_bs, queries, qry_bs, values, theta, nullptr, nullptr, nullptr, feat, mstat,
                                                dfeat, ddens, dtheta, K, Q, C);
    count_launch();
    int rc = check_launch("setconv_grp_kernel<dtheta>");
    if (rc != NPF_OK || !dvalues) return rc;
    setconv_grp_dv_kernel<<<dim3(B, split_for(B, (K + kGroup - 1) / kGroup)), 256, smem, st>>>(keys, key_bs, queries, qry_bs, theta, mstat, dfeat, dvalues, K, Q, C);
    count_launch();
    return check_launch("setconv_grp_dv_kernel");
}

}  // namespace npf
