// SetConv with the exponential-quadratic RBF (upstream npf/architectures/setcnn.py:126-142, 234-268), x_dim == 1.
//
//   sigma = 1e-5 + softplus(theta);  a_qk = -((x_q - x_k)/sigma)^2
//   feat[b,q,:] = sum_k softmax_k(a_qk) V[b,k,:]        dens[b,q] = sum_k exp(a_qk)
//
// The reference materialises weight*values as a [B,Q,K,C] tensor (71 % of its ConvCNP step).  Here nothing of
// size Q*K ever reaches memory: one warp owns one query, streams the keys it needs and keeps the C running sums
// in registers.  For a regular key grid (induced points) only the run-time sigma-window of keys whose softmax
// weight is >= 2^-60 of the largest is visited -- exact in fp32.
//
// Generic kernels (any K, Q, C <= 256).  The shared-memory/TMA-staged fast path for the induced->target direction
// is in setconv_tile.cu.
#include "common.cuh"

namespace npf {

constexpr float kWindowLog = 41.6f;  // exp(-41.6) ~ 2^-60
constexpr int kMaxChunks = 8;        // C <= 256

struct Window { int lo, hi; };

__device__ __forceinline__ float logit(float xq, float xk, float sigma) {
    const float t = fabsf(xk - xq) / sigma;  // same op order as dist/sigma then pow(2), setcnn.py:129-134
    return -(t * t);
}

// Key range that can carry weight for query xq on a regular increasing grid; whole range otherwise.
__device__ __forceinline__ Window key_window(const float* __restrict__ keys, int K, float xq, float sigma, int regular) {
    Window w{0, K - 1};
    if (!regular || K < 3) return w;
    const float x0 = __ldg(keys), x1 = __ldg(keys + K - 1);
    const float dx = (x1 - x0) / (float)(K - 1);
    if (!(dx > 0.f)) return w;
    float pos = (xq - x0) / dx;
    pos = fminf(fmaxf(pos, 0.f), (float)(K - 1));
    const int n0 = (int)rintf(pos);
    const float dn = xq - __ldg(keys + n0);
    const float D = sqrtf(dn * dn + kWindowLog * sigma * sigma);
    float lo = floorf((xq - D - x0) / dx) - 1.f;
    float hi = ceilf((xq + D - x0) / dx) + 1.f;
    if (!(lo == lo) || !(hi == hi)) return w;  // NaN guard
    lo = fminf(fmaxf(lo, 0.f), (float)(K - 1));
    hi = fminf(fmaxf(hi, 0.f), (float)(K - 1));
    w.lo = (int)lo; w.hi = (int)hi;
    if (w.lo > n0) w.lo = n0;
    if (w.hi < n0) w.hi = n0;
    return w;
}

// ----------------------------------------------------------------------------------------------------------------
// forward: one warp per query
// ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) setconv_fwd_kernel(const float* __restrict__ keys, long key_bs,
                                                          const float* __restrict__ queries, long qry_bs,
                                                          const float* __restrict__ values, const float* __restrict__ theta,
                                                          float* __restrict__ feat, float* __restrict__ dens,
                                                          float* __restrict__ mstat, int K, int Q, int C, int regular) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * 8 + warp;
    const int b = blockIdx.y;
    if (q >= Q) return;
    const float sigma = 1e-5f + softplus_f(__ldg(theta));
    const float* kb = keys + (long)b * key_bs;
    const float xq = __ldg(queries + (long)b * qry_bs + q);
    const Window w = key_window(kb, K, xq, sigma, regular);
    const float* vb = values + (long)b * K * C;

    // pass 1: max logit, sum exp(a - m), sum exp(a)
    float m = -INFINITY;
    for (int k = w.lo + lane; k <= w.hi; k += 32) m = fmaxf(m, logit(xq, __ldg(kb + k), sigma));
    m = warp_max(m);
    float s = 0.f, d = 0.f;
    for (int k = w.lo + lane; k <= w.hi; k += 32) {
        const float a = logit(xq, __ldg(kb + k), sigma);
        s += expf(a - m);
        d += expf(a);
    }
    s = warp_sum(s);
    d = warp_sum(d);
    const float inv_s = 1.f / s;
    const long oq = (long)b * Q + q;

    if (C <= 4) {
        // few channels (context -> induced): lanes own keys
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int k = w.lo + lane; k <= w.hi; k += 32) {
            const float e = expf(logit(xq, __ldg(kb + k), sigma) - m);
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (c < C) acc[c] = fmaf(e, __ldg(vb + (long)k * C + c), acc[c]);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            acc[c] = warp_sum(acc[c]);
            if (c < C && lane == 0) feat[oq * C + c] = acc[c] * inv_s;
        }
    } else {
        // many channels (induced -> target): lanes own channels, keys are broadcast by shuffle
        const int nch = (C + 31) >> 5;
        float acc[kMaxChunks];
#pragma unroll
        for (int i = 0; i < kMaxChunks; ++i) acc[i] = 0.f;
        for (int base = w.lo; base <= w.hi; base += 32) {
            const int kmine = base + lane;
            const float e_mine = (kmine <= w.hi) ? expf(logit(xq, __ldg(kb + kmine), sigma) - m) : 0.f;
            const int cnt = min(32, w.hi - base + 1);
            for (int j = 0; j < cnt; ++j) {
                const float e = __shfl_sync(0xffffffffu, e_mine, j);
                const float* vr = vb + (long)(base + j) * C;
#pragma unroll
                for (int i = 0; i < kMaxChunks; ++i) {
                    const int c = lane + 32 * i;
                    if (i < nch && c < C) acc[i] = fmaf(e, __ldg(vr + c), acc[i]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < kMaxChunks; ++i) {
            const int c = lane + 32 * i;
            if (i < nch && c < C) feat[oq * C + c] = acc[i] * inv_s;
        }
    }
    if (lane == 0) {
        dens[oq] = d;
        mstat[oq * 2 + 0] = m;
        mstat[oq * 2 + 1] = s;
    }
}

// ----------------------------------------------------------------------------------------------------------------
// backward w.r.t. theta: one warp per query, block partials -> one atomic per CTA
//   dsigma = (-2/sigma) * sum_q [ T_q - G_q*A1_q + ddens_q*A2_q ]
//   T_q = dF_q . sum_k w_qk (a_qk - m_q) V_k ;  G_q = dF_q . feat_q ;  A1_q = sum_k w_qk (a_qk - m_q) ;
//   A2_q = sum_k e^{a_qk} a_qk.   The softmax part is sum_k w_k a_k (g_k - G); because sum_k w_k (g_k - G) = 0 the
//   logits may be shifted by any constant: shifting by the max logit m_q keeps both products O(1) instead of
//   O((d/sigma)^2) and removes the catastrophic cancellation (exactly 0 for a single key, like autograd's softmax).
// ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) setconv_bwd_theta_kernel(const float* __restrict__ keys, long key_bs,
                                                                const float* __restrict__ queries, long qry_bs,
                                                                const float* __restrict__ values, const float* __restrict__ theta,
                                                                const float* __restrict__ feat, const float* __restrict__ mstat,
                                                                const float* __restrict__ dfeat, const float* __restrict__ ddens,
                                                                float* __restrict__ dtheta, int K, int Q, int C, int regular) {
    __shared__ float part[8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * 8 + warp;
    const int b = blockIdx.y;
    const float th = __ldg(theta);
    const float sigma = 1e-5f + softplus_f(th);
    float contrib = 0.f;
    if (q < Q) {
        const float* kb = keys + (long)b * key_bs;
        const float xq = __ldg(queries + (long)b * qry_bs + q);
        const Window w = key_window(kb, K, xq, sigma, regular);
        const float* vb = values + (long)b * K * C;
        const long oq = (long)b * Q + q;
        const float m = __ldg(mstat + oq * 2), inv_s = 1.f / __ldg(mstat + oq * 2 + 1);
        const float* dF = dfeat + oq * C;
        float A1 = 0.f, A2 = 0.f, T = 0.f, G = 0.f;
        for (int c = lane; c < C; c += 32) G = fmaf(__ldg(dF + c), __ldg(feat + oq * C + c), G);
        if (C <= 4) {
            float df[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) df[c] = (c < C) ? __ldg(dF + c) : 0.f;
            for (int k = w.lo + lane; k <= w.hi; k += 32) {
                const float a = logit(xq, __ldg(kb + k), sigma);
                const float wa = expf(a - m) * inv_s * (a - m);
                A1 += wa;
                A2 = fmaf(expf(a), a, A2);
                float g = 0.f;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (c < C) g = fmaf(df[c], __ldg(vb + (long)k * C + c), g);
                T = fmaf(wa, g, T);
            }
        } else {
            const int nch = (C + 31) >> 5;
            float df[kMaxChunks];
#pragma unroll
            for (int i = 0; i < kMaxChunks; ++i) {
                const int c = lane + 32 * i;
                df[i] = (i < nch && c < C) ? __ldg(dF + c) : 0.f;
            }
            for (int base = w.lo; base <= w.hi; base += 32) {
                const int kmine = base + lane;
                float wa_mine = 0.f;
                if (kmine <= w.hi) {
                    const float a = logit(xq, __ldg(kb + kmine), sigma);
                    wa_mine = expf(a - m) * inv_s * (a - m);
                    A1 += wa_mine;
                    A2 = fmaf(expf(a), a, A2);
                }
                const int cnt = min(32, w.hi - base + 1);
                for (int j = 0; j < cnt; ++j) {
                    const float wa = __shfl_sync(0xffffffffu, wa_mine, j);
                    const float* vr = vb + (long)(base + j) * C;
                    float g = 0.f;
#pragma unroll
                    for (int i = 0; i < kMaxChunks; ++i) {
                        const int c = lane + 32 * i;
                        if (i < nch && c < C) g = fmaf(df[i], __ldg(vr + c), g);
                    }
                    T = fmaf(wa, g, T);
                }
            }
        }
        A1 = warp_sum(A1); A2 = warp_sum(A2); T = warp_sum(T); G = warp_sum(G);
        contrib = T - G * A1 + __ldg(ddens + oq) * A2;
    }
    if (lane == 0) part[warp] = contrib;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) tot += part[i];
        // dsigma/dtheta = sigmoid(theta)
        atomicAdd(dtheta, tot * (-2.f / sigma) * sigmoid_f(th));
    }
}

// ----------------------------------------------------------------------------------------------------------------
// backward w.r.t. values: gather form, one warp per key row.  dV[b,k,:] = sum_q w_qk dF[b,q,:]
// lanes first evaluate w_qk for 32 queries at a time; rows visit only the queries with non-negligible weight.
// ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) setconv_bwd_values_kernel(const float* __restrict__ keys, long key_bs,
                                                                 const float* __restrict__ queries, long qry_bs,
                                                                 const float* __restrict__ theta, const float* __restrict__ mstat,
                                                                 const float* __restrict__ dfeat, float* __restrict__ dvalues,
                                                                 int K, int Q, int C) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int k = blockIdx.x * 8 + warp;
    const int b = blockIdx.y;
    if (k >= K) return;
    const float sigma = 1e-5f + softplus_f(__ldg(theta));
    const float xk = __ldg(keys + (long)b * key_bs + k);
    const float* qb = queries + (long)b * qry_bs;
    const int nch = (C + 31) >> 5;
    float acc[kMaxChunks];
#pragma unroll
    for (int i = 0; i < kMaxChunks; ++i) acc[i] = 0.f;
    for (int base = 0; base < Q; base += 32) {
        const int qm = base + lane;
        float w_mine = 0.f;
        if (qm < Q) {
            const long oq = (long)b * Q + qm;
            const float a = logit(__ldg(qb + qm), xk, sigma);
            w_mine = expf(a - __ldg(mstat + oq * 2)) / __ldg(mstat + oq * 2 + 1);
        }
        unsigned live = __ballot_sync(0xffffffffu, w_mine > 0.f);
        while (live) {
            const int j = __ffs(live) - 1;
            live &= live - 1;
            const float wq = __shfl_sync(0xffffffffu, w_mine, j);
            const float* dF = dfeat + ((long)b * Q + base + j) * C;
#pragma unroll
            for (int i = 0; i < kMaxChunks; ++i) {
                const int c = lane + 32 * i;
                if (i < nch && c < C) acc[i] = fmaf(wq, __ldg(dF + c), acc[i]);
            }
        }
    }
    float* out = dvalues + ((long)b * K + k) * C;
#pragma unroll
    for (int i = 0; i < kMaxChunks; ++i) {
        const int c = lane + 32 * i;
        if (i < nch && c < C) out[c] = acc[i];
    }
}

// ----------------------------------------------------------------------------------------------------------------
// Few value channels (context -> induced: C = y_dim <= 4): one THREAD per query, the task's keys and values staged in
// shared memory (broadcast reads).  mode 0 forward, mode 1 theta gradient.
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float logit_r(float xq, float xk, float inv_sigma) {
    const float t = (xk - xq) * inv_sigma;
    return -(t * t);
}

template <int MODE>
__global__ void __launch_bounds__(256) setconv_small_kernel(const float* __restrict__ keys, long key_bs, const float* __restrict__ queries,
                                                            long qry_bs, const float* __restrict__ values, const float* __restrict__ theta,
                                                            float* __restrict__ feat_o, float* __restrict__ dens_o, float* __restrict__ mstat_o,
                                                            const float* __restrict__ feat_i, const float* __restrict__ mstat_i,
                                                            const float* __restrict__ dfeat, const float* __restrict__ ddens,
                                                            float* __restrict__ dtheta, int K, int Q, int C, int ldf, int ldd) {
    extern __shared__ float sm[];
    __shared__ float part[8];
    float* sk = sm;            // [K]
    float* sv = sm + K;        // [K][C]
    const int b = blockIdx.y;
    const float th = __ldg(theta);
    const float sigma = 1e-5f + softplus_f(th);
    const float inv_sigma = 1.f / sigma;       // one division per thread instead of one per (query, key) pair
    for (int i = threadIdx.x; i < K; i += blockDim.x) sk[i] = __ldg(keys + (long)b * key_bs + i);
    for (int i = threadIdx.x; i < K * C; i += blockDim.x) sv[i] = __ldg(values + (long)b * K * C + i);
    __syncthreads();
    // four lanes per query, each sweeping every fourth key: 4x the warps of a thread-per-query layout (this kernel is bound by
    // the latency of its exp chains, not by issue slots), partial maxima / sums joined with two shuffles
    const int q = blockIdx.x * (blockDim.x >> 2) + (threadIdx.x >> 2), kpart = threadIdx.x & 3;
    float contrib = 0.f;
    const bool qok = q < Q;
    {
        const int qq = qok ? q : Q - 1;            // padding lanes shadow the last query (they must take part in the shuffles)
        const float xq = __ldg(queries + (long)b * qry_bs + qq);
        const long oq = (long)b * Q + qq;
        if (MODE == 0) {
            float m = -INFINITY;
#pragma unroll 8
            for (int k = kpart; k < K; k += 4) m = fmaxf(m, logit_r(xq, sk[k], inv_sigma));
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 2));
            float s = 0.f, acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
            for (int k = kpart; k < K; k += 4) {
                const float e = expf(logit_r(xq, sk[k], inv_sigma) - m);
                s += e;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (c < C) acc[c] = fmaf(e, sv[k * C + c], acc[c]);
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], 1);
                acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], 2);
            }
            if (qok && kpart == 0) {
                const float inv = 1.f / s;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (c < C) feat_o[oq * ldf + c] = acc[c] * inv;
                dens_o[oq * ldd] = expf(m) * s;    // sum_k exp(a_k) = exp(m) sum_k exp(a_k - m): one exp per query, not per pair
                mstat_o[oq * 2] = m; mstat_o[oq * 2 + 1] = s;
            }
        } else {
            const float m = __ldg(mstat_i + oq * 2), inv_s = 1.f / __ldg(mstat_i + oq * 2 + 1);
            float df[4], G = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                df[c] = (c < C) ? __ldg(dfeat + oq * ldf + c) : 0.f;
                if (c < C) G = fmaf(df[c], __ldg(feat_i + oq * ldf + c), G);
            }
            float A1 = 0.f, A2 = 0.f, T = 0.f;
#pragma unroll 4
            for (int k = kpart; k < K; k += 4) {
                const float a = logit_r(xq, sk[k], inv_sigma);
                const float e = expf(a - m);
                const float wa = e * inv_s * (a - m);
                A1 += wa;
                A2 = fmaf(e, a, A2);               // sum_k exp(a_k) a_k = exp(m) sum_k exp(a_k - m) a_k
                float g = 0.f;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (c < C) g = fmaf(df[c], sv[k * C + c], g);
                T = fmaf(wa, g, T);
            }
            A1 += __shfl_xor_sync(0xffffffffu, A1, 1); A1 += __shfl_xor_sync(0xffffffffu, A1, 2);
            A2 += __shfl_xor_sync(0xffffffffu, A2, 1); A2 += __shfl_xor_sync(0xffffffffu, A2, 2);
            T += __shfl_xor_sync(0xffffffffu, T, 1); T += __shfl_xor_sync(0xffffffffu, T, 2);
            if (qok && kpart == 0) contrib = T - G * A1 + __ldg(ddens + oq * ldd) * (A2 * expf(m));
        }
    }
    if (MODE == 1) {
        contrib = warp_sum(contrib);
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = contrib;
        __syncthreads();
        if (threadIdx.x == 0) {
            float tot = 0.f;
            for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += part[i];
            atomicAdd(dtheta, tot * (-2.f / sigma) * sigmoid_f(th));
        }
    }
}

// ----------------------------------------------------------------------------------------------------------------
// Few value channels, SORTED keys (context -> induced, C = y_dim <= 4, K <= 1024): one CTA per task sorts the task's
// context positions once (rank counting in shared memory, values carried along) and every query then visits only the keys
// that can carry weight: with d_min the distance to the nearest key, softmax weights below 2^-60 of the largest belong to
// keys with d^2 > d_min^2 + 41.6 sigma^2 -- found by one binary search and two short walks.  The dense version evaluated
// all K keys for every query (12.6 M exp for the 3 MB of data of config 2: 19 + 22 us); here a query touches ~10-20 keys.
// Same formulas as setconv_small_kernel (max logit = logit of the nearest key; sums in key order of the sorted set);
// exact in fp32 in the same sense as the sigma-window of the regular-grid kernels.  mode 0 forward, mode 1 theta gradient.
// ----------------------------------------------------------------------------------------------------------------
constexpr int kSortedMaxK = 1024;

template <int MODE>
__global__ void __launch_bounds__(256) setconv_sorted_kernel(const float* __restrict__ keys, long key_bs, const float* __restrict__ queries,
                                                              long qry_bs, const float* __restrict__ values, const float* __restrict__ theta,
                                                              float* __restrict__ feat_o, float* __restrict__ dens_o, float* __restrict__ mstat_o,
                                                              const float* __restrict__ feat_i, const float* __restrict__ mstat_i,
                                                              const float* __restrict__ dfeat, const float* __restrict__ ddens,
                                                              float* __restrict__ dtheta, int K, int Q, int C, int ldf, int ldd) {
    extern __shared__ float sm[];
    __shared__ float part[8];
    float* sk = sm;                  // [K] sorted positions
    float* sv = sm + K;              // [K][C] values in sorted order
    float* raw = sv + (size_t)K * C; // [K] unsorted positions
    const int b = blockIdx.x;
    const float th = __ldg(theta);
    const float sigma = 1e-5f + softplus_f(th);
    const float inv_sigma = 1.f / sigma;
    for (int i = threadIdx.x; i < K; i += blockDim.x) raw[i] = __ldg(keys + (long)b * key_bs + i);
    __syncthreads();
    for (int i = threadIdx.x; i < K; i += blockDim.x) {
        const float x = raw[i];
        int rank = 0;
        for (int j = 0; j < K; ++j) {
            const float y = raw[j];
            rank += (y < x) || (y == x && j < i);
        }
        sk[rank] = x;
        for (int c = 0; c < C; ++c) sv[rank * C + c] = __ldg(values + ((long)b * K + i) * C + c);
    }
    __syncthreads();
    const float win = kWindowLog * sigma * sigma;
    float contrib = 0.f;
    for (int q = threadIdx.x; q < Q; q += blockDim.x) {
        const float xq = __ldg(queries + (long)b * qry_bs + q);
        const long oq = (long)b * Q + q;
        // lower bound: first sorted key >= xq
        int lo = 0, hi = K;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (sk[mid] < xq) lo = mid + 1; else hi = mid; }
        const int p = lo;
        const int n0 = (p == 0) ? 0 : ((p == K) ? K - 1 : ((xq - sk[p - 1]) <= (sk[p] - xq) ? p - 1 : p));
        const float dn = sk[n0] - xq;
        const float D = sqrtf(fmaf(dn, dn, win)) * 1.0001f + 1e-30f;
        int k0 = n0, k1 = n0;
        if (D == D && D < INFINITY) {
            while (k0 > 0 && sk[k0 - 1] >= xq - D) --k0;
            while (k1 < K - 1 && sk[k1 + 1] <= xq + D) ++k1;
        } else { k0 = 0; k1 = K - 1; }
        if (MODE == 0) {
            float m = logit_r(xq, sk[n0], inv_sigma);
            if (n0 > 0) m = fmaxf(m, logit_r(xq, sk[n0 - 1], inv_sigma));
            if (n0 < K - 1) m = fmaxf(m, logit_r(xq, sk[n0 + 1], inv_sigma));
            float s = 0.f, acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int k = k0; k <= k1; ++k) {
                const float e = expf(logit_r(xq, sk[k], inv_sigma) - m);
                s += e;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (c < C) acc[c] = fmaf(e, sv[k * C + c], acc[c]);
            }
            const float inv = 1.f / s;
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (c < C) feat_o[oq * ldf + c] = acc[c] * inv;
            dens_o[oq * ldd] = expf(m) * s;
            mstat_o[oq * 2] = m; mstat_o[oq * 2 + 1] = s;
        } else {
            const float m = __ldg(mstat_i + oq * 2), inv_s = 1.f / __ldg(mstat_i + oq * 2 + 1);
            float df[4], G = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                df[c] = (c < C) ? __ldg(dfeat + oq * ldf + c) : 0.f;
                if (c < C) G = fmaf(df[c], __ldg(feat_i + oq * ldf + c), G);
            }
            float A1 = 0.f, A2 = 0.f, T = 0.f;
            for (int k = k0; k <= k1; ++k) {
                const float a = logit_r(xq, sk[k], inv_sigma);
                const float e = expf(a - m);
                const float wa = e * inv_s * (a - m);
                A1 += wa;
                A2 = fmaf(e, a, A2);
                float g = 0.f;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (c < C) g = fmaf(df[c], sv[k * C + c], g);
                T = fmaf(wa, g, T);
            }
            contrib += T - G * A1 + __ldg(ddens + oq * ldd) * (A2 * expf(m));
        }
    }
    if (MODE == 1) {
        contrib = warp_sum(contrib);
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = contrib;
        __syncthreads();
        if (threadIdx.x == 0) {
            float tot = 0.f;
            for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += part[i];
            atomicAdd(dtheta, tot * (-2.f / sigma) * sigmoid_f(th));
        }
    }
}

static bool sorted_ok(int K) { return K <= kSortedMaxK; }

// implemented in setconv_tile.cu: shared-memory staged fast path; NPF_ENOTSUP if the shape is not covered
int setconv_tile_fwd(const float* keys, long key_bs, const float* queries, long qry_bs, const float* values,
                     const float* theta, float* feat, float* dens, float* mstat, int B, int K, int Q, int C,
                     cudaStream_t st);
int setconv_tile_bwd(const float* keys, long key_bs, const float* queries, long qry_bs, const float* values,
                     const float* theta, const float* feat, const float* mstat, const float* dfeat,
                     const float* ddens, float* dvalues, float* dtheta, int B, int K, int Q, int C, cudaStream_t st);

}  // namespace npf

using namespace npf;

extern "C" int npf_setconv_fwd(const float* keys, long key_bs, const float* queries, long qry_bs,
                               const float* values, const float* theta, float* feat, float* dens, float* mstat,
                               int B, int K, int Q, int Cin, int keys_regular, int ldf, int ldd, npf_stream_t stream) {
    NPF_REQUIRE(keys && queries && values && theta && feat && dens && mstat, "npf_setconv_fwd: null pointer");
    const bool small = Cin <= 4 && !keys_regular && (size_t)K * (1 + Cin) * sizeof(float) <= 40 * 1024;
    NPF_REQUIRE(ldf >= Cin && ldd >= 1, "npf_setconv_fwd: feat / dens strides too small");
    NPF_REQUIRE((ldf == Cin && ldd == 1) || small, "npf_setconv_fwd: strided feat / dens only on the few-channel path (Cin <= 4, irregular keys)");
    NPF_REQUIRE(B >= 0 && K >= 1 && Q >= 0 && Cin >= 1, "npf_setconv_fwd: bad shape B=%d K=%d Q=%d C=%d", B, K, Q, Cin);
    NPF_REQUIRE(Cin <= 32 * kMaxChunks, "npf_setconv_fwd: at most %d channels", 32 * kMaxChunks);
    NPF_REQUIRE(B <= 65535, "npf_setconv_fwd: batch > 65535");
    if (B == 0 || Q == 0) return NPF_OK;
    cudaStream_t st = as_stream(stream);
    if (keys_regular) {
        int rc = setconv_tile_fwd(keys, key_bs, queries, qry_bs, values, theta, feat, dens, mstat, B, K, Q, Cin, st);
        if (rc != NPF_ENOTSUP) return rc;
    }
    if (small && sorted_ok(K)) {
        setconv_sorted_kernel<0><<<(unsigned)B, 256, (size_t)K * (2 + Cin) * sizeof(float), st>>>(
            keys, key_bs, queries, qry_bs, values, theta, feat, dens, mstat, nullptr, nullptr, nullptr, nullptr, nullptr, K, Q, Cin, ldf, ldd);
        count_launch();
        return check_launch("setconv_sorted_kernel<fwd>");
    }
    if (small) {
        const int nblk = (int)cdiv(Q, 64), thr = 256;                                  // 64 queries x 4 key lanes per block
        dim3 grid((unsigned)nblk, (unsigned)B);
        setconv_small_kernel<0><<<grid, thr, (size_t)K * (1 + Cin) * sizeof(float), st>>>(
            keys, key_bs, queries, qry_bs, values, theta, feat, dens, mstat, nullptr, nullptr, nullptr, nullptr, nullptr, K, Q, Cin, ldf, ldd);
        count_launch();
        return check_launch("setconv_small_kernel<fwd>");
    }
    dim3 grid((unsigned)cdiv(Q, 8), (unsigned)B);
    setconv_fwd_kernel<<<grid, 256, 0, st>>>(keys, key_bs, queries, qry_bs, values, theta, feat, dens, mstat, K, Q, Cin,
                                             keys_regular);
    count_launch();
    return check_launch("setconv_fwd_kernel");
}

extern "C" int npf_setconv_bwd(const float* keys, long key_bs, const float* queries, long qry_bs,
                               const float* values, const float* theta, const float* feat, const float* dens,
                               const float* mstat, const float* dfeat, const float* ddens, float* dvalues,
                               float* dtheta, int B, int K, int Q, int Cin, int keys_regular, int ldf, int ldd, npf_stream_t stream) {
    (void)dens;
    const bool small = Cin <= 4 && !keys_regular && (size_t)K * (1 + Cin) * sizeof(float) <= 40 * 1024;
    NPF_REQUIRE(ldf >= Cin && ldd >= 1, "npf_setconv_bwd: feat / dens strides too small");
    NPF_REQUIRE((ldf == Cin && ldd == 1) || (small && !dvalues), "npf_setconv_bwd: strided feat / dens only on the few-channel path without dvalues");
    NPF_REQUIRE(keys && queries && values && theta && feat && mstat && dfeat && ddens && dtheta,
                "npf_setconv_bwd: null pointer");
    NPF_REQUIRE(B >= 0 && K >= 1 && Q >= 0 && Cin >= 1 && Cin <= 32 * kMaxChunks, "npf_setconv_bwd: bad shape");
    NPF_REQUIRE(B <= 65535, "npf_setconv_bwd: batch > 65535");
    if (B == 0) return NPF_OK;
    cudaStream_t st = as_stream(stream);
    if (Q == 0) {
        if (dvalues) cudaMemsetAsync(dvalues, 0, sizeof(float) * (size_t)B * K * Cin, st);
        return NPF_OK;
    }
    if (keys_regular) {
        int rc = setconv_tile_bwd(keys, key_bs, queries, qry_bs, values, theta, feat, mstat, dfeat, ddens, dvalues,
                                  dtheta, B, K, Q, Cin, st);
        if (rc != NPF_ENOTSUP) return rc;
    }
    if (small && sorted_ok(K)) {
        setconv_sorted_kernel<1><<<(unsigned)B, 256, (size_t)K * (2 + Cin) * sizeof(float), st>>>(
            keys, key_bs, queries, qry_bs, values, theta, nullptr, nullptr, nullptr, feat, mstat, dfeat, ddens, dtheta, K, Q, Cin, ldf, ldd);
        count_launch();
        int rc = check_launch("setconv_sorted_kernel<dtheta>");
        if (rc != NPF_OK) return rc;
    } else if (small) {
        const int nblk = (int)cdiv(Q, 64), thr = 256;
        dim3 grid((unsigned)nblk, (unsigned)B);
        setconv_small_kernel<1><<<grid, thr, (size_t)K * (1 + Cin) * sizeof(float), st>>>(
            keys, key_bs, queries, qry_bs, values, theta, nullptr, nullptr, nullptr, feat, mstat, dfeat, ddens, dtheta, K, Q, Cin, ldf, ldd);
        count_launch();
        int rc = check_launch("setconv_small_kernel<dtheta>");
        if (rc != NPF_OK) return rc;
    } else {
        dim3 grid((unsigned)cdiv(Q, 8), (unsigned)B);
        setconv_bwd_theta_kernel<<<grid, 256, 0, st>>>(keys, key_bs, queries, qry_bs, values, theta, feat, mstat, dfeat,
                                                       ddens, dtheta, K, Q, Cin, keys_regular);
        count_launch();
        int rc = check_launch("setconv_bwd_theta_kernel");
        if (rc != NPF_OK) return rc;
    }
    if (dvalues) {
        dim3 grid((unsigned)cdiv(K, 8), (unsigned)B);
        setconv_bwd_values_kernel<<<grid, 256, 0, st>>>(keys, key_bs, queries, qry_bs, theta, mstat, dfeat, dvalues, K, Q,
                                                        Cin);
        count_launch();
        return check_launch("setconv_bwd_values_kernel");
    }
    return NPF_OK;
}
