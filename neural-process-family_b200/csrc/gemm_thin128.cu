// Thin linear layers whose WIDE side is exactly 128 (the r_dim / hidden width of every model in the family): the
// first layer of the x / xy encoders and SetConv's resizer (K <= 8 -> 128) and the predictive head (128 -> 2 y_dim <= 8),
// forward and whole backward, each as ONE streaming pass with a warp per row:
//
//   thin_in128_fwd  <R> : Y[m, :]  = act( sum_r x[m, r] W[:, r] + b )                                   writes [M,128]
//   thin_in128_bwd  <R> : dX[m, r] = dY[m, :] . W[:, r];  dW[:, r] += dY^T x;  db += colsum(dY)         reads  [M,128] once
//   thin_out128_fwd <J> : Y[m, j]  = act( act_in(x[m, :]) . W[j, :] + b[j] )                            reads  [M,128]
//   thin_out128_bwd <J> : dX[m, :] = (sum_j dY[m, j] W[j, :]) (.) (x > 0);  dW[j, :] += dY[m, j] act_in(x[m, :]);  db[j] += sum_m dY[m, j]
//                                                                                                        reads + writes [M,128] once
// A lane owns 4 consecutive columns of the 128-wide side (one LDG.128 / STG.128 per row: 512 contiguous bytes per warp
// instruction), the narrow side lives in registers (compile-time R / J), rows are processed kRows at a time so that kRows
// independent 16-byte accesses per thread are in flight, and the CTA's column sums go through shared memory before ONE
// global atomic per entry.  Grids are persistent (a few CTAs per SM): no per-row index arithmetic, no divisions.
#include "common.cuh"
#include "gemm_thin.cuh"

namespace npf {

constexpr int kT128Threads = 256;
constexpr int kT128Rows = 4;            // rows in flight per warp (8 rows per pass measured slower: 160+ registers, 12 % occupancy)

__device__ __forceinline__ float4 relu4(float4 v) { return make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f)); }
__device__ __forceinline__ float dot4(float4 a, float4 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w))); }
__device__ __forceinline__ void fma4(float4& acc, float s, float4 v) {
    acc.x = fmaf(s, v.x, acc.x); acc.y = fmaf(s, v.y, acc.y); acc.z = fmaf(s, v.z, acc.z); acc.w = fmaf(s, v.w, acc.w);
}

struct Thin128Params {
    const float* X; long ldx;        // narrow operand for *_in (x [M,R]) / wide operand for *_out (x [M,128])
    const float* W; long ldw;        // in: W [128, R] (row stride ldw);  out: W [J, 128]
    const float* b;                  // fwd bias
    const float* dY; long lddy;      // bwd: in: [M,128];  out: [M,J]
    float* Y; long ldy;              // fwd output / bwd dX
    float* dW; long lddw; float* db; // bwd accumulators (+=)
    long M;
    int relu_in, relu_out, use_mask;
};

// ---------------------------------------------------------------------------------------------- K = R <= 8 -> 128
template <int R>
__global__ void __launch_bounds__(kT128Threads) thin_in128_fwd_kernel(Thin128Params p) {
    const int lane = threadIdx.x & 31;
    const long warp = ((long)blockIdx.x * kT128Threads + threadIdx.x) >> 5, nwarps = ((long)gridDim.x * kT128Threads) >> 5;
    float4 w[R];
#pragma unroll
    for (int r = 0; r < R; ++r)
        w[r] = make_float4(__ldg(p.W + (long)(4 * lane + 0) * p.ldw + r), __ldg(p.W + (long)(4 * lane + 1) * p.ldw + r),
                           __ldg(p.W + (long)(4 * lane + 2) * p.ldw + r), __ldg(p.W + (long)(4 * lane + 3) * p.ldw + r));
    const float4 bias = p.b ? __ldg(reinterpret_cast<const float4*>(p.b) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
    pdl_trigger();
    pdl_wait();          // weights / bias above are parameters; x is a preceding kernel's output
    for (long m0 = warp * kT128Rows; m0 < p.M; m0 += nwarps * kT128Rows) {
        float x[kT128Rows][R];
#pragma unroll
        for (int u = 0; u < kT128Rows; ++u)
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float v = (m0 + u < p.M) ? __ldg(p.X + (m0 + u) * p.ldx + r) : 0.f;       // warp-uniform address: one sector, broadcast
                x[u][r] = p.relu_in ? fmaxf(v, 0.f) : v;
            }
#pragma unroll
        for (int u = 0; u < kT128Rows; ++u) {
            if (m0 + u >= p.M) break;
            float4 y = bias;
#pragma unroll
            for (int r = 0; r < R; ++r) fma4(y, x[u][r], w[r]);
            if (p.relu_out) y = relu4(y);
            *reinterpret_cast<float4*>(p.Y + (m0 + u) * p.ldy + 4 * lane) = y;
        }
    }
}

template <int R>
__global__ void __launch_bounds__(kT128Threads) thin_in128_bwd_kernel(Thin128Params p) {
    __shared__ float s_acc[(R + 1) * 128];
    for (int i = threadIdx.x; i < (R + 1) * 128; i += kT128Threads) s_acc[i] = 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long warp = ((long)blockIdx.x * kT128Threads + threadIdx.x) >> 5, nwarps = ((long)gridDim.x * kT128Threads) >> 5;
    float4 w[R], aw[R], ab = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        aw[r] = make_float4(0.f, 0.f, 0.f, 0.f);
        w[r] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.Y)
            w[r] = make_float4(__ldg(p.W + (long)(4 * lane + 0) * p.ldw + r), __ldg(p.W + (long)(4 * lane + 1) * p.ldw + r),
                               __ldg(p.W + (long)(4 * lane + 2) * p.ldw + r), __ldg(p.W + (long)(4 * lane + 3) * p.ldw + r));
    }
    pdl_trigger();
    pdl_wait();
    for (long m0 = warp * kT128Rows; m0 < p.M; m0 += nwarps * kT128Rows) {
        float4 dy[kT128Rows];
        float x[kT128Rows][R];
#pragma unroll
        for (int u = 0; u < kT128Rows; ++u) {
            const bool ok = m0 + u < p.M;
            dy[u] = ok ? __ldg(reinterpret_cast<const float4*>(p.dY + (m0 + u) * p.lddy) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float v = ok ? __ldg(p.X + (m0 + u) * p.ldx + r) : 0.f;
                x[u][r] = p.relu_in ? fmaxf(v, 0.f) : v;
            }
        }
#pragma unroll
        for (int u = 0; u < kT128Rows; ++u) {
            ab.x += dy[u].x; ab.y += dy[u].y; ab.z += dy[u].z; ab.w += dy[u].w;
#pragma unroll
            for (int r = 0; r < R; ++r) fma4(aw[r], x[u][r], dy[u]);
        }
        if (p.Y) {
            float dx[kT128Rows][R];
#pragma unroll
            for (int u = 0; u < kT128Rows; ++u)
#pragma unroll
                for (int r = 0; r < R; ++r) dx[u][r] = warp_sum(dot4(dy[u], w[r]));
#pragma unroll
            for (int u = 0; u < kT128Rows; ++u)
#pragma unroll
                for (int r = 0; r < R; ++r)
                    if (lane == r && m0 + u < p.M) p.Y[(m0 + u) * p.ldy + r] = dx[u][r];
        }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
        float* d = s_acc + r * 128 + 4 * lane;
        atomicAdd(d + 0, aw[r].x); atomicAdd(d + 1, aw[r].y); atomicAdd(d + 2, aw[r].z); atomicAdd(d + 3, aw[r].w);
    }
    {
        float* d = s_acc + R * 128 + 4 * lane;
        atomicAdd(d + 0, ab.x); atomicAdd(d + 1, ab.y); atomicAdd(d + 2, ab.z); atomicAdd(d + 3, ab.w);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < (R + 1) * 128; i += kT128Threads) {
        const int r = i >> 7, c = i & 127;
        if (r < R) atomicAdd(p.dW + (long)c * p.lddw + r, s_acc[i]);
        else if (p.db) atomicAdd(p.db + c, s_acc[i]);
    }
}

// ---------------------------------------------------------------------------------------------- 128 -> N = J <= 8
template <int J>
__global__ void __launch_bounds__(kT128Threads) thin_out128_fwd_kernel(Thin128Params p) {
    const int lane = threadIdx.x & 31;
    const long warp = ((long)blockIdx.x * kT128Threads + threadIdx.x) >> 5, nwarps = ((long)gridDim.x * kT128Threads) >> 5;
    float4 w[J];
#pragma unroll
    for (int j = 0; j < J; ++j) w[j] = __ldg(reinterpret_cast<const float4*>(p.W + (long)j * p.ldw) + lane);
    const float bias = (p.b && lane < J) ? __ldg(p.b + lane) : 0.f;
    pdl_trigger();
    pdl_wait();
    for (long m0 = warp * kT128Rows; m0 < p.M; m0 += nwarps * kT128Rows) {
        float4 x[kT128Rows];
#pragma unroll
        for (int u = 0; u < kT128Rows; ++u) {
            x[u] = (m0 + u < p.M) ? __ldg(reinterpret_cast<const float4*>(p.X + (m0 + u) * p.ldx) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.relu_in) x[u] = relu4(x[u]);
        }
#pragma unroll
        for (int u = 0; u < kT128Rows; ++u) {
            float mine = 0.f;
#pragma unroll
            for (int j = 0; j < J; ++j) {
                const float s = warp_sum(dot4(x[u], w[j]));
                if (lane == j) mine = s;
            }
            if (lane < J && m0 + u < p.M) {
                float y = mine + bias;
                if (p.relu_out) y = fmaxf(y, 0.f);
                p.Y[(m0 + u) * p.ldy + lane] = y;
            }
        }
    }
}

template <int J>
__global__ void __launch_bounds__(kT128Threads) thin_out128_bwd_kernel(Thin128Params p) {
    __shared__ float s_acc[J * 128 + 8];
    for (int i = threadIdx.x; i < J * 128 + 8; i += kT128Threads) s_acc[i] = 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long warp = ((long)blockIdx.x * kT128Threads + threadIdx.x) >> 5, nwarps = ((long)gridDim.x * kT128Threads) >> 5;
    float4 w[J], aw[J];
    float ab[J];
#pragma unroll
    for (int j = 0; j < J; ++j) {
        w[j] = __ldg(reinterpret_cast<const float4*>(p.W + (long)j * p.ldw) + lane);
        aw[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        ab[j] = 0.f;
    }
    pdl_trigger();
    pdl_wait();
    for (long m0 = warp * kT128Rows; m0 < p.M; m0 += nwarps * kT128Rows) {
        float4 x[kT128Rows];
        float dy[kT128Rows][J];
#pragma unroll
        for (int u = 0; u < kT128Rows; ++u) {
            const bool ok = m0 + u < p.M;
            x[u] = ok ? __ldg(reinterpret_cast<const float4*>(p.X + (m0 + u) * p.ldx) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int j = 0; j < J; ++j) dy[u][j] = ok ? __ldg(p.dY + (m0 + u) * p.lddy + j) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < kT128Rows; ++u) {
            const float4 xa = p.relu_in ? relu4(x[u]) : x[u];
            float4 dx = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int j = 0; j < J; ++j) {
                fma4(dx, dy[u][j], w[j]);
                fma4(aw[j], dy[u][j], xa);
                ab[j] += dy[u][j];
            }
            if (p.use_mask) {
                dx.x = x[u].x > 0.f ? dx.x : 0.f; dx.y = x[u].y > 0.f ? dx.y : 0.f;
                dx.z = x[u].z > 0.f ? dx.z : 0.f; dx.w = x[u].w > 0.f ? dx.w : 0.f;
            }
            if (p.Y && m0 + u < p.M) *reinterpret_cast<float4*>(p.Y + (m0 + u) * p.ldy + 4 * lane) = dx;
        }
    }
#pragma unroll
    for (int j = 0; j < J; ++j) {
        float* d = s_acc + j * 128 + 4 * lane;
        atomicAdd(d + 0, aw[j].x); atomicAdd(d + 1, aw[j].y); atomicAdd(d + 2, aw[j].z); atomicAdd(d + 3, aw[j].w);
        if (lane == 0) atomicAdd(s_acc + J * 128 + j, ab[j]);        // every lane holds the same row sums
    }
    __syncthreads();
    for (int i = threadIdx.x; i < J * 128; i += kT128Threads) atomicAdd(p.dW + (long)(i >> 7) * p.lddw + (i & 127), s_acc[i]);
    if (p.db && threadIdx.x < J) atomicAdd(p.db + threadIdx.x, s_acc[J * 128 + threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------- launchers
static inline bool a16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; }
static inline unsigned t128_grid(long M, int per_sm) {
    long g = cdiv(M, (long)(kT128Threads / 32) * kT128Rows);
    if (g > (long)per_sm * kNumSMs) g = (long)per_sm * kNumSMs;
    return (unsigned)(g < 1 ? 1 : g);
}
#define NPF_T128_SWITCH(n, KERNEL, grid)                                                  \
    switch (n) {                                                                            \
        case 1: launch_pdl(KERNEL<1>, dim3(grid), dim3(kT128Threads), 0, st, p); break;                         \
        case 2: launch_pdl(KERNEL<2>, dim3(grid), dim3(kT128Threads), 0, st, p); break;                         \
        case 3: launch_pdl(KERNEL<3>, dim3(grid), dim3(kT128Threads), 0, st, p); break;                         \
        case 4: launch_pdl(KERNEL<4>, dim3(grid), dim3(kT128Threads), 0, st, p); break;                         \
        case 5: launch_pdl(KERNEL<5>, dim3(grid), dim3(kT128Threads), 0, st, p); break;                         \
        case 6: launch_pdl(KERNEL<6>, dim3(grid), dim3(kT128Threads), 0, st, p); break;                         \
        case 7: launch_pdl(KERNEL<7>, dim3(grid), dim3(kT128Threads), 0, st, p); break;                         \
        case 8: launch_pdl(KERNEL<8>, dim3(grid), dim3(kT128Threads), 0, st, p); break;                         \
        default: return NPF_ENOTSUP;                                                        \
    }

// Y[M,128] = act(act_in(X[M,R]) W[128,R]^T + b)
int thin128_in_fwd(const float* X, long ldx, const float* W, long ldw, const float* b, float* Y, long ldy, long M, int R, int relu_in,
                   int relu_out, cudaStream_t st) {
    if (R < 1 || R > 8 || (ldy & 3) || !a16(Y) || (b && !a16(b))) return NPF_ENOTSUP;
    Thin128Params p{};
    p.X = X; p.ldx = ldx; p.W = W; p.ldw = ldw; p.b = b; p.Y = Y; p.ldy = ldy; p.M = M; p.relu_in = relu_in; p.relu_out = relu_out;
    const unsigned grid = t128_grid(M, 8);
    NPF_T128_SWITCH(R, thin_in128_fwd_kernel, grid)
    count_launch();
    return check_launch("thin_in128_fwd_kernel");
}

// dX[M,R] = dY[M,128] W[128,R] (dX may be null); dW[128,R] += dY^T act_in(X); db[128] += colsum(dY) (db may be null)
int thin128_in_bwd(const float* dY, long lddy, const float* X, long ldx, const float* W, long ldw, float* dX, long lddx, float* dW, long lddw,
                   float* db, long M, int R, int relu_in, cudaStream_t st) {
    if (R < 1 || R > 8 || (lddy & 3) || !a16(dY)) return NPF_ENOTSUP;
    Thin128Params p{};
    p.dY = dY; p.lddy = lddy; p.X = X; p.ldx = ldx; p.W = W; p.ldw = ldw; p.Y = dX; p.ldy = lddx; p.dW = dW; p.lddw = lddw; p.db = db;
    p.M = M; p.relu_in = relu_in;
    const unsigned grid = t128_grid(M, 2);
    NPF_T128_SWITCH(R, thin_in128_bwd_kernel, grid)
    count_launch();
    return check_launch("thin_in128_bwd_kernel");
}

// Y[M,J] = act(act_in(X[M,128]) W[J,128]^T + b)
int thin128_out_fwd(const float* X, long ldx, const float* W, long ldw, const float* b, float* Y, long ldy, long M, int J, int relu_in,
                    int relu_out, cudaStream_t st) {
    if (J < 1 || J > 8 || (ldx & 3) || !a16(X) || (ldw & 3) || !a16(W)) return NPF_ENOTSUP;
    Thin128Params p{};
    p.X = X; p.ldx = ldx; p.W = W; p.ldw = ldw; p.b = b; p.Y = Y; p.ldy = ldy; p.M = M; p.relu_in = relu_in; p.relu_out = relu_out;
    const unsigned grid = t128_grid(M, 8);
    NPF_T128_SWITCH(J, thin_out128_fwd_kernel, grid)
    count_launch();
    return check_launch("thin_out128_fwd_kernel");
}

// dX[M,128] = (dY[M,J] W[J,128]) (.) (X > 0 if use_mask) (dX may be null); dW[J,128] += dY^T act_in(X); db[J] += colsum(dY)
int thin128_out_bwd(const float* dY, long lddy, const float* X, long ldx, const float* W, long ldw, float* dX, long lddx, float* dW, long lddw,
                    float* db, long M, int J, int relu_in, int use_mask, cudaStream_t st) {
    if (J < 1 || J > 8 || (ldx & 3) || !a16(X) || (ldw & 3) || !a16(W) || (dX && ((lddx & 3) || !a16(dX)))) return NPF_ENOTSUP;
    Thin128Params p{};
    p.dY = dY; p.lddy = lddy; p.X = X; p.ldx = ldx; p.W = W; p.ldw = ldw; p.Y = dX; p.ldy = lddx; p.dW = dW; p.lddw = lddw; p.db = db;
    p.M = M; p.relu_in = relu_in; p.use_mask = use_mask;
    const unsigned grid = t128_grid(M, 2);
    NPF_T128_SWITCH(J, thin_out128_bwd_kernel, grid)
    count_launch();
    return check_launch("thin_out128_bwd_kernel");
}

}  // namespace npf
