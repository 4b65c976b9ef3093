// Channel-last depthwise convolution (1-D and 2-D) for the ResConvBlock stack
// (upstream npf/architectures/cnn.py:204-215 conv2_depthwise / conv1.depthwise; npf/utils/helpers.py:354-403).
//
//   Y[b,h,w,c] = sum_{i,j} Wt[c,i,j] * act(X)[b,h+i-kh/2,w+j-kw/2,c] + bias[c] (+ res[b,h,w,c])
//   act(x) = relu(scale[c]*x + shift[c])  (NPF_RELU_IN; scale/shift = folded BatchNorm affine, optional)
//
// One CTA stages a (TH+kh-1) x (TW+KW-1) x CT halo tile of act(X) and the CT channels' filters in shared memory;
// a thread owns 4 channels x 8 consecutive outputs along w and slides over the input row in registers, so each
// staged float4 is read once per filter row instead of once per tap.  The same kernel with flipped filters and a
// relu-mask epilogue is the data gradient; the filter gradient kernel uses the mirrored register scheme.
// KW is a compile-time (padded) filter width in {9, 11, 19}; narrower filters are centred and zero-padded.
#include "common.cuh"

namespace npf {

struct DwParams {
    const float* X;      // input (fwd: activations; bwd-data: dY)
    const float* Wt;     // [C, kh, kw]
    const float* bias;   // [C] or null
    const float* res;    // residual added to the output, or null
    float* Y;
    const float* Xorig;  // bwd-data only: forward input, for the relu/affine mask
    const float* scale;  // per-channel pre-activation affine (null = identity)
    const float* shift;
    float* dscale;       // bwd-data only (optional): gradients of the affine
    float* dshift;
    int H, Wd, C, kh, kw;
    int TH, TW, CT;
    int tiles_w;
    int relu_in;  // apply act() while staging X
    int flip;     // use spatially flipped filters (data gradient)
    int mask;     // epilogue: multiply by act'(Xorig)
    int accum;
};

// 4 channels x one tap: two packed fp32x2 FMAs (FFMA2, sm_100): the depthwise kernels are bound by the number of FMA instructions
// they issue (121 taps x 16 float4 per thread in the 2-D case), and a float4's (x, y) / (z, w) halves are aligned register pairs
__device__ __forceinline__ float4 f4_fma(const float4 a, const float4 b, const float4 c) {
    const float2 lo = __ffma2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y), make_float2(c.x, c.y));
    const float2 hi = __ffma2_rn(make_float2(a.z, a.w), make_float2(b.z, b.w), make_float2(c.z, c.w));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

template <int KW>
__global__ void __launch_bounds__(256) dwconv_kernel(DwParams p) {
    extern __shared__ __align__(16) float smem[];
    const int CT = p.CT, CQ = CT >> 2;
    const int rows = p.TH + p.kh - 1, cols = p.TW + KW - 1;
    float4* Xs = reinterpret_cast<float4*>(smem);                 // [rows][cols][CQ]
    float4* Ws = Xs + (size_t)rows * cols * CQ;                   // [kh][KW][CQ]

    const int tile = blockIdx.x;
    const int h0 = (tile / p.tiles_w) * p.TH, w0 = (tile % p.tiles_w) * p.TW;
    const int c0 = blockIdx.y * CT;
    const int b = blockIdx.z;
    const int ph = p.kh / 2, pw = KW / 2, joff = (KW - p.kw) / 2;
    const int nthr = blockDim.x * blockDim.y * blockDim.z;
    const int tid = threadIdx.x + blockDim.x * (threadIdx.y + blockDim.y * threadIdx.z);
    const long img = (long)b * p.H * p.Wd;

    // stage filters (centred in the padded width, optionally flipped)
    for (int idx = tid; idx < p.kh * KW * CT; idx += nthr) {
        const int c = idx % CT, j = (idx / CT) % KW, i = idx / (CT * KW);
        float v = 0.f;
        const int jr = j - joff;
        if (jr >= 0 && jr < p.kw && c0 + c < p.C) {
            const int ii = p.flip ? p.kh - 1 - i : i, jj = p.flip ? p.kw - 1 - jr : jr;
            v = __ldg(p.Wt + ((long)(c0 + c) * p.kh + ii) * p.kw + jj);
        }
        reinterpret_cast<float*>(Ws)[((size_t)i * KW + j) * CT + c] = v;
    }
    // stage the halo tile of act(X); zero outside the image (padding applies to the activated signal)
    for (int idx = tid; idx < rows * cols * CQ; idx += nthr) {
        const int q = idx % CQ, col = (idx / CQ) % cols, r = idx / (CQ * cols);
        const int gh = h0 + r - ph, gw = w0 + col - pw, c = c0 + 4 * q;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gh >= 0 && gh < p.H && gw >= 0 && gw < p.Wd && c < p.C) {
            v = __ldg(reinterpret_cast<const float4*>(p.X + (img + (long)gh * p.Wd + gw) * p.C + c));
            if (p.relu_in) {
                if (p.scale) {
                    const float4 s = __ldg(reinterpret_cast<const float4*>(p.scale + c));
                    const float4 t = __ldg(reinterpret_cast<const float4*>(p.shift + c));
                    v = make_float4(fmaf(s.x, v.x, t.x), fmaf(s.y, v.y, t.y), fmaf(s.z, v.z, t.z), fmaf(s.w, v.w, t.w));
                }
                v = make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
            }
        }
        Xs[idx] = v;
    }
    __syncthreads();

    const int q = threadIdx.x, s = threadIdx.y, r = threadIdx.z;
    float4 acc[8];
#pragma unroll
    for (int pp = 0; pp < 8; ++pp) acc[pp] = make_float4(0.f, 0.f, 0.f, 0.f);

    for (int i = 0; i < p.kh; ++i) {
        float4 wr[KW];
#pragma unroll
        for (int j = 0; j < KW; ++j) wr[j] = Ws[((size_t)i * KW + j) * CQ + q];
        const float4* xrow = Xs + ((size_t)(r + i) * cols + s * 8) * CQ + q;
#pragma unroll
        for (int xc = 0; xc < KW + 7; ++xc) {
            const float4 xv = xrow[(size_t)xc * CQ];
#pragma unroll
            for (int pp = 0; pp < 8; ++pp) {
                const int j = xc - pp;
                if (j >= 0 && j < KW) acc[pp] = f4_fma(wr[j], xv, acc[pp]);
            }
        }
    }

    const int c = c0 + 4 * q;
    const int gh = h0 + r;
    float4 ds = make_float4(0.f, 0.f, 0.f, 0.f), dt = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < p.C && gh < p.H) {
        float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) bv = __ldg(reinterpret_cast<const float4*>(p.bias + c));
        float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.mask && p.scale) {
            sc = __ldg(reinterpret_cast<const float4*>(p.scale + c));
            sh = __ldg(reinterpret_cast<const float4*>(p.shift + c));
        }
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) {
            const int gw = w0 + s * 8 + pp;
            if (gw >= p.Wd) continue;
            const long off = (img + (long)gh * p.Wd + gw) * p.C + c;
            float4 v = make_float4(acc[pp].x + bv.x, acc[pp].y + bv.y, acc[pp].z + bv.z, acc[pp].w + bv.w);
            if (p.mask) {
                const float4 x = __ldg(reinterpret_cast<const float4*>(p.Xorig + off));
                const float4 pre = make_float4(fmaf(sc.x, x.x, sh.x), fmaf(sc.y, x.y, sh.y), fmaf(sc.z, x.z, sh.z), fmaf(sc.w, x.w, sh.w));
                v.x = pre.x > 0.f ? v.x : 0.f; v.y = pre.y > 0.f ? v.y : 0.f;
                v.z = pre.z > 0.f ? v.z : 0.f; v.w = pre.w > 0.f ? v.w : 0.f;
                if (p.dscale) {
                    dt.x += v.x; dt.y += v.y; dt.z += v.z; dt.w += v.w;
                    ds = f4_fma(v, x, ds);
                }
                v.x *= sc.x; v.y *= sc.y; v.z *= sc.z; v.w *= sc.w;
            }
            if (p.res) {
                const float4 rv = __ldg(reinterpret_cast<const float4*>(p.res + off));
                v.x += rv.x; v.y += rv.y; v.z += rv.z; v.w += rv.w;
            }
            float4* out = reinterpret_cast<float4*>(p.Y + off);
            if (p.accum) {
                const float4 o = *out;
                v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
            }
            *out = v;
        }
    }
    if (p.mask && p.dscale) {
        // block-reduce the affine gradients over (s, r) through shared memory (reuse the tile space), then atomics
        __syncthreads();
        float* red = smem;  // [2][CT]
        for (int idx = tid; idx < 2 * CT; idx += nthr) red[idx] = 0.f;
        __syncthreads();
        if (c < p.C) {
            atomicAdd(red + 4 * q + 0, ds.x); atomicAdd(red + 4 * q + 1, ds.y);
            atomicAdd(red + 4 * q + 2, ds.z); atomicAdd(red + 4 * q + 3, ds.w);
            atomicAdd(red + CT + 4 * q + 0, dt.x); atomicAdd(red + CT + 4 * q + 1, dt.y);
            atomicAdd(red + CT + 4 * q + 2, dt.z); atomicAdd(red + CT + 4 * q + 3, dt.w);
        }
        __syncthreads();
        for (int idx = tid; idx < CT; idx += nthr) {
            if (c0 + idx < p.C) {
                atomicAdd(p.dscale + c0 + idx, red[idx]);
                atomicAdd(p.dshift + c0 + idx, red[CT + idx]);
            }
        }
    }
}

// Filter gradient: dWt[c,i,j] += sum_{b,h,w} dY[b,h,w,c] * act(X)[b,h+i-kh/2,w+j-kw/2,c]
// block = (CT/4 channel quads, kh filter rows, NS strip lanes)
template <int KW>
__global__ void __launch_bounds__(256) dwconv_wgrad_kernel(DwParams p, const float* __restrict__ dY, float* __restrict__ dWt) {
    extern __shared__ __align__(16) float smem[];
    const int CT = p.CT, CQ = CT >> 2;
    const int rows = p.TH + p.kh - 1, cols = p.TW + KW - 1;
    float4* Xs = reinterpret_cast<float4*>(smem);                  // [rows][cols][CQ]
    float4* Gs = Xs + (size_t)rows * cols * CQ;                    // [TH][TW][CQ]
    float* dWs = reinterpret_cast<float*>(Gs + (size_t)p.TH * p.TW * CQ);  // [kh][KW][CT]

    const int tile = blockIdx.x;
    const int h0 = (tile / p.tiles_w) * p.TH, w0 = (tile % p.tiles_w) * p.TW;
    const int c0 = blockIdx.y * CT;
    const int b = blockIdx.z;
    const int ph = p.kh / 2, pw = KW / 2, joff = (KW - p.kw) / 2;
    const int nthr = blockDim.x * blockDim.y * blockDim.z;
    const int tid = threadIdx.x + blockDim.x * (threadIdx.y + blockDim.y * threadIdx.z);
    const long img = (long)b * p.H * p.Wd;

    for (int idx = tid; idx < p.kh * KW * CT; idx += nthr) dWs[idx] = 0.f;
    for (int idx = tid; idx < rows * cols * CQ; idx += nthr) {
        const int q = idx % CQ, col = (idx / CQ) % cols, r = idx / (CQ * cols);
        const int gh = h0 + r - ph, gw = w0 + col - pw, c = c0 + 4 * q;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gh >= 0 && gh < p.H && gw >= 0 && gw < p.Wd && c < p.C) {
            v = __ldg(reinterpret_cast<const float4*>(p.X + (img + (long)gh * p.Wd + gw) * p.C + c));
            if (p.relu_in) {
                if (p.scale) {
                    const float4 s = __ldg(reinterpret_cast<const float4*>(p.scale + c));
                    const float4 t = __ldg(reinterpret_cast<const float4*>(p.shift + c));
                    v = make_float4(fmaf(s.x, v.x, t.x), fmaf(s.y, v.y, t.y), fmaf(s.z, v.z, t.z), fmaf(s.w, v.w, t.w));
                }
                v = make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
            }
        }
        Xs[idx] = v;
    }
    for (int idx = tid; idx < p.TH * p.TW * CQ; idx += nthr) {
        const int q = idx % CQ, col = (idx / CQ) % p.TW, r = idx / (CQ * p.TW);
        const int gh = h0 + r, gw = w0 + col, c = c0 + 4 * q;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gh < p.H && gw < p.Wd && c < p.C)
            v = __ldg(reinterpret_cast<const float4*>(dY + (img + (long)gh * p.Wd + gw) * p.C + c));
        Gs[idx] = v;
    }
    __syncthreads();

    const int q = threadIdx.x, i = threadIdx.y, ls = threadIdx.z, NS = blockDim.z;
    float4 acc[KW];
#pragma unroll
    for (int j = 0; j < KW; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int nstrips = p.TW >> 3;
    for (int r = 0; r < p.TH; ++r) {
        for (int st = ls; st < nstrips; st += NS) {
            float4 dy[8];
#pragma unroll
            for (int pp = 0; pp < 8; ++pp) dy[pp] = Gs[((size_t)r * p.TW + st * 8 + pp) * CQ + q];
            const float4* xrow = Xs + ((size_t)(r + i) * cols + st * 8) * CQ + q;
#pragma unroll
            for (int xc = 0; xc < KW + 7; ++xc) {
                const float4 xv = xrow[(size_t)xc * CQ];
#pragma unroll
                for (int j = 0; j < KW; ++j) {
                    const int pp = xc - j;
                    if (pp >= 0 && pp < 8) acc[j] = f4_fma(dy[pp], xv, acc[j]);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < KW; ++j) {
        float* d = dWs + ((size_t)i * KW + j) * CT + 4 * q;
        atomicAdd(d + 0, acc[j].x); atomicAdd(d + 1, acc[j].y); atomicAdd(d + 2, acc[j].z); atomicAdd(d + 3, acc[j].w);
    }
    __syncthreads();
    for (int idx = tid; idx < p.kh * KW * CT; idx += nthr) {
        const int c = idx % CT, j = (idx / CT) % KW, ii = idx / (CT * KW);
        const int jr = j - joff;
        if (jr >= 0 && jr < p.kw && c0 + c < p.C)
            atomicAdd(dWt + ((long)(c0 + c) * p.kh + ii) * p.kw + jr, dWs[idx]);
    }
}

// ----------------------------------------------------------------------------------------------------------------
// 1-D fast path (ConvCNP / ConvLNP): no shared-memory tile.  A thread owns 4 channels x 8 consecutive positions and
// pulls its KW+7 input float4s straight from global memory in one batch (KW+7 independent 16-byte loads in flight per
// thread; neighbouring threads' halos hit L1/L2, DRAM sees each element once), then runs the taps out of registers.
// ----------------------------------------------------------------------------------------------------------------
struct Dw1Params {
    const float* X; const float* Wt; const float* bias; const float* res; float* Y;
    const float* Xorig; const float* scale; const float* shift; const float* addgrad;
    int L, C, kw;
    int relu_in, flip, mask, accum;
    long n_groups;        // B * ceil(L / 8)
    int groups_per_seq;
};

__device__ __forceinline__ float4 act4(float4 v, bool affine, const float4 s, const float4 t) {
    if (affine) v = make_float4(fmaf(s.x, v.x, t.x), fmaf(s.y, v.y, t.y), fmaf(s.z, v.z, t.z), fmaf(s.w, v.w, t.w));
    return make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
}

template <int KW>
__global__ void __launch_bounds__(256, KW <= 11 ? 2 : 1) dwconv1d_kernel(Dw1Params p) {
    extern __shared__ __align__(16) float4 Ws4[];   // [KW][CQ]
    const int CQ = p.C >> 2, G = 256 / CQ;
    const int q = threadIdx.x % CQ, g = threadIdx.x / CQ;
    const int pw = KW / 2, joff = (KW - p.kw) / 2;
    for (int idx = threadIdx.x; idx < KW * p.C; idx += 256) {
        const int c = idx % p.C, j = idx / p.C, jr = j - joff;
        float v = 0.f;
        if (jr >= 0 && jr < p.kw) v = __ldg(p.Wt + (long)c * p.kw + (p.flip ? p.kw - 1 - jr : jr));
        reinterpret_cast<float*>(Ws4)[(size_t)j * p.C + c] = v;
    }
    pdl_trigger();
    __syncthreads();
    pdl_wait();          // filters are parameters; the folded norm affine and the activations come from preceding kernels
    const int c = 4 * q;
    const bool affine = p.relu_in && p.scale != nullptr;
    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.scale && (p.relu_in || p.mask)) {
        sc = __ldg(reinterpret_cast<const float4*>(p.scale + c));
        sh = __ldg(reinterpret_cast<const float4*>(p.shift + c));
    }
    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.bias) bv = __ldg(reinterpret_cast<const float4*>(p.bias + c));
    // persistent: the filters are staged once per CTA, then the CTA strides over the position groups
    for (long gid = (long)blockIdx.x * G + g; gid < p.n_groups; gid += (long)gridDim.x * G) {
    const long b = gid / p.groups_per_seq;
    const int l0 = (int)(gid % p.groups_per_seq) * 8;
    const float* xb = p.X + (b * p.L) * (long)p.C + c;
    float4 xin[KW + 7];
#pragma unroll
    for (int xc = 0; xc < KW + 7; ++xc) {
        const int pos = l0 + xc - pw;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (pos >= 0 && pos < p.L) v = __ldg(reinterpret_cast<const float4*>(xb + (long)pos * p.C));
        xin[xc] = v;
    }
    if (p.relu_in) {
#pragma unroll
        for (int xc = 0; xc < KW + 7; ++xc) {
            const int pos = l0 + xc - pw;
            if (pos >= 0 && pos < p.L) xin[xc] = act4(xin[xc], affine, sc, sh);   // padding stays exactly 0
        }
    }
    float4 acc[8];
#pragma unroll
    for (int pp = 0; pp < 8; ++pp) acc[pp] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < KW; ++j) {
        const float4 w = Ws4[j * CQ + q];
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) acc[pp] = f4_fma(w, xin[pp + j], acc[pp]);
    }
#pragma unroll
    for (int pp = 0; pp < 8; ++pp) {
        const int pos = l0 + pp;
        if (pos >= p.L) continue;
        const long off = ((b * p.L) + pos) * (long)p.C + c;
        float4 v = make_float4(acc[pp].x + bv.x, acc[pp].y + bv.y, acc[pp].z + bv.z, acc[pp].w + bv.w);
        if (p.mask) {
            const float4 x = __ldg(reinterpret_cast<const float4*>(p.Xorig + off));
            const float4 pre = make_float4(fmaf(sc.x, x.x, sh.x), fmaf(sc.y, x.y, sh.y), fmaf(sc.z, x.z, sh.z), fmaf(sc.w, x.w, sh.w));
            v.x = pre.x > 0.f ? v.x * sc.x : 0.f; v.y = pre.y > 0.f ? v.y * sc.y : 0.f;
            v.z = pre.z > 0.f ? v.z * sc.z : 0.f; v.w = pre.w > 0.f ? v.w * sc.w : 0.f;
        }
        if (p.res) {
            const float4 rv = __ldg(reinterpret_cast<const float4*>(p.res + off));
            v.x += rv.x; v.y += rv.y; v.z += rv.z; v.w += rv.w;
        }
        if (p.addgrad) {   // gradient of the residual branch (the block input is also the conv input)
            const float4 rv = __ldg(reinterpret_cast<const float4*>(p.addgrad + off));
            v.x += rv.x; v.y += rv.y; v.z += rv.z; v.w += rv.w;
        }
        float4* out = reinterpret_cast<float4*>(p.Y + off);
        if (p.accum) { const float4 o = *out; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
        *out = v;
    }
    }   // position-group loop
}

// 1-D filter + bias gradient in one pass: dWt[c,j] += sum dY[b,l,c] act(X)[b,l+j-p,c] ; dbias[c] += sum dY[b,l,c].
// Persistent grid; a thread keeps its KW filter-tap sums for 4 channels in registers over all its position groups.
template <int KW>
__global__ void __launch_bounds__(256) dwconv1d_wgrad_kernel(Dw1Params p, const float* __restrict__ dY, float* __restrict__ dWt,
                                                             float* __restrict__ dbias) {
    extern __shared__ __align__(16) float4 red4[];   // [G][KW + 1][CQ]
    const int CQ = p.C >> 2, G = 256 / CQ;
    const int q = threadIdx.x % CQ, g = threadIdx.x / CQ;
    const int pw = KW / 2, joff = (KW - p.kw) / 2;
    const int c = 4 * q;
    const bool affine = p.relu_in && p.scale != nullptr;
    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (affine) {
        sc = __ldg(reinterpret_cast<const float4*>(p.scale + c));
        sh = __ldg(reinterpret_cast<const float4*>(p.shift + c));
    }
    float4 acc[KW], accb = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < KW; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (long gid = (long)blockIdx.x * G + g; gid < p.n_groups; gid += (long)gridDim.x * G) {
        const long b = gid / p.groups_per_seq;
        const int l0 = (int)(gid % p.groups_per_seq) * 8;
        const float* xb = p.X + (b * p.L) * (long)p.C + c;
        const float* gb = dY + (b * p.L) * (long)p.C + c;
        float4 xin[KW + 7], dy[8];
#pragma unroll
        for (int xc = 0; xc < KW + 7; ++xc) {
            const int pos = l0 + xc - pw;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pos >= 0 && pos < p.L) v = __ldg(reinterpret_cast<const float4*>(xb + (long)pos * p.C));
            xin[xc] = v;
        }
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) {
            const int pos = l0 + pp;
            dy[pp] = (pos < p.L) ? __ldg(reinterpret_cast<const float4*>(gb + (long)pos * p.C)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (p.relu_in) {
#pragma unroll
            for (int xc = 0; xc < KW + 7; ++xc) {
                const int pos = l0 + xc - pw;
                if (pos >= 0 && pos < p.L) xin[xc] = act4(xin[xc], affine, sc, sh);
            }
        }
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) {
            accb.x += dy[pp].x; accb.y += dy[pp].y; accb.z += dy[pp].z; accb.w += dy[pp].w;
#pragma unroll
            for (int j = 0; j < KW; ++j) acc[j] = f4_fma(dy[pp], xin[pp + j], acc[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < KW; ++j) red4[((size_t)g * (KW + 1) + j) * CQ + q] = acc[j];
    red4[((size_t)g * (KW + 1) + KW) * CQ + q] = accb;
    __syncthreads();
    const float* red = reinterpret_cast<const float*>(red4);
    for (int idx = threadIdx.x; idx < (KW + 1) * p.C; idx += 256) {
        const int ch = idx % p.C, j = idx / p.C;
        float s = 0.f;
        for (int gg = 0; gg < G; ++gg) s += red[((size_t)gg * (KW + 1) + j) * p.C + ch];
        if (j == KW) { if (dbias) atomicAdd(dbias + ch, s); }
        else {
            const int jr = j - joff;
            if (jr >= 0 && jr < p.kw) atomicAdd(dWt + (long)ch * p.kw + jr, s);
        }
    }
}

static bool dw1_ok(int H, int C) { return H == 1 && C % 4 == 0 && C <= 1024 && 256 % (C / 4) == 0; }

template <int KW>
static int launch_dw1(Dw1Params& p, int B, cudaStream_t st) {
    const int CQ = p.C / 4, G = 256 / CQ;
    p.groups_per_seq = (p.L + 7) / 8;
    p.n_groups = (long)B * p.groups_per_seq;
    const size_t smem = sizeof(float) * (size_t)KW * p.C;
    static int occ = 0;
    if (!occ) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dwconv1d_kernel<KW>, 256, smem) != cudaSuccess || occ < 1) { occ = 1; cudaGetLastError(); }
    }
    long grid = cdiv(p.n_groups, G);
    if (grid > (long)kNumSMs * occ) grid = (long)kNumSMs * occ;
    launch_pdl(dwconv1d_kernel<KW>, dim3((unsigned)grid), dim3(256), smem, st, p);
    count_launch();
    return check_launch("dwconv1d_kernel");
}

template <int KW>
static int launch_dw1_wgrad(Dw1Params& p, const float* dY, float* dWt, float* dbias, int B, cudaStream_t st) {
    const int CQ = p.C / 4, G = 256 / CQ;
    p.groups_per_seq = (p.L + 7) / 8;
    p.n_groups = (long)B * p.groups_per_seq;
    const size_t smem = sizeof(float) * (size_t)G * (KW + 1) * p.C;
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(dwconv1d_wgrad_kernel<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr = true; }
    if (smem > 200 * 1024) return NPF_ENOTSUP;
    static int occ = 0;
    if (!occ) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dwconv1d_wgrad_kernel<KW>, 256, smem) != cudaSuccess || occ < 1) { occ = 1; cudaGetLastError(); }
    }
    long grid = cdiv(p.n_groups, G);
    if (grid > (long)kNumSMs * occ) grid = (long)kNumSMs * occ;
    dwconv1d_wgrad_kernel<KW><<<(unsigned)grid, 256, smem, st>>>(p, dY, dWt, dbias);
    count_launch();
    return check_launch("dwconv1d_wgrad_kernel");
}

// Whole 1-D backward in one pass over dY and X (KW <= 11): the data gradient needs the dY window around 8 positions, and
// with the substitution m = l + j - pw the filter gradient needs the SAME window against act(X) at the 8 centres:
//     dX[m]  = act'(X[m]) * sum_j Wt[j] dY[m + pw - j]  (+ dY[m] for the residual branch)
//     dWt[j] += sum_m act(X)[m] dY[m + pw - j]          dbias += sum_m dY[m]
// so one register window of dY (KW + 7 float4) and the 8 centre X values feed both; X and dY are read once, dX written once.
template <int KW>
__global__ void __launch_bounds__(256, 1) dwconv1d_bwd_fused_kernel(Dw1Params p, float* __restrict__ dWt, float* __restrict__ dbias) {
    extern __shared__ __align__(16) float4 dyn4[];   // [KW][CQ] flipped filters, then [G][KW + 1][CQ] reduction scratch
    const int CQ = p.C >> 2, G = 256 / CQ;
    float4* Ws4 = dyn4;
    float4* red4 = dyn4 + (size_t)KW * CQ;
    const int q = threadIdx.x % CQ, g = threadIdx.x / CQ;
    const int pw = KW / 2, joff = (KW - p.kw) / 2;
    for (int idx = threadIdx.x; idx < KW * p.C; idx += 256) {
        const int c = idx % p.C, j = idx / p.C, jr = j - joff;
        reinterpret_cast<float*>(Ws4)[(size_t)j * p.C + c] = (jr >= 0 && jr < p.kw) ? __ldg(p.Wt + (long)c * p.kw + (p.kw - 1 - jr)) : 0.f;
    }
    pdl_trigger();
    __syncthreads();
    pdl_wait();
    const int c = 4 * q;
    const bool affine = p.mask && p.scale != nullptr;
    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (affine) {
        sc = __ldg(reinterpret_cast<const float4*>(p.scale + c));
        sh = __ldg(reinterpret_cast<const float4*>(p.shift + c));
    }
    float4 accw[KW], accb = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < KW; ++j) accw[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (long gid = (long)blockIdx.x * G + g; gid < p.n_groups; gid += (long)gridDim.x * G) {
        const long b = gid / p.groups_per_seq;
        const int l0 = (int)(gid % p.groups_per_seq) * 8;
        const float* gb = p.X + (b * p.L) * (long)p.C + c;          // dY
        const float* xb = p.Xorig + (b * p.L) * (long)p.C + c;      // layer input
        float4 dyw[KW + 7], xv[8];
#pragma unroll
        for (int xc = 0; xc < KW + 7; ++xc) {
            const int pos = l0 + xc - pw;
            dyw[xc] = (pos >= 0 && pos < p.L) ? __ldg(reinterpret_cast<const float4*>(gb + (long)pos * p.C)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int pp = 0; pp < 8; ++pp)
            xv[pp] = (l0 + pp < p.L) ? __ldg(reinterpret_cast<const float4*>(xb + (long)(l0 + pp) * p.C)) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 acc[8];
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) acc[pp] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < KW; ++j) {
            const float4 w = Ws4[j * CQ + q];
#pragma unroll
            for (int pp = 0; pp < 8; ++pp) acc[pp] = f4_fma(w, dyw[pp + j], acc[pp]);
        }
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) {
            const int pos = l0 + pp;
            if (pos >= p.L) continue;
            const float4 x = xv[pp];
            float4 v = acc[pp], ax = x;
            if (p.mask) {
                const float4 pre = make_float4(fmaf(sc.x, x.x, sh.x), fmaf(sc.y, x.y, sh.y), fmaf(sc.z, x.z, sh.z), fmaf(sc.w, x.w, sh.w));
                v.x = pre.x > 0.f ? v.x * sc.x : 0.f; v.y = pre.y > 0.f ? v.y * sc.y : 0.f;
                v.z = pre.z > 0.f ? v.z * sc.z : 0.f; v.w = pre.w > 0.f ? v.w * sc.w : 0.f;
                ax = make_float4(fmaxf(pre.x, 0.f), fmaxf(pre.y, 0.f), fmaxf(pre.z, 0.f), fmaxf(pre.w, 0.f));
            }
            const float4 dyc = dyw[pp + pw];
            if (p.addgrad) { v.x += dyc.x; v.y += dyc.y; v.z += dyc.z; v.w += dyc.w; }
            *reinterpret_cast<float4*>(p.Y + ((b * p.L) + pos) * (long)p.C + c) = v;
            accb.x += dyc.x; accb.y += dyc.y; accb.z += dyc.z; accb.w += dyc.w;
#pragma unroll
            for (int j = 0; j < KW; ++j) accw[j] = f4_fma(ax, dyw[pp + j], accw[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < KW; ++j) red4[((size_t)g * (KW + 1) + j) * CQ + q] = accw[j];
    red4[((size_t)g * (KW + 1) + KW) * CQ + q] = accb;
    __syncthreads();
    const float* red = reinterpret_cast<const float*>(red4);
    for (int idx = threadIdx.x; idx < (KW + 1) * p.C; idx += 256) {
        const int ch = idx % p.C, j = idx / p.C;
        float s = 0.f;
        for (int gg = 0; gg < G; ++gg) s += red[((size_t)gg * (KW + 1) + j) * p.C + ch];
        if (j == KW) { if (dbias) atomicAdd(dbias + ch, s); }
        else {
            const int jr = j - joff;           // accw[j] pairs with the flipped tap: dWt[kw - 1 - jr]
            if (jr >= 0 && jr < p.kw) atomicAdd(dWt + (long)ch * p.kw + (p.kw - 1 - jr), s);
        }
    }
}

template <int KW>
static int launch_dw1_bwd_fused(Dw1Params& p, float* dWt, float* dbias, int B, cudaStream_t st) {
    const int CQ = p.C / 4, G = 256 / CQ;
    p.groups_per_seq = (p.L + 7) / 8;
    p.n_groups = (long)B * p.groups_per_seq;
    const size_t smem = sizeof(float) * ((size_t)KW * p.C + (size_t)G * (KW + 1) * p.C);
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(dwconv1d_bwd_fused_kernel<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr = true; }
    if (smem > 200 * 1024) return NPF_ENOTSUP;
    long grid = cdiv(p.n_groups, G);
    if (grid > (long)kNumSMs) grid = kNumSMs;
    launch_pdl(dwconv1d_bwd_fused_kernel<KW>, dim3((unsigned)grid), dim3(256), smem, st, p, dWt, dbias);
    count_launch();
    return check_launch("dwconv1d_bwd_fused_kernel");
}

// ----------------------------------------------------------------------------------------------------------------
// 2-D fast path (GridConvCNP / GridConvLNP, 32x32-ish images, k = 9 / 11): FFMA-bound (121 taps per output), so the kernels are
// organised around register reuse and the shared-memory pipe.  A WARP owns one channel pair, and every lane of it works on the SAME
// two channels (packed fp32x2: one FFMA2 per tap and pixel), so
//   * a filter tap is one address for the whole warp: LDS.128 broadcasts (two taps each, one wavefront);
//   * a lane owns 8 rows x 4 columns of the 32 x 32 output tile (64 float2 accumulators); an input row segment (4 + KW - 1 pixels, 7
//     LDS.128) is loaded ONCE and feeds every (output row, tap row) combination it belongs to: 44 FFMA2 per combination;
//   * the tile is stored plane by plane (pair, row, column) with a 16-byte shift on every other 8-row block, which makes the 32-byte
//     lane stride of the window loads conflict-free across the four row blocks of a warp.
// Per warp and tile: 3 872 FFMA2 against ~1 030 shared-memory wavefronts: FMA-bound.  CTA = one image tile x 8 channels (4 warps),
// 63 KB of shared memory: three CTAs per SM.
// ----------------------------------------------------------------------------------------------------------------
constexpr int V2T = 32;          // output tile edge
constexpr int V2P = 4;           // channel pairs (warps) per CTA

template <int KW>
__global__ void __launch_bounds__(V2P * 32, 3) dwconv2d_v2_kernel(DwParams p) {
    constexpr int ROWS = V2T + KW - 1, COLS = V2T + KW - 1;
    constexpr int PITCH = COLS * 8 + 16;                 // bytes per staged row (float2 per pixel) + room for the 16-byte shift
    constexpr int PLANE = ROWS * PITCH;
    constexpr int WP = KW + 1;                           // taps per filter row, padded to an even count (LDS.128 = two taps)
    constexpr int XC = 4 + KW - 1;                       // input pixels per lane and row
    static_assert(PITCH % 16 == 0 && XC % 2 == 0 && WP % 2 == 0, "layout");
    extern __shared__ __align__(16) uint8_t smem_v2[];
    uint8_t* xs = smem_v2;                                // [V2P][ROWS][PITCH]
    float2* ws = reinterpret_cast<float2*>(smem_v2 + V2P * PLANE);     // [V2P][KW][WP]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tile = blockIdx.x;
    const int h0 = (tile / p.tiles_w) * V2T, w0 = (tile % p.tiles_w) * V2T;
    const int c0 = blockIdx.y * (2 * V2P);
    const int b = blockIdx.z;
    const int ph = KW / 2, joff = (KW - p.kw) / 2;        // kh == kw (<= KW); narrower filters are centred in the padded one
    const long img = (long)b * p.H * p.Wd;

    // ---- filters: ws[pair][i][j] = (W[c0 + 2 pair][i][j], W[c0 + 2 pair + 1][i][j]), flipped for the data gradient, zero padding
    for (int idx = tid; idx < V2P * KW * WP; idx += V2P * 32) {
        const int j = idx % WP, i = (idx / WP) % KW, pr = idx / (WP * KW);
        float2 v = make_float2(0.f, 0.f);
        const int ir = i - joff, jr = j - joff;
        if (ir >= 0 && ir < p.kh && jr >= 0 && jr < p.kw) {
            const int ii = p.flip ? p.kh - 1 - ir : ir, jj = p.flip ? p.kw - 1 - jr : jr;
            const float* w = p.Wt + ((long)(c0 + 2 * pr) * p.kh + ii) * p.kw + jj;
            v = make_float2(__ldg(w), __ldg(w + (long)p.kh * p.kw));
        }
        ws[idx] = v;
    }
    // ---- input tile with halo: thread = (pixel, half of the 8 channels); activation only on real pixels (the padding stays exactly 0)
    {
        constexpr int SB = 14;                              // loads in flight per thread: the accumulators are not live yet, two round trips stage the tile
        const bool affine = p.relu_in && p.scale != nullptr;
        const int half = tid & 1;
        float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
        if (affine) { sc = __ldg(reinterpret_cast<const float4*>(p.scale + c0 + 4 * half)); sh = __ldg(reinterpret_cast<const float4*>(p.shift + c0 + 4 * half)); }
        for (int base = 0; base < ROWS * COLS; base += SB * (V2P * 16)) {
            float4 v[SB];
            int pix[SB];
#pragma unroll
            for (int u = 0; u < SB; ++u) {
                pix[u] = base + u * (V2P * 16) + (tid >> 1);
                v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (pix[u] < ROWS * COLS) {
                    const int rr = pix[u] / COLS, cc = pix[u] - rr * COLS;
                    const int gh = h0 + rr - ph, gw = w0 + cc - ph;
                    if (gh >= 0 && gh < p.H && gw >= 0 && gw < p.Wd) {
                        v[u] = __ldg(reinterpret_cast<const float4*>(p.X + (img + (long)gh * p.Wd + gw) * p.C + c0 + 4 * half));
                        if (p.relu_in) v[u] = act4(v[u], affine, sc, sh);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < SB; ++u) {
                if (pix[u] >= ROWS * COLS) continue;
                const int rr = pix[u] / COLS, cc = pix[u] - rr * COLS;
                uint8_t* d = xs + (2 * half) * PLANE + rr * PITCH + ((rr >> 3) & 1) * 16 + cc * 8;
                *reinterpret_cast<float2*>(d) = make_float2(v[u].x, v[u].y);
                *reinterpret_cast<float2*>(d + PLANE) = make_float2(v[u].z, v[u].w);
            }
        }
    }
    __syncthreads();

    // ---- main loop: lane = (column quad cq, row block rb) of the warp's channel pair
    const int cq = lane & 7, rb = lane >> 3;
    const uint8_t* plane = xs + warp * PLANE + (4 * cq) * 8;
    const float2* wp = ws + warp * (KW * WP);
    float2 acc[8][4];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = make_float2(0.f, 0.f);
#pragma unroll 1
    for (int rr = 0; rr < 8 + KW - 1; ++rr) {            // tile row 8 rb + rr feeds output row r through tap row i = rr - r
        const int trow = 8 * rb + rr;
        const uint8_t* rowp = plane + trow * PITCH + ((trow >> 3) & 1) * 16;
        float2 x[XC];
#pragma unroll
        for (int k = 0; k < XC / 2; ++k) {
            const float4 t = *reinterpret_cast<const float4*>(rowp + 16 * k);
            x[2 * k] = make_float2(t.x, t.y);
            x[2 * k + 1] = make_float2(t.z, t.w);
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int i = rr - r;
            if (i < 0 || i >= KW) continue;                // uniform over the warp
            float2 w[WP];
#pragma unroll
            for (int k = 0; k < WP / 2; ++k) {
                const float4 t = *reinterpret_cast<const float4*>(wp + i * WP + 2 * k);      // one address per warp: broadcast
                w[2 * k] = make_float2(t.x, t.y);
                w[2 * k + 1] = make_float2(t.z, t.w);
            }
#pragma unroll
            for (int j = 0; j < KW; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = __ffma2_rn(w[j], x[c + j], acc[r][c]);
        }
    }

    // ---- epilogue.  The accumulators go through shared memory (the input planes are dead) so that global memory is touched the way the
    // staging touches it: thread = (pixel, half of the 8 channels), 16-byte accesses, 32 contiguous bytes per pixel.  Written straight
    // from the accumulator layout (lane = 4 columns of ONE channel pair) every store / mask load / residual load instruction would
    // touch 32 different cache lines for 8 bytes each: four times the LSU wavefronts, and it was those that bounded the kernel.
    __syncthreads();
    {
        float2* op = reinterpret_cast<float2*>(xs) + warp * (V2T * V2T);          // [pair][32 rows][32 cols]
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int c = 0; c < 4; c += 2)
                *reinterpret_cast<float4*>(op + (8 * rb + r) * V2T + 4 * cq + c) = make_float4(acc[r][c].x, acc[r][c].y, acc[r][c + 1].x, acc[r][c + 1].y);
    }
    __syncthreads();
    {
        const int half = tid & 1;
        const int ch = c0 + 4 * half;
        const float2* o0 = reinterpret_cast<const float2*>(xs) + (2 * half) * (V2T * V2T);
        float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) bv = __ldg(reinterpret_cast<const float4*>(p.bias + ch));
        float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.mask && p.scale) { sc = __ldg(reinterpret_cast<const float4*>(p.scale + ch)); sh = __ldg(reinterpret_cast<const float4*>(p.shift + ch)); }
#pragma unroll 1
        constexpr int EB = 8;
        for (int base = 0; base < V2T * V2T; base += EB * (V2P * 16)) {
            float4 xo[EB], rv[EB], ov[EB];
            long off[EB];
            bool ok[EB];
#pragma unroll
            for (int u = 0; u < EB; ++u) {
                const int pix = base + u * (V2P * 16) + (tid >> 1);
                const int gh = h0 + (pix >> 5), gw = w0 + (pix & 31);
                ok[u] = gh < p.H && gw < p.Wd;
                off[u] = (img + (long)gh * p.Wd + gw) * p.C + ch;
                if (ok[u]) {
                    if (p.mask) xo[u] = __ldg(reinterpret_cast<const float4*>(p.Xorig + off[u]));
                    if (p.res) rv[u] = __ldg(reinterpret_cast<const float4*>(p.res + off[u]));
                    if (p.accum) ov[u] = *reinterpret_cast<const float4*>(p.Y + off[u]);
                }
            }
#pragma unroll
            for (int u = 0; u < EB; ++u) {
                if (!ok[u]) continue;
                const int pix = base + u * (V2P * 16) + (tid >> 1);
                const float2 a = o0[pix], bq = o0[V2T * V2T + pix];
                float4 v = make_float4(a.x + bv.x, a.y + bv.y, bq.x + bv.z, bq.y + bv.w);
                if (p.mask) {
                    v.x = fmaf(sc.x, xo[u].x, sh.x) > 0.f ? v.x * sc.x : 0.f;
                    v.y = fmaf(sc.y, xo[u].y, sh.y) > 0.f ? v.y * sc.y : 0.f;
                    v.z = fmaf(sc.z, xo[u].z, sh.z) > 0.f ? v.z * sc.z : 0.f;
                    v.w = fmaf(sc.w, xo[u].w, sh.w) > 0.f ? v.w * sc.w : 0.f;
                }
                if (p.res) { v.x += rv[u].x; v.y += rv[u].y; v.z += rv[u].z; v.w += rv[u].w; }
                if (p.accum) { v.x += ov[u].x; v.y += ov[u].y; v.z += ov[u].z; v.w += ov[u].w; }
                *reinterpret_cast<float4*>(p.Y + off[u]) = v;
            }
        }
    }
}

template <int KW>
static int launch_dw2(DwParams& p, int B, cudaStream_t st) {
    constexpr int ROWS = V2T + KW - 1, PITCH = ROWS * 8 + 16;
    const size_t smem = (size_t)V2P * ROWS * PITCH + (size_t)V2P * KW * (KW + 1) * sizeof(float2);
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(dwconv2d_v2_kernel<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024); attr = true; }
    p.tiles_w = (int)cdiv(p.Wd, V2T);
    dim3 grid((unsigned)(p.tiles_w * cdiv(p.H, V2T)), (unsigned)(p.C / (2 * V2P)), (unsigned)B);
    dwconv2d_v2_kernel<KW><<<grid, V2P * 32, smem, st>>>(p);
    count_launch();
    return check_launch("dwconv2d_v2_kernel");
}

// ----------------------------------------------------------------------------------------------------------------
// 2-D filter gradient: dW[c,i,j] = sum_{b,h,w} dY[b,h,w,c] act(X)[b,h+i-p,w+j-p,c].
// A persistent CTA = 8 channels (4 pairs) x 3 groups of 4 filter rows = 12 warps; it walks a share of the images and keeps its
// 4 x KW packed accumulators per lane IN REGISTERS for all of them: the cross-lane reduction (shuffles) and the atomics happen once per
// CTA, not once per image.  Per image the act(X) halo tile and the dY tile are staged as channel-pair planes (the layout of
// dwconv2d_v2_kernel, shifted every 4 rows); a lane owns 4 rows x 4 columns of a 16-row half of the tile: the 4 x 4 dY values sit in
// registers, every act(X) row segment (4 + KW - 1 pixels, 7 LDS.128) it loads feeds up to 4 filter rows x KW taps x 4 columns = 176 FFMA2.
// ----------------------------------------------------------------------------------------------------------------
constexpr int WGI = 4;           // filter rows per warp group
constexpr int WGG = 3;           // warp groups (3 x 4 >= KW)

template <int KW>
__global__ void __launch_bounds__(V2P * WGG * 32, 1) dwconv2d_wgrad_v2_kernel(DwParams p, const float* __restrict__ dY, float* __restrict__ dWt, int B, int ipc) {
    constexpr int ROWS = V2T + KW - 1, COLS = V2T + KW - 1;
    constexpr int PITCH = COLS * 8 + 16, PLANE = ROWS * PITCH;
    constexpr int GPITCH = V2T * 8 + 16, GPLANE = V2T * GPITCH;
    constexpr int XC = 4 + KW - 1;
    constexpr int NT = V2P * WGG * 32;
    static_assert(KW <= WGI * WGG && XC % 2 == 0, "filter rows per group");
    extern __shared__ __align__(16) uint8_t smem_v2[];
    uint8_t* xs = smem_v2;                                // act(X): [V2P][ROWS][PITCH]
    uint8_t* gs = smem_v2 + V2P * PLANE;                  // dY:     [V2P][32][GPITCH]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int pair = warp & (V2P - 1), grp = warp / V2P;
    const int i0 = WGI * grp, IC = min(WGI, KW - i0);    // this warp's filter rows [i0, i0 + IC)
    const int tile = blockIdx.x;
    const int h0 = (tile / p.tiles_w) * V2T, w0 = (tile % p.tiles_w) * V2T;
    const int c0 = blockIdx.y * (2 * V2P);
    const int ph = KW / 2, joff = (KW - p.kw) / 2;
    const int cq = lane & 7, rb = lane >> 3;

    float2 acc[WGI][KW];
#pragma unroll
    for (int ii = 0; ii < WGI; ++ii)
#pragma unroll
        for (int j = 0; j < KW; ++j) acc[ii][j] = make_float2(0.f, 0.f);

    const bool affine = p.relu_in && p.scale != nullptr;
    const int half = tid & 1;
    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (affine) { sc = __ldg(reinterpret_cast<const float4*>(p.scale + c0 + 4 * half)); sh = __ldg(reinterpret_cast<const float4*>(p.shift + c0 + 4 * half)); }

    const int b_begin = blockIdx.z * ipc, b_end = min(B, b_begin + ipc);
    for (int b = b_begin; b < b_end; ++b) {
        const long img = (long)b * p.H * p.Wd;
        // ---- stage act(X) with halo and dY: thread = (pixel, half of the 8 channels)
        for (int base = 0; base < ROWS * COLS; base += 4 * (NT / 2)) {
            float4 v[4];
            int pix[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                pix[u] = base + u * (NT / 2) + (tid >> 1);
                v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (pix[u] < ROWS * COLS) {
                    const int rr = pix[u] / COLS, cc = pix[u] - rr * COLS;
                    const int gh = h0 + rr - ph, gw = w0 + cc - ph;
                    if (gh >= 0 && gh < p.H && gw >= 0 && gw < p.Wd) {
                        v[u] = __ldg(reinterpret_cast<const float4*>(p.X + (img + (long)gh * p.Wd + gw) * p.C + c0 + 4 * half));
                        if (p.relu_in) v[u] = act4(v[u], affine, sc, sh);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (pix[u] >= ROWS * COLS) continue;
                const int rr = pix[u] / COLS, cc = pix[u] - rr * COLS;
                uint8_t* d = xs + (2 * half) * PLANE + rr * PITCH + ((rr >> 2) & 1) * 16 + cc * 8;
                *reinterpret_cast<float2*>(d) = make_float2(v[u].x, v[u].y);
                *reinterpret_cast<float2*>(d + PLANE) = make_float2(v[u].z, v[u].w);
            }
        }
        for (int base = 0; base < V2T * V2T; base += 4 * (NT / 2)) {
            float4 v[4];
            int pix[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                pix[u] = base + u * (NT / 2) + (tid >> 1);
                v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (pix[u] < V2T * V2T) {
                    const int gh = h0 + (pix[u] >> 5), gw = w0 + (pix[u] & 31);
                    if (gh < p.H && gw < p.Wd) v[u] = __ldg(reinterpret_cast<const float4*>(dY + (img + (long)gh * p.Wd + gw) * p.C + c0 + 4 * half));
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (pix[u] >= V2T * V2T) continue;
                const int rr = pix[u] >> 5, cc = pix[u] & 31;
                uint8_t* d = gs + (2 * half) * GPLANE + rr * GPITCH + ((rr >> 2) & 1) * 16 + cc * 8;
                *reinterpret_cast<float2*>(d) = make_float2(v[u].x, v[u].y);
                *reinterpret_cast<float2*>(d + GPLANE) = make_float2(v[u].z, v[u].w);
            }
        }
        __syncthreads();
        // ---- two 16-row halves of the tile; lane = (column quad cq, 4-row block rb)
#pragma unroll 1
        for (int hh = 0; hh < 2; ++hh) {
            const int r0 = 16 * hh + 4 * rb;                       // first output row of this lane
            float2 dy[4][4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const uint8_t* gp = gs + pair * GPLANE + (r0 + r) * GPITCH + (((r0 + r) >> 2) & 1) * 16 + (4 * cq) * 8;
                const float4 t0 = *reinterpret_cast<const float4*>(gp), t1 = *reinterpret_cast<const float4*>(gp + 16);
                dy[r][0] = make_float2(t0.x, t0.y); dy[r][1] = make_float2(t0.z, t0.w);
                dy[r][2] = make_float2(t1.x, t1.y); dy[r][3] = make_float2(t1.z, t1.w);
            }
            const uint8_t* plane = xs + pair * PLANE + (4 * cq) * 8;
#pragma unroll
            for (int rr = 0; rr < 4 + WGI - 1; ++rr) {             // act(X) tile row r0 + i0 + rr meets output row r through filter row i0 + (rr - r)
                if (rr >= 4 + IC - 1) continue;                    // uniform over the warp
                const int trow = r0 + i0 + rr;
                const uint8_t* rowp = plane + trow * PITCH + ((trow >> 2) & 1) * 16;
                float2 x[XC];
#pragma unroll
                for (int k = 0; k < XC / 2; ++k) {
                    const float4 t = *reinterpret_cast<const float4*>(rowp + 16 * k);
                    x[2 * k] = make_float2(t.x, t.y);
                    x[2 * k + 1] = make_float2(t.z, t.w);
                }
#pragma unroll
                for (int ii = 0; ii < WGI; ++ii) {
                    const int r = rr - ii;
                    if (r < 0 || r >= 4 || ii >= IC) continue;
#pragma unroll
                    for (int j = 0; j < KW; ++j)
#pragma unroll
                        for (int c = 0; c < 4; ++c) acc[ii][j] = __ffma2_rn(dy[r][c], x[c + j], acc[ii][j]);
                }
            }
        }
        __syncthreads();
    }
    // ---- one reduction over the warp's lanes and one atomic per tap and channel for the whole share of images
#pragma unroll
    for (int ii = 0; ii < WGI; ++ii) {
        if (ii >= IC) continue;
#pragma unroll
        for (int j = 0; j < KW; ++j) {
            float2 v = acc[ii][j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                v.x += __shfl_xor_sync(0xffffffffu, v.x, o);
                v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
            }
            const int ir = i0 + ii - joff, jr = j - joff;
            if (lane == 0 && ir >= 0 && ir < p.kh && jr >= 0 && jr < p.kw) {
                float* d = dWt + ((long)(c0 + 2 * pair) * p.kh + ir) * p.kw + jr;
                atomicAdd(d, v.x);
                atomicAdd(d + (long)p.kh * p.kw, v.y);
            }
        }
    }
}

template <int KW>
static int launch_dw2_wgrad(DwParams& p, const float* dY, float* dWt, int B, cudaStream_t st) {
    constexpr int ROWS = V2T + KW - 1, PITCH = ROWS * 8 + 16;
    const size_t smem = (size_t)V2P * ROWS * PITCH + (size_t)V2P * V2T * (V2T * 8 + 16);
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(dwconv2d_wgrad_v2_kernel<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024); attr = true; }
    p.tiles_w = (int)cdiv(p.Wd, V2T);
    const int tiles = p.tiles_w * (int)cdiv(p.H, V2T), groups = p.C / (2 * V2P);
    int nz = kNumSMs / (tiles * groups);                              // image shares: at most one CTA per SM (one resident CTA each: no second wave)
    if (nz < 1) nz = 1;
    if (nz > B) nz = B;
    const int ipc = (int)cdiv(B, nz);
    nz = (int)cdiv(B, ipc);
    dim3 grid((unsigned)tiles, (unsigned)groups, (unsigned)nz);
    dwconv2d_wgrad_v2_kernel<KW><<<grid, V2P * WGG * 32, smem, st>>>(p, dY, dWt, B, ipc);
    count_launch();
    return check_launch("dwconv2d_wgrad_v2_kernel");
}

// The 2-D kernels need C % (2 V2P) == 0 and a square filter; shapes outside dw2_ok run the generic dwconv_kernel.
static bool dw2_ok(int H, int C, int kh, int kw) { return H > 1 && C % 16 == 0 && kh == kw && kh <= 11; }

// sum[c] += sum_m X[m,c] ; sumsq[c] += sum_m X[m,c]^2   (also used for the conv bias gradient with sumsq == null)
__global__ void __launch_bounds__(256) channel_stats_kernel(const float* __restrict__ X, const float* __restrict__ center, float* sum,
                                                            float* sumsq, long M, int C, long rows_per_block) {
    __shared__ float s1[8][33], s2[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.y * 32 + tx;
    const long m0 = (long)blockIdx.x * rows_per_block, m1 = min(M, m0 + rows_per_block);
    float a = 0.f, b = 0.f;
    if (c < C) {
        const float ctr = center ? __ldg(center + c) : 0.f;
        for (long m = m0 + ty; m < m1; m += 8) {
            const float v = __ldg(X + m * C + c) - ctr;
            a += v;
            b = fmaf(v, v, b);
        }
    }
    s1[ty][tx] = a; s2[ty][tx] = b;
    __syncthreads();
    if (ty == 0 && c < C) {
#pragma unroll
        for (int i = 1; i < 8; ++i) { a += s1[i][tx]; b += s2[i][tx]; }
        if (sum) atomicAdd(sum + c, a);
        if (sumsq) atomicAdd(sumsq + c, b);
    }
}

static int pick_kw(int kw) { return kw <= 9 ? 9 : (kw <= 11 ? 11 : (kw <= 19 ? 19 : -1)); }

static void pick_tiles(DwParams& p, dim3& block) {
    if (p.H == 1) { p.TH = 1; p.TW = 64; p.CT = p.C >= 128 ? 128 : ((p.C + 3) / 4) * 4; }
    else          { p.TH = 8; p.TW = 16; p.CT = p.C >= 32 ? 32 : ((p.C + 3) / 4) * 4; }
    block = dim3(p.CT / 4, p.TW / 8, p.TH);
    p.tiles_w = (int)cdiv(p.Wd, p.TW);
}

template <int KW>
static int launch_dw(DwParams& p, int B, cudaStream_t st) {
    dim3 block;
    pick_tiles(p, block);
    const size_t smem = ((size_t)(p.TH + p.kh - 1) * (p.TW + KW - 1) * p.CT + (size_t)p.kh * KW * p.CT) * sizeof(float);
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(dwconv_kernel<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr_set = true;
    }
    if (smem > 200 * 1024) { set_error("dwconv: tile needs %zu B of shared memory", smem); return NPF_ENOTSUP; }
    dim3 grid((unsigned)(p.tiles_w * cdiv(p.H, p.TH)), (unsigned)cdiv(p.C, p.CT), (unsigned)B);
    dwconv_kernel<KW><<<grid, block, smem, st>>>(p);
    count_launch();
    return check_launch("dwconv_kernel");
}

template <int KW>
static int launch_dw_wgrad(DwParams& p, const float* dY, float* dWt, int B, cudaStream_t st) {
    dim3 block;
    pick_tiles(p, block);
    int ns = 256 / ((p.CT / 4) * p.kh);
    if (ns < 1) ns = 1;
    if (ns > p.TW / 8) ns = p.TW / 8;
    block = dim3(p.CT / 4, p.kh, ns);
    if (block.x * block.y * block.z > 256) { set_error("dwconv wgrad: kh=%d too large", p.kh); return NPF_ENOTSUP; }
    const size_t smem = ((size_t)(p.TH + p.kh - 1) * (p.TW + KW - 1) * p.CT + (size_t)p.TH * p.TW * p.CT +
                         (size_t)p.kh * KW * p.CT) * sizeof(float);
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(dwconv_wgrad_kernel<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr_set = true;
    }
    if (smem > 200 * 1024) { set_error("dwconv wgrad: tile needs %zu B of shared memory", smem); return NPF_ENOTSUP; }
    dim3 grid((unsigned)(p.tiles_w * cdiv(p.H, p.TH)), (unsigned)cdiv(p.C, p.CT), (unsigned)B);
    dwconv_wgrad_kernel<KW><<<grid, block, smem, st>>>(p, dY, dWt);
    count_launch();
    return check_launch("dwconv_wgrad_kernel");
}

// Y[m,c] (+)= a[c] * X[m,c] + b[c]
__global__ void channel_affine_kernel(const float* __restrict__ X, const float* __restrict__ a, const float* __restrict__ b,
                                      float* __restrict__ Y, long n, int C, int accumulate) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const float v = fmaf(__ldg(a + c), __ldg(X + i), __ldg(b + c));
        Y[i] = accumulate ? Y[i] + v : v;
    }
}

static int launch_stats(const float* X, const float* center, float* sum, float* sumsq, long M, int C, cudaStream_t st) {
    long rows_per_block = cdiv(M, 2L * kNumSMs);
    if (rows_per_block < 64) rows_per_block = 64;
    dim3 grid((unsigned)cdiv(M, rows_per_block), (unsigned)cdiv(C, 32));
    channel_stats_kernel<<<grid, 256, 0, st>>>(X, center, sum, sumsq, M, C, rows_per_block);
    count_launch();
    return check_launch("channel_stats_kernel");
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace npf

using namespace npf;


extern "C" int npf_dwconv_fwd(const float* X, const float* Wt, const float* bias, const float* res, float* Y, int B,
                              int H, int Wd, int C, int kh, int kw, int flags, const float* pre_scale,
                              const float* pre_shift, npf_stream_t stream) {
    NPF_REQUIRE(X && Wt && Y, "npf_dwconv_fwd: null pointer");
    NPF_REQUIRE(B >= 0 && H >= 1 && Wd >= 1 && C >= 4 && C % 4 == 0, "npf_dwconv_fwd: bad shape (C must be a multiple of 4)");
    NPF_REQUIRE(kh >= 1 && kw >= 1 && (kh & 1) && (kw & 1), "npf_dwconv_fwd: kernel sizes must be odd");
    NPF_REQUIRE(H > 1 || kh == 1, "npf_dwconv_fwd: 1-D signals use H = 1, kh = 1");
    NPF_REQUIRE((pre_scale == nullptr) == (pre_shift == nullptr), "npf_dwconv_fwd: scale and shift go together");
    NPF_REQUIRE(aligned16(X) && aligned16(Y) && (!res || aligned16(res)) && (!bias || aligned16(bias)) &&
                    (!pre_scale || (aligned16(pre_scale) && aligned16(pre_shift))),
                "npf_dwconv_fwd: pointers must be 16-byte aligned");
    NPF_REQUIRE(B <= 65535, "npf_dwconv_fwd: batch > 65535");
    if (B == 0) return NPF_OK;
    DwParams p{};
    p.X = X; p.Wt = Wt; p.bias = bias; p.res = res; p.Y = Y;
    p.scale = pre_scale; p.shift = pre_shift;
    p.H = H; p.Wd = Wd; p.C = C; p.kh = kh; p.kw = kw;
    p.relu_in = (flags & NPF_RELU_IN) ? 1 : 0;
    p.accum = (flags & NPF_ACCUM) ? 1 : 0;
    cudaStream_t st = as_stream(stream);
    int rc;
    if (dw1_ok(H, C) && pick_kw(kw) > 0) {
        Dw1Params q{};
        q.X = X; q.Wt = Wt; q.bias = bias; q.res = res; q.Y = Y; q.scale = pre_scale; q.shift = pre_shift;
        q.L = Wd; q.C = C; q.kw = kw; q.relu_in = p.relu_in; q.accum = p.accum;
        switch (pick_kw(kw)) {
            case 9: return launch_dw1<9>(q, B, st);
            case 11: return launch_dw1<11>(q, B, st);
            default: return launch_dw1<19>(q, B, st);
        }
    }
    if (dw2_ok(H, C, kh, kw)) return kw <= 9 ? launch_dw2<9>(p, B, st) : launch_dw2<11>(p, B, st);
    switch (pick_kw(kw)) {
        case 9: rc = launch_dw<9>(p, B, st); break;
        case 11: rc = launch_dw<11>(p, B, st); break;
        case 19: rc = launch_dw<19>(p, B, st); break;
        default: set_error("npf_dwconv_fwd: kernel width %d > 19", kw); return NPF_ENOTSUP;
    }
    return rc;
}

extern "C" int npf_dwconv_bwd(const float* dY, const float* X, const float* Wt, float* dX, float* dWt, float* dbias,
                              int B, int H, int Wd, int C, int kh, int kw, int flags, const float* pre_scale,
                              const float* pre_shift, float* dpre_scale, float* dpre_shift, npf_stream_t stream) {
    NPF_REQUIRE(dY && X && Wt, "npf_dwconv_bwd: null pointer");
    NPF_REQUIRE(B >= 0 && H >= 1 && Wd >= 1 && C >= 4 && C % 4 == 0, "npf_dwconv_bwd: bad shape");
    NPF_REQUIRE(kh >= 1 && kw >= 1 && (kh & 1) && (kw & 1), "npf_dwconv_bwd: kernel sizes must be odd");
    NPF_REQUIRE((pre_scale == nullptr) == (pre_shift == nullptr), "npf_dwconv_bwd: scale and shift go together");
    NPF_REQUIRE((dpre_scale == nullptr) == (dpre_shift == nullptr), "npf_dwconv_bwd: dscale and dshift go together");
    NPF_REQUIRE(!dpre_scale || (pre_scale && dX), "npf_dwconv_bwd: affine gradients need the affine and dX");
    NPF_REQUIRE(aligned16(dY) && aligned16(X) && (!dX || aligned16(dX)), "npf_dwconv_bwd: pointers must be 16-byte aligned");
    NPF_REQUIRE(B <= 65535, "npf_dwconv_bwd: batch > 65535");
    if (B == 0) return NPF_OK;
    cudaStream_t st = as_stream(stream);
    const int relu_in = (flags & NPF_RELU_IN) ? 1 : 0;
    int rc = NPF_OK;
    const int kwsel = pick_kw(kw);
    if (kwsel < 0) { set_error("npf_dwconv_bwd: kernel width %d > 19", kw); return NPF_ENOTSUP; }
    const bool fast1d = dw1_ok(H, C) && !dpre_scale;
    if (fast1d && dX && dWt && !(flags & NPF_ACCUM) && kwsel <= 11) {   // one pass: data + filter + bias gradient
        Dw1Params q{};
        q.X = dY; q.Wt = Wt; q.Y = dX; q.Xorig = X; q.scale = pre_scale; q.shift = pre_shift;
        q.addgrad = (flags & NPF_ADD_DY) ? dY : nullptr;
        q.L = Wd; q.C = C; q.kw = kw; q.mask = relu_in;
        rc = kwsel == 9 ? launch_dw1_bwd_fused<9>(q, dWt, dbias, B, st) : launch_dw1_bwd_fused<11>(q, dWt, dbias, B, st);
        if (rc != NPF_ENOTSUP) return rc;
    }
    if (fast1d) {
        if (dX) {
            Dw1Params q{};
            q.X = dY; q.Wt = Wt; q.Y = dX; q.Xorig = X; q.scale = pre_scale; q.shift = pre_shift;
            q.addgrad = (flags & NPF_ADD_DY) ? dY : nullptr;
            q.L = Wd; q.C = C; q.kw = kw; q.flip = 1; q.mask = relu_in; q.accum = (flags & NPF_ACCUM) ? 1 : 0;
            switch (kwsel) {
                case 9: rc = launch_dw1<9>(q, B, st); break;
                case 11: rc = launch_dw1<11>(q, B, st); break;
                default: rc = launch_dw1<19>(q, B, st); break;
            }
            if (rc != NPF_OK) return rc;
        }
        if (dWt) {
            Dw1Params q{};
            q.X = X; q.scale = pre_scale; q.shift = pre_shift; q.L = Wd; q.C = C; q.kw = kw; q.relu_in = relu_in;
            switch (kwsel) {
                case 9: rc = launch_dw1_wgrad<9>(q, dY, dWt, dbias, B, st); break;
                case 11: rc = launch_dw1_wgrad<11>(q, dY, dWt, dbias, B, st); break;
                default: rc = launch_dw1_wgrad<19>(q, dY, dWt, dbias, B, st); break;
            }
            if (rc != NPF_ENOTSUP) return rc;
        } else if (dbias) {
            return launch_stats(dY, nullptr, dbias, nullptr, (long)B * H * Wd, C, st);
        } else {
            return rc;
        }
    }
    if (dX && !fast1d) {
        DwParams p{};
        p.X = dY; p.Wt = Wt; p.Y = dX; p.Xorig = X;
        p.scale = pre_scale; p.shift = pre_shift; p.dscale = dpre_scale; p.dshift = dpre_shift;
        p.H = H; p.Wd = Wd; p.C = C; p.kh = kh; p.kw = kw;
        p.relu_in = 0; p.flip = 1; p.mask = relu_in; p.accum = (flags & NPF_ACCUM) ? 1 : 0;
        p.res = (flags & NPF_ADD_DY) ? dY : nullptr;   // residual-branch gradient added in the epilogue
        if (dw2_ok(H, C, kh, kw) && !dpre_scale) { rc = kw <= 9 ? launch_dw2<9>(p, B, st) : launch_dw2<11>(p, B, st); if (rc != NPF_OK) return rc; } else
        switch (kwsel) {
            case 9: rc = launch_dw<9>(p, B, st); break;
            case 11: rc = launch_dw<11>(p, B, st); break;
            default: rc = launch_dw<19>(p, B, st); break;
        }
        if (rc != NPF_OK) return rc;
    }
    if (dWt) {
        DwParams p{};
        p.X = X; p.scale = pre_scale; p.shift = pre_shift;
        p.H = H; p.Wd = Wd; p.C = C; p.kh = kh; p.kw = kw; p.relu_in = relu_in;
        if (dw2_ok(H, C, kh, kw)) { rc = kw <= 9 ? launch_dw2_wgrad<9>(p, dY, dWt, B, st) : launch_dw2_wgrad<11>(p, dY, dWt, B, st); } else
        switch (kwsel) {
            case 9: rc = launch_dw_wgrad<9>(p, dY, dWt, B, st); break;
            case 11: rc = launch_dw_wgrad<11>(p, dY, dWt, B, st); break;
            default: rc = launch_dw_wgrad<19>(p, dY, dWt, B, st); break;
        }
        if (rc != NPF_OK) return rc;
    }
    if (dbias) rc = launch_stats(dY, nullptr, dbias, nullptr, (long)B * H * Wd, C, st);
    return rc;
}

extern "C" int npf_channel_stats(const float* X, const float* center, float* sum, float* sumsq, long M, int C,
                                 npf_stream_t stream) {
    NPF_REQUIRE(X && (sum || sumsq), "npf_channel_stats: null pointer");
    NPF_REQUIRE(M >= 0 && C >= 1, "npf_channel_stats: bad shape");
    if (M == 0) return NPF_OK;
    return launch_stats(X, center, sum, sumsq, M, C, as_stream(stream));
}

extern "C" int npf_channel_affine(const float* X, const float* a, const float* b, float* Y, long M, int C, int accumulate,
                                  npf_stream_t stream) {
    NPF_REQUIRE(X && a && b && Y, "npf_channel_affine: null pointer");
    NPF_REQUIRE(M >= 0 && C >= 1, "npf_channel_affine: bad shape");
    const long n = M * C;
    if (n == 0) return NPF_OK;
    long blocks = cdiv(n, 256);
    if (blocks > 16L * kNumSMs) blocks = 16L * kNumSMs;
    channel_affine_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(X, a, b, Y, n, C, accumulate);
    count_launch();
    return check_launch("channel_affine_kernel");
}
