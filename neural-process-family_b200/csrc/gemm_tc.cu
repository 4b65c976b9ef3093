// Tensor-core path of the 128-wide linear layers: tcgen05.mma (UMMA) with the accumulator in TMEM.
//
//   NPF_PREC_BF16   : operands rounded to bf16, fp32 accumulate                        (1e-2 parity)
//   NPF_PREC_BF16X3 : x = hi + lo (both bf16); x.w ~ hi.hi + hi.lo + lo.hi, fp32 accumulate (1e-4 parity; 3 MMAs)
//
// Activations stay fp32 in HBM (layout contract of the library), so operands are converted on the fly: the CTA's
// threads load the fp32 tile with coalesced 16-byte loads, apply the prologue (relu), split/round to bf16 and write
// the UMMA canonical *no-swizzle* layout straight into shared memory (8x8 "core matrices" of 128 contiguous
// bytes; LBO = stride between core matrices along the reduction dim, SBO = along rows).  One elected thread then
// issues the K/16 MMAs (x1 or x3), commits to an mbarrier, and all 8 warps drain the 128xN fp32 accumulator from
// TMEM (tcgen05.ld 32x32b) through the bias / relu / rank-1 / relu-mask epilogue into global memory.
// The weight matrix is converted and staged ONCE per CTA (persistent over row tiles).
//
//   linear_tc_kernel : fwd  Y = act(X) W^T            (A = X rows K-major,  B = W   [N x K] K-major)
//                      bwd  dX = dY W                 (A = dY rows K-major, B = W^T [K x N], staged transposed)
//   wgrad_tc_kernel  : dW += dY^T X                   (A = dY, B = X, both MN-major: the reduction runs over rows)
//
// Shapes covered: reduction dim <= 128 and output dim <= 256, both multiples of 16.  Anything else reports
// NPF_ENOTSUP and the caller uses the fp32 FFMA kernel.
#include <cstdio>
#include "tc_common.cuh"

namespace npf {

// ------------------------------------------------------------------------------------------------ K-major staging
// Tile of R rows x KR reduction elements, element (row, k) at byte
//     (k/8) * LBO + (row/8) * 128 + (row%8) * 16 + (k%8) * 2,      LBO = R * 16
// (core matrix = 8 rows x 8 k = 128 contiguous bytes).  Source: fp32 row-major with leading dimension ld.
// A half-warp owns one core matrix per step (conflict-free 8-byte stores; 8 full 32-byte sectors per load).
// Loads are split from the convert+store so that a whole tile (16 x 16 B per thread = 64 KB per CTA) is in
// flight at once, and so that the NEXT tile can be prefetched into registers under the current tile's MMA + epilogue.
constexpr int kLinThreads = 512;            // linear_tc_kernel: 16 warps (32 half-warps stage 32 core matrices per step)
constexpr int kHW = kLinThreads / 16;
constexpr int kPre = 8;                     // float4 registers per thread per batch: 128 x 128 tile / 4 / 512 threads

__device__ __forceinline__ int ilog2(int x) { return 31 - __clz(x); }

// All tile extents on this path are powers of two (checked on the host), so the (core-matrix -> row group, k chunk)
// maps are shifts, and because 32 half-warps step through core matrices 32 at a time the k chunk of a thread is
// CONSTANT: only the row group advances -> one pointer increment and one smem-offset increment per step.
template <bool VEC>
__device__ __forceinline__ void load_kmajor(float4 (&pre)[kPre], const float* __restrict__ src, long ld, long row0, int rows_valid,
                                            int R, int KR, int cm_base) {
    const int hw = threadIdx.x >> 4, l16 = threadIdx.x & 15;
    const int r = l16 & 7, half = l16 >> 3;
    const int n_kc = KR >> 3, lg = ilog2(n_kc);
    const int cm0 = cm_base + hw;
    const int kc = cm0 & (n_kc - 1);
    int rg = cm0 >> lg;
    const int rg_step = kHW >> lg, n_rg = R >> 3;   // n_kc <= 16 divides kHW = 32
    const float* g = src + (row0 + rg * 8 + r) * ld + kc * 8 + half * 4;
    const long gstep = (long)rg_step * 8 * ld;
#pragma unroll
    for (int i = 0; i < kPre; ++i) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rg < n_rg && rg * 8 + r < rows_valid) {
            if (VEC) v = __ldg(reinterpret_cast<const float4*>(g));
            else { v.x = __ldg(g); v.y = __ldg(g + 1); v.z = __ldg(g + 2); v.w = __ldg(g + 3); }
        }
        pre[i] = v;
        rg += rg_step;
        g += gstep;
    }
}

template <int NSPLIT>
__device__ __forceinline__ void store_kmajor(const float4 (&pre)[kPre], uint8_t* hi, uint8_t* lo, int R, int KR, int cm_base, int relu) {
    const int hw = threadIdx.x >> 4, l16 = threadIdx.x & 15;
    const int r = l16 & 7, half = l16 >> 3;
    const int n_kc = KR >> 3, lg = ilog2(n_kc);
    const int cm0 = cm_base + hw;
    const int kc = cm0 & (n_kc - 1);
    int rg = cm0 >> lg;
    const int rg_step = kHW >> lg, n_rg = R >> 3;
    uint32_t off = (uint32_t)kc * ((uint32_t)R * 16u) + (uint32_t)rg * 128u + (uint32_t)r * 16u + (uint32_t)half * 8u;
#pragma unroll
    for (int i = 0; i < kPre; ++i) {
        if (rg < n_rg) {
            float4 v = pre[i];
            if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
            const uint32_t h01 = pack_bf16(v.x, v.y), h23 = pack_bf16(v.z, v.w);
            *reinterpret_cast<uint2*>(hi + off) = make_uint2(h01, h23);
            if (NSPLIT == 3) {   // residuals against the packed hi halves (bf16 -> fp32 is a 16-bit shift)
                const float rx = v.x - __uint_as_float(h01 << 16), ry = v.y - __uint_as_float(h01 & 0xFFFF0000u);
                const float rz = v.z - __uint_as_float(h23 << 16), rw = v.w - __uint_as_float(h23 & 0xFFFF0000u);
                *reinterpret_cast<uint2*>(lo + off) = make_uint2(pack_bf16(rx, ry), pack_bf16(rz, rw));
            }
        }
        rg += rg_step;
        off += (uint32_t)rg_step * 128u;
    }
}

// Transposed staging of the weights for the data gradient: B'(row = k_out, red = n) = W[n, k_out], K-major in n.
// Batched float4 loads along k_out (coalesced rows of W), four 2-byte scatter stores each (once per CTA).
template <int NSPLIT>
__device__ __forceinline__ void stage_kmajor_transposed(uint8_t* hi, uint8_t* lo, const float* __restrict__ W, long ldw, int R /*rows = K_out*/,
                                                        int KR /*reduction = N*/, int vec_ok) {
    const uint32_t lbo = (uint32_t)R * 16u;
    const int rq = R >> 2, lgq = ilog2(rq), total = rq * KR;      // float4 count; rq is a power of two <= 64
    const int row0 = (threadIdx.x & (rq - 1)) * 4;                // constant per thread (512 is a multiple of rq)
    for (int base = 0; base < total; base += kLinThreads * kPre) {
        float4 pre[kPre];
        const int n0 = (base + threadIdx.x) >> lgq, n_step = kLinThreads >> lgq;
#pragma unroll
        for (int i = 0; i < kPre; ++i) {
            const int n = n0 + i * n_step;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n < KR) {
                const float* g = W + (long)n * ldw + row0;
                if (vec_ok) v = __ldg(reinterpret_cast<const float4*>(g));
                else { v.x = __ldg(g); v.y = __ldg(g + 1); v.z = __ldg(g + 2); v.w = __ldg(g + 3); }
            }
            pre[i] = v;
        }
#pragma unroll
        for (int i = 0; i < kPre; ++i) {
            const int n = n0 + i * n_step;
            if (n >= KR) continue;
            const float vv[4] = {pre[i].x, pre[i].y, pre[i].z, pre[i].w};
            const uint32_t off0 = (uint32_t)(n >> 3) * lbo + (uint32_t)(row0 >> 3) * 128u + (uint32_t)(row0 & 7) * 16u + (uint32_t)(n & 7) * 2u;
#pragma unroll
            for (int e = 0; e < 4; ++e) {      // rows row0 .. row0+3 stay inside one 8-row group (row0 is a multiple of 4)
                const uint32_t off = off0 + (uint32_t)e * 16u;
                const __nv_bfloat16 h = __float2bfloat16_rn(vv[e]);
                *reinterpret_cast<__nv_bfloat16*>(hi + off) = h;
                if (NSPLIT == 3) *reinterpret_cast<__nv_bfloat16*>(lo + off) = __float2bfloat16_rn(vv[e] - __bfloat162float(h));
            }
        }
    }
}

struct TcLinParams {
    const float* A; long lda;       // [M, KR] activations (X or dY)
    const float* W; long ldw;       // fwd: [NO, KR]; bwd-data: [KR, NO]
    float* C; long ldc;             // [M, NO]
    const float* bias;              // [NO] or null
    const float* u; const float* w2; long ldw2;   // rank-1 epilogue
    const float* mask; long ldm;    // relu mask source [M, NO]
    int M, KR, NO;
    int relu_in, relu_out, transposed_w, a_vec, w_vec, c_vec;
    int n_tiles;
    int rows_per_cta;   // linear_ws_kernel: contiguous row range per CTA (multiple of 8)
};

// ------------------------------------------------------------------------------------------------ fwd / bwd-data
constexpr int kScratchLd = 36;     // floats per staged row: 32 + 4 keeps both the row-wise STS.128 and the LDS.128 conflict-free

// KR_T / NO_T: compile-time reduction / output extents (0 = run-time values from the parameter block); HAS_U / HAS_MASK:
// rank-1 epilogue term / relu-mask epilogue compiled in.  The 128 x 128 instantiations are the hot ones: with the
// extents known every staging predicate and index computation folds away.
template <int NSPLIT, int KR_T, int NO_T, bool HAS_U, bool HAS_MASK, bool VEC>
__global__ void __launch_bounds__(kLinThreads, 1) linear_tc_kernel(TcLinParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t mma_bar;
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float s_bias[256], s_w2[256];

    const int KR = KR_T ? KR_T : p.KR, NO = NO_T ? NO_T : p.NO;
    const uint32_t a_bytes = 128u * KR * 2u, b_bytes = (uint32_t)NO * KR * 2u;
    uint8_t* a_hi = smem_raw;
    uint8_t* a_lo = a_hi + a_bytes;                               // only touched when NSPLIT == 3
    uint8_t* b_hi = smem_raw + (NSPLIT == 3 ? 2 : 1) * a_bytes;
    uint8_t* b_lo = b_hi + b_bytes;
    float* scratch_all = reinterpret_cast<float*>(smem_raw + (NSPLIT == 3 ? 2 : 1) * (a_bytes + b_bytes));

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float* scratch = scratch_all + warp * (32 * kScratchLd);
    const uint32_t ncols = NO <= 32 ? 32u : (NO <= 64 ? 64u : (NO <= 128 ? 128u : 256u));
    if (warp == 0) tmem_alloc(&tmem_slot, ncols);
    if (tid == 0) mbar_init(&mma_bar, 1);
    for (int c = tid; c < 256; c += kLinThreads) {
        s_bias[c] = (p.bias && c < NO) ? __ldg(p.bias + c) : 0.f;
        s_w2[c] = (p.w2 && c < NO) ? __ldg(p.w2 + (long)c * p.ldw2) : 0.f;
    }

    float4 pre[kPre];
    int tile = blockIdx.x;
    // first activation tile: in flight while the weights are staged
    if (tile < p.n_tiles) load_kmajor<VEC>(pre, p.A, p.lda, (long)tile * 128, min(128, p.M - tile * 128), 128, KR, 0);
    // weights: converted and staged once per CTA
    if (p.transposed_w) {
        stage_kmajor_transposed<NSPLIT>(b_hi, b_lo, p.W, p.ldw, NO, KR, p.w_vec);
    } else {
        const int n_cm = (NO >> 3) * (KR >> 3);
        for (int base = 0; base < n_cm; base += kHW * kPre) {
            float4 wpre[kPre];
            if (p.w_vec) load_kmajor<true>(wpre, p.W, p.ldw, 0, NO, NO, KR, base);
            else load_kmajor<false>(wpre, p.W, p.ldw, 0, NO, NO, KR, base);
            store_kmajor<NSPLIT>(wpre, b_hi, b_lo, NO, KR, base, 0);
        }
    }
    if (tile < p.n_tiles) store_kmajor<NSPLIT>(pre, a_hi, a_lo, 128, KR, 0, p.relu_in);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t idesc = make_idesc(128, NO, 0, 0);
    const uint32_t a_lbo = 128u * 16u, b_lbo = (uint32_t)NO * 16u;

    // epilogue geometry: warp w drains TMEM lanes 32*(w&3)..+31 (its 32 rows) for the column chunks w>>2, w>>2 + 4, ...
    const int CW = NO < 32 ? NO : 32;            // chunk width (16 or 32 columns)
    const int n_chunks = NO / CW;
    const int lane_base = 32 * (warp & 3);
    const int qpr = CW >> 2, rpi = 32 / qpr;     // float4 per staged row, rows per coalesced instruction
    const int r_in = lane / qpr, c4 = (lane % qpr) * 4;

    uint32_t phase = 0;
    for (; tile < p.n_tiles; tile += gridDim.x) {
        const int m0 = tile * 128;
        if (tid == 0) {
            const uint32_t sa_hi = smem_u32(a_hi), sa_lo = smem_u32(a_lo), sb_hi = smem_u32(b_hi), sb_lo = smem_u32(b_lo);
            uint32_t acc = 0;
            for (int ks = 0; ks < KR / 16; ++ks) {
                const uint32_t ao = (uint32_t)ks * 2u * a_lbo, bo = (uint32_t)ks * 2u * b_lbo;
                umma_bf16(tmem, make_desc(sa_hi + ao, a_lbo, 128), make_desc(sb_hi + bo, b_lbo, 128), idesc, acc);
                acc = 1;
                if (NSPLIT == 3) {
                    umma_bf16(tmem, make_desc(sa_hi + ao, a_lbo, 128), make_desc(sb_lo + bo, b_lbo, 128), idesc, 1);
                    umma_bf16(tmem, make_desc(sa_lo + ao, a_lbo, 128), make_desc(sb_hi + bo, b_lbo, 128), idesc, 1);
                }
            }
            umma_commit(&mma_bar);   // implies tcgen05.fence::before_thread_sync
        }
        // prefetch the next tile into registers: in flight under this tile's MMA and epilogue
        const int next = tile + gridDim.x;
        if (next < p.n_tiles) load_kmajor<VEC>(pre, p.A, p.lda, (long)next * 128, min(128, p.M - next * 128), 128, KR, 0);

        mbar_wait(&mma_bar, phase);
        phase ^= 1;
        tc_fence_after();

        for (int ch = warp >> 2; ch < n_chunks; ch += 4) {
            const int c0 = ch * CW;
            // TMEM -> registers (thread = row) -> per-warp smem tile
            if (CW == 32) {
                float v[32];
                tmem_ld32(tmem + ((uint32_t)lane_base << 16) + (uint32_t)c0, v);
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4*>(scratch + lane * kScratchLd + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            } else {
                float v[16];
                tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)c0, v);
#pragma unroll
                for (int j = 0; j < 16; j += 4)
                    *reinterpret_cast<float4*>(scratch + lane * kScratchLd + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            }
            __syncwarp();
            // smem -> global, row-contiguous: a warp instruction covers `rpi` rows x CW columns (full 32-byte sectors)
            const float4 bb = *reinterpret_cast<const float4*>(&s_bias[c0 + c4]);
            const float4 ww = *reinterpret_cast<const float4*>(&s_w2[c0 + c4]);
            for (int r0 = 0; r0 < 32; r0 += rpi) {
                const int r = r0 + r_in;
                const int row = m0 + lane_base + r;
                if (row < p.M) {
                    float4 x = *reinterpret_cast<const float4*>(scratch + r * kScratchLd + c4);
                    x.x += bb.x; x.y += bb.y; x.z += bb.z; x.w += bb.w;
                    if (HAS_U && p.u) {
                        const float up = __ldg(p.u + row);
                        x.x = fmaf(up, ww.x, x.x); x.y = fmaf(up, ww.y, x.y); x.z = fmaf(up, ww.z, x.z); x.w = fmaf(up, ww.w, x.w);
                    }
                    if (p.relu_out) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
                    if (HAS_MASK && p.mask) {
                        const float* mk = p.mask + (long)row * p.ldm + c0 + c4;
                        float4 mv;
                        if (VEC) mv = __ldg(reinterpret_cast<const float4*>(mk));
                        else mv = make_float4(__ldg(mk), __ldg(mk + 1), __ldg(mk + 2), __ldg(mk + 3));
                        x.x = mv.x > 0.f ? x.x : 0.f; x.y = mv.y > 0.f ? x.y : 0.f; x.z = mv.z > 0.f ? x.z : 0.f; x.w = mv.w > 0.f ? x.w : 0.f;
                    }
                    float* out = p.C + (long)row * p.ldc + c0 + c4;
                    if (VEC) *reinterpret_cast<float4*>(out) = x;
                    else { out[0] = x.x; out[1] = x.y; out[2] = x.z; out[3] = x.w; }
                }
            }
            __syncwarp();
        }
        tc_fence_before();   // TMEM reads done (and the MMAs have consumed the A buffer) before it is overwritten
        __syncthreads();
        if (next < p.n_tiles) {
            store_kmajor<NSPLIT>(pre, a_hi, a_lo, 128, KR, 0, p.relu_in);
            fence_async_smem();   // generic-proxy smem writes -> visible to the tensor core (async proxy)
        }
        __syncthreads();
        tc_fence_after();
    }
    if (warp == 0) tmem_dealloc(tmem, ncols);
}

// ------------------------------------------------------------------------------------------------ warp-specialised 128 x 128 x 128
// The hot shape (reduction 128, output 128, 16-byte aligned rows) runs as a three-role pipeline, one persistent CTA per SM:
//   warps 0..7  producers : fp32 tile -> registers (16 x LDG.128 per thread in flight) -> bf16 hi/lo -> smem stage s  -> full[s]
//   warp  8     MMA       : waits full[s] + tempty[t], issues 8 (x3) tcgen05.mma into accumulator t, commits -> empty[s], tfull[t]
//   warps 9..16 epilogue  : waits tfull[t], tcgen05.ld -> per-warp smem transpose -> bias / rank-1 / relu / mask -> coalesced STG
// Two smem operand stages and two TMEM accumulators (2 x 128 columns): tile i+1 is loaded and converted while tile i is
// multiplied and tile i-1 is drained, so the HBM stream never waits on the math.  The weights are staged once per CTA in the
// row layout of W; the data gradient reads the very same staging through an MN-major descriptor (transpose for free).
constexpr int kWsProdWarps = 16;
constexpr int kWsEpiWarp0 = 17;
constexpr int kWsEpiWarps = 8;
constexpr int kWsThreads = (kWsEpiWarp0 + kWsEpiWarps) * 32;     // 800
constexpr int kWsPre = 8;                                        // float4 per producer thread per tile
constexpr int kWsScratchLd = 20;                                 // 16 columns + 4 pad (conflict-free STS.128)

template <int NSPLIT>
__device__ __forceinline__ void cvt_store(const float4& vin, uint8_t* hi, uint8_t* lo, uint32_t off, int relu) {
    float4 v = vin;
    if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
    const uint32_t h01 = pack_bf16(v.x, v.y), h23 = pack_bf16(v.z, v.w);
    *reinterpret_cast<uint2*>(hi + off) = make_uint2(h01, h23);
    if (NSPLIT == 3) {
        const float rx = v.x - __uint_as_float(h01 << 16), ry = v.y - __uint_as_float(h01 & 0xFFFF0000u);
        const float rz = v.z - __uint_as_float(h23 << 16), rw = v.w - __uint_as_float(h23 & 0xFFFF0000u);
        *reinterpret_cast<uint2*>(lo + off) = make_uint2(pack_bf16(rx, ry), pack_bf16(rz, rw));
    }
}

// producer-side tile load: thread (kc = tid/16, r = tid%8, half) owns the 16 bytes (row 8i + r, k = 8 kc + 4 half) of every
// 8-row group i -> per instruction a half-warp covers 8 rows x 32 bytes (full sectors) and stores one 128-byte core matrix
__device__ __forceinline__ void ws_load_tile(float4 (&pre)[kWsPre], const float* __restrict__ g, long ld, int r, int rows_valid) {
#pragma unroll
    for (int i = 0; i < kWsPre; ++i) {
        pre[i] = (i * 8 + r < rows_valid) ? __ldg(reinterpret_cast<const float4*>(g)) : make_float4(0.f, 0.f, 0.f, 0.f);
        g += 8 * ld;
    }
}

// SWIZZLE_128B K-major staging of a [128 rows x 128 k] bf16 operand: two atoms of 64 k (128 bytes per row, 16 KB per atom),
//     byte(row, k) = (k / 64) * 16384 + row * 128 + ((((k % 64) / 8) ^ (row % 8)) * 16) + (k % 8) * 2
// (the 16-byte chunk index XOR-ed with the row index: what the tensor core undoes in hardware; atoms 1024-byte aligned).
// Read K-major: start + atom * 16384 + (ks % 4) * 32, SBO = 1024 (8-row groups).  The same bytes read MN-major are the
// transpose: mn = k (two 64-wide atoms, LBO = 16384), reduction = row (8-row groups, SBO = 1024), start + ks * 2048.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return make_desc(saddr, lbo_bytes, sbo_bytes) | (2ull << 61);
}
// producer mapping (SW128): warp w owns rows 16 w .. 16 w + 15; per row the 32 lanes load the 512 contiguous bytes
// (one LDG.128 each) and store 8 bytes of hi and of lo: per instruction 2 x 128 contiguous (permuted) bytes -> no conflicts
__device__ __forceinline__ void ws_load_rows(float4 (&pre)[kWsPre], const float* __restrict__ g, long ld, int row_first, int rows_valid) {
#pragma unroll
    for (int i = 0; i < kWsPre; ++i) {
        pre[i] = (row_first + i < rows_valid) ? __ldg(reinterpret_cast<const float4*>(g)) : make_float4(0.f, 0.f, 0.f, 0.f);
        g += ld;
    }
}

// L2 prefetch of a 128-row x 512-byte tile (512 lines of 128 bytes) by `nthreads` threads: the tile AFTER the one whose loads
// were just issued.  DRAM latency under load (~4 us) then overlaps two tile periods and the register-staged loads of the next
// iteration hit L2, without spending registers or shared memory on a deeper ring.
__device__ __forceinline__ void prefetch_tile_l2(const float* __restrict__ base, long ld, long row0, int rows_valid, int t, int nthreads) {
    for (int l = t; l < 512; l += nthreads) {
        const int r = l >> 2;
        if (r < rows_valid) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (row0 + r) * ld + (l & 3) * 32));
    }
}

template <int NSPLIT, bool HAS_U, bool HAS_MASK, bool SW>
__global__ void __launch_bounds__(kWsThreads, 1) linear_ws_kernel(TcLinParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[2], bar_empty[2], bar_tfull[2], bar_tempty[2];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float s_bias[128], s_w2[128];

    constexpr uint32_t kTile = 128u * 128u * 2u;                 // one bf16 128 x 128 operand: 32 KB
    constexpr uint32_t kStage = (NSPLIT == 3 ? 2u : 1u) * kTile;
    uint8_t* b_hi = smem_raw + 2 * kStage;
    uint8_t* b_lo = b_hi + kTile;
    float* scratch_all = reinterpret_cast<float*>(smem_raw + 3 * kStage);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    if (tid == 32) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_full[i], kWsProdWarps * 32);
            mbar_init(&bar_empty[i], 1);
            mbar_init(&bar_tfull[i], 1);
            mbar_init(&bar_tempty[i], kWsEpiWarps * 32);
        }
    }
    if (tid < 128) {
        s_bias[tid] = p.bias ? __ldg(p.bias + tid) : 0.f;
        s_w2[tid] = (HAS_U && p.w2) ? __ldg(p.w2 + (long)tid * p.ldw2) : 0.f;
    }

    static_assert(SW, "the warp-specialised kernel stages SWIZZLE_128B operands");
    // producer geometry (also used for the weight staging below): warp w owns rows 8 w .. 8 w + 7 of a 128-row tile; per row
    // the 32 lanes load the 512 contiguous bytes (one LDG.128 each) and store 8 bytes of hi and of lo.  SIXTEEN producer warps
    // with 8 loads each rather than 8 x 16: at equal bytes in flight a streaming kernel on this part gets 5.7 vs 4.7 TB/s
    // (profiles/microbench/stream_probe.cu) -- the memory pipe wants warps, not deep per-warp queues.
    // balanced contiguous row ranges: every CTA gets M / gridDim rows (8-row granularity) = whole 128-row tiles + one partial
    // tile, instead of 128-row tiles dealt round-robin (768 tiles over 148 SMs would cost 6 rounds for 5.2 tiles of work)
    const int r_begin = blockIdx.x * p.rows_per_cta, r_end = min(p.M, r_begin + p.rows_per_cta);
    const int n_local = r_end > r_begin ? (r_end - r_begin + 127) >> 7 : 0;
    const uint32_t pchunk = (uint32_t)(lane >> 1) & 7u;
    const uint32_t psoff = (uint32_t)(lane >> 4) * 16384u + (uint32_t)(warp * 8) * 128u + (uint32_t)(lane & 1) * 8u;
    pdl_trigger();      // the next kernel may start its own parameter-only prologue as SMs free up

    // weights [128 x 128] fp32 row-major, staged once per CTA by the 16 producer warps in the layout of the A tiles
    if (warp < kWsProdWarps) {
        float4 wv[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float* g = p.W + (long)(warp * 8 + i) * p.ldw + lane * 4;
            if (p.w_vec) wv[i] = __ldg(reinterpret_cast<const float4*>(g));
            else wv[i] = make_float4(__ldg(g), __ldg(g + 1), __ldg(g + 2), __ldg(g + 3));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) cvt_store<NSPLIT>(wv[i], b_hi, b_lo, psoff + (uint32_t)i * 128u + ((pchunk ^ (uint32_t)i) << 4), 0);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    // everything above touched parameters only (weights, bias); activations of the preceding kernel from here on
    pdl_wait();

    if (warp < kWsProdWarps) {
        // ------------------------------------------------------------------ producers
        const float* pg = p.A + (long)(warp * 8) * p.lda + lane * 4;
        float4 pre[kWsPre];
        if (n_local > 0) {
            ws_load_rows(pre, pg + (long)r_begin * p.lda, p.lda, warp * 8, min(128, r_end - r_begin));
            if (n_local > 1) prefetch_tile_l2(p.A, p.lda, (long)r_begin + 128, min(128, r_end - r_begin - 128), tid, kWsProdWarps * 32);
        }
        for (int it = 0; it < n_local; ++it) {
            const int s = it & 1;
            mbar_wait(&bar_empty[s], ((it >> 1) & 1) ^ 1);
            uint8_t* hi = smem_raw + s * kStage;
            uint8_t* lo = hi + kTile;
#pragma unroll
            for (int i = 0; i < kWsPre; ++i) cvt_store<NSPLIT>(pre[i], hi, lo, psoff + (uint32_t)i * 128u + ((pchunk ^ (uint32_t)i) << 4), p.relu_in);
            fence_async_smem();
            mbar_arrive(&bar_full[s]);
            if (it + 1 < n_local) {
                const int nrow = r_begin + (it + 1) * 128;
                ws_load_rows(pre, pg + (long)nrow * p.lda, p.lda, warp * 8, min(128, r_end - nrow));
                if (it + 2 < n_local) prefetch_tile_l2(p.A, p.lda, (long)nrow + 128, min(128, r_end - nrow - 128), tid, kWsProdWarps * 32);
            }
        }
    } else if (warp == kWsProdWarps) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc(128, 128, 0, p.transposed_w ? 1 : 0);
            const uint32_t sb_hi = smem_u32(b_hi), sb_lo = smem_u32(b_lo);
            // fwd: B = W rows (n) K-major in k.  bwd-data: B = W^T, i.e. the same bytes read MN-major (mn = k_out, red = n)
            const uint32_t b_step = p.transposed_w ? 256u : 4096u, b_lbo = p.transposed_w ? 128u : 2048u, b_sbo = p.transposed_w ? 2048u : 128u;
            for (int it = 0; it < n_local; ++it) {
                const int s = it & 1;
                const uint32_t par = (it >> 1) & 1;
                mbar_wait(&bar_full[s], par);
                mbar_wait(&bar_tempty[s], par ^ 1);
                tc_fence_after();
                const uint32_t sa_hi = smem_u32(smem_raw + s * kStage), sa_lo = sa_hi + kTile;
                const uint32_t d = tmem + (uint32_t)s * 128u;
                const uint64_t da_h = make_desc_sw128(sa_hi, 16, 1024), da_l = make_desc_sw128(sa_lo, 16, 1024);
                const uint64_t db_h = p.transposed_w ? make_desc_sw128(sb_hi, 16384, 1024) : make_desc_sw128(sb_hi, 16, 1024);
                const uint64_t db_l = p.transposed_w ? make_desc_sw128(sb_lo, 16384, 1024) : make_desc_sw128(sb_lo, 16, 1024);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks) {
                    uint64_t a_h, a_l, b_h, b_l;
                    if (SW) {
                        const uint32_t ao = (uint32_t)(ks >> 2) * 16384u + (uint32_t)(ks & 3) * 32u;
                        a_h = desc_adv(da_h, ao);
                        a_l = desc_adv(da_l, ao);
                        b_h = desc_adv(db_h, p.transposed_w ? ks * 2048u : ao);
                        b_l = desc_adv(db_l, p.transposed_w ? ks * 2048u : ao);
                    } else {
                        a_h = make_desc(sa_hi + ks * 4096u, 2048, 128);
                        a_l = make_desc(sa_lo + ks * 4096u, 2048, 128);
                        b_h = make_desc(sb_hi + ks * b_step, b_lbo, b_sbo);
                        b_l = make_desc(sb_lo + ks * b_step, b_lbo, b_sbo);
                    }
                    umma_bf16(d, a_h, b_h, idesc, ks ? 1u : 0u);
                    if (NSPLIT == 3) {
                        umma_bf16(d, a_h, b_l, idesc, 1);
                        umma_bf16(d, a_l, b_h, idesc, 1);
                    }
                }
                umma_commit(&bar_empty[s]);      // operand stage s free once these MMAs retire
                umma_commit(&bar_tfull[s]);      // accumulator s complete
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue
        const int e = warp - kWsEpiWarp0;
        const int lane_base = 32 * (warp & 3);                    // the TMEM lane quadrant this warp may read
        const int col_base = (e >> 2) * 64;                       // two warps per quadrant: 64 columns each, 4 chunks of 16
        float* scratch = scratch_all + e * (32 * kWsScratchLd);
        const int r_in = lane >> 2, c4 = (lane & 3) * 4;          // store geometry: 8 rows x 64 bytes per instruction
        for (int it = 0; it < n_local; ++it) {
            const int s = it & 1;
            const int m0 = r_begin + it * 128 + lane_base;
            float4 mk[4];
            if (HAS_MASK) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int row = m0 + j * 8 + r_in;
                    mk[j] = row < r_end ? __ldg(reinterpret_cast<const float4*>(p.mask + (long)row * p.ldm + col_base + c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            mbar_wait(&bar_tfull[s], (it >> 1) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int ch = 0; ch < 4; ++ch) {
                const int c0 = col_base + ch * 16;
                float v[16];
                tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(s * 128 + c0), v);
                if (ch == 3) {                                     // accumulator drained: hand it back before the stores
                    tc_fence_before();
                    mbar_arrive(&bar_tempty[s]);
                }
#pragma unroll
                for (int j = 0; j < 16; j += 4)
                    *reinterpret_cast<float4*>(scratch + lane * kWsScratchLd + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                __syncwarp();
                float4 mn[4];
                if (HAS_MASK && ch < 3) {                          // next chunk's mask in flight under this chunk's stores
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int row = m0 + j * 8 + r_in;
                        mn[j] = row < r_end ? __ldg(reinterpret_cast<const float4*>(p.mask + (long)row * p.ldm + c0 + 16 + c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                const float4 bb = *reinterpret_cast<const float4*>(&s_bias[c0 + c4]);
                const float4 ww = *reinterpret_cast<const float4*>(&s_w2[c0 + c4]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int r = j * 8 + r_in;
                    const int row = m0 + r;
                    if (row < r_end) {
                        float4 x = *reinterpret_cast<const float4*>(scratch + r * kWsScratchLd + c4);
                        x.x += bb.x; x.y += bb.y; x.z += bb.z; x.w += bb.w;
                        if (HAS_U) {
                            const float up = __ldg(p.u + row);
                            x.x = fmaf(up, ww.x, x.x); x.y = fmaf(up, ww.y, x.y); x.z = fmaf(up, ww.z, x.z); x.w = fmaf(up, ww.w, x.w);
                        }
                        if (p.relu_out) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
                        if (HAS_MASK) {
                            x.x = mk[j].x > 0.f ? x.x : 0.f; x.y = mk[j].y > 0.f ? x.y : 0.f;
                            x.z = mk[j].z > 0.f ? x.z : 0.f; x.w = mk[j].w > 0.f ? x.w : 0.f;
                        }
                        *reinterpret_cast<float4*>(p.C + (long)row * p.ldc + c0 + c4) = x;
                    }
                }
                if (HAS_MASK && ch < 3) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) mk[j] = mn[j];
                }
                __syncwarp();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------------------------------------ MLP chain forward (128-wide)
// L consecutive Linear(128 -> 128) [+ ReLU] layers for a row block that stays ON CHIP between layers: a CTA owns up to 256
// rows (two 128-row tiles); layer l's output leaves the tensor core through TMEM, gets its bias / ReLU in the epilogue, is
// written once to HBM as the saved activation Y_l AND re-split into bf16 hi / lo straight into the shared-memory A-operand
// image of layer l+1.  Against one kernel per layer this removes the read of every intermediate activation, L - 1 launches
// with their parameter prologues and pipeline fill / drain -- the per-layer kernels of the 32 768-row decoder MLP spend
// most of their 15 us there (1.7 tiles per SM).  Roles: 16 stager warps (X rows at the start, then W_l per layer, prefetched
// into registers while layer l-1 is multiplied), 1 MMA warp, 8 epilogue warps.
constexpr int kChainMaxLayers = 8;
constexpr int kChainRows = 256;
struct ChainParams {
    const float* X; long ldx;
    const float* W[kChainMaxLayers]; long ldw[kChainMaxLayers];
    const float* b[kChainMaxLayers];
    float* Y[kChainMaxLayers]; long ldy[kChainMaxLayers];
    int L, M, rows_per_cta, relu_in;
    unsigned relu_mask;          // bit l: ReLU after layer l
};

template <int NSPLIT>
__global__ void __launch_bounds__(kWsThreads, 1) mlp_chain_fwd_kernel(ChainParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_wfull, bar_wfree, bar_xready[2], bar_aready[2], bar_drained[2], bar_mma[2];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float s_bias[kChainMaxLayers][128];     // all layers' biases (parameters), staged once

    constexpr uint32_t kTile = 128u * 128u * 2u;                   // one bf16 128 x 128 image: 32 KB
    constexpr uint32_t kImg = (NSPLIT == 3 ? 2u : 1u) * kTile;     // hi [+ lo]
    uint8_t* w_hi = smem_raw + 2 * kImg;
    uint8_t* w_lo = w_hi + kTile;
    float* scratch_all = reinterpret_cast<float*>(smem_raw + 3 * kImg);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    if (tid == 32) {
        mbar_init(&bar_wfull, kWsProdWarps * 32);
        mbar_init(&bar_wfree, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_xready[i], kWsProdWarps * 32);
            mbar_init(&bar_aready[i], kWsEpiWarps * 32);
            mbar_init(&bar_drained[i], kWsEpiWarps * 32);
            mbar_init(&bar_mma[i], 1);
        }
    }
    // row blocks of rows_per_cta (<= 256) rows: block k of this CTA is blockIdx.x + k gridDim.x; `it` counts (block, layer) pairs
    const int n_blocks = (p.M + p.rows_per_cta - 1) / p.rows_per_cta;
    const int L = p.L;
    const uint32_t pchunk = (uint32_t)(lane >> 1) & 7u;
    for (int i = tid; i < L * 128; i += kWsThreads) s_bias[i >> 7][i & 127] = p.b[i >> 7] ? __ldg(p.b[i >> 7] + (i & 127)) : 0.f;
    pdl_trigger();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;

    if (warp < kWsProdWarps) {
        // ------------------------------------------------------------------ stagers: warp w owns rows 8 w .. 8 w + 7 of a 128-row image
        const uint32_t psoff = (uint32_t)(lane >> 4) * 16384u + (uint32_t)(warp * 8) * 128u + (uint32_t)(lane & 1) * 8u;
        float4 pre[kWsPre];
        auto load_w = [&](int l) {
#pragma unroll
            for (int i = 0; i < kWsPre; ++i) pre[i] = __ldg(reinterpret_cast<const float4*>(p.W[l] + (long)(warp * 8 + i) * p.ldw[l]) + lane);
        };
        auto store_w = [&]() {
#pragma unroll
            for (int i = 0; i < kWsPre; ++i) cvt_store<NSPLIT>(pre[i], w_hi, w_lo, psoff + (uint32_t)i * 128u + ((pchunk ^ (uint32_t)(i & 7)) << 4), 0);
            fence_async_smem();
            mbar_arrive(&bar_wfull);
        };
        int it = 0;
        for (int blk = blockIdx.x, bi = 0; blk < n_blocks; blk += gridDim.x, ++bi) {
            const int r_begin = blk * p.rows_per_cta, r_end = min(p.M, r_begin + p.rows_per_cta);
            const int n_tiles = (r_end - r_begin + 127) >> 7;
            load_w(0);                                               // weights are parameters: may be read before the predecessor kernel is done
            if (it > 0) mbar_wait(&bar_wfree, (it - 1) & 1);         // last layer of the previous block has read W and both images
            store_w();
            if (bi == 0) pdl_wait();
            for (int t = 0; t < n_tiles; ++t) {                      // the block's input rows -> A images
                const int row0 = r_begin + t * 128;
                ws_load_rows(pre, p.X + ((long)row0 + warp * 8) * p.ldx + lane * 4, p.ldx, warp * 8, min(128, r_end - row0));
                uint8_t* hi = smem_raw + t * kImg;
#pragma unroll
                for (int i = 0; i < kWsPre; ++i) cvt_store<NSPLIT>(pre[i], hi, hi + kTile, psoff + (uint32_t)i * 128u + ((pchunk ^ (uint32_t)(i & 7)) << 4), p.relu_in);
                fence_async_smem();
                mbar_arrive(&bar_xready[t]);
            }
            ++it;
            for (int l = 1; l < L; ++l, ++it) {
                load_w(l);                                           // in flight while layer l-1 is multiplied
                mbar_wait(&bar_wfree, (it - 1) & 1);                 // the MMAs of layer l-1 have read the weight buffer
                store_w();
            }
        }
    } else if (warp == kWsProdWarps) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc(128, 128, 0, 0);
            const uint32_t sb_hi = smem_u32(w_hi), sb_lo = smem_u32(w_lo);
            int it = 0;
            for (int blk = blockIdx.x, bi = 0; blk < n_blocks; blk += gridDim.x, ++bi) {
                const int r_begin = blk * p.rows_per_cta, r_end = min(p.M, r_begin + p.rows_per_cta);
                const int n_tiles = (r_end - r_begin + 127) >> 7;
                for (int l = 0; l < L; ++l, ++it) {
                    mbar_wait(&bar_wfull, it & 1);
                    for (int t = 0; t < n_tiles; ++t) {
                        if (l == 0) {
                            mbar_wait(&bar_xready[t], bi & 1);
                            if (bi > 0) mbar_wait(&bar_drained[t], (bi - 1) & 1);                     // previous block's last accumulator read out
                        } else {
                            mbar_wait(&bar_aready[t], (bi * (L - 1) + l - 1) & 1);                    // image rewritten and TMEM drained by layer l-1's epilogue
                        }
                        tc_fence_after();
                        const uint32_t sa_hi = smem_u32(smem_raw + t * kImg), sa_lo = sa_hi + kTile;
                        const uint64_t da_h = make_desc_sw128(sa_hi, 16, 1024), da_l = make_desc_sw128(sa_lo, 16, 1024);
                        const uint64_t db_h = make_desc_sw128(sb_hi, 16, 1024), db_l = make_desc_sw128(sb_lo, 16, 1024);
                        const uint32_t d = tmem + (uint32_t)t * 128u;
#pragma unroll
                        for (int ks = 0; ks < 8; ++ks) {
                            const uint32_t ao = (uint32_t)(ks >> 2) * 16384u + (uint32_t)(ks & 3) * 32u;
                            const uint64_t a_h = desc_adv(da_h, ao), b_h = desc_adv(db_h, ao);
                            umma_bf16(d, a_h, b_h, idesc, ks ? 1u : 0u);
                            if (NSPLIT == 3) {
                                umma_bf16(d, a_h, desc_adv(db_l, ao), idesc, 1);
                                umma_bf16(d, desc_adv(da_l, ao), b_h, idesc, 1);
                            }
                        }
                        umma_commit(&bar_mma[t]);
                    }
                    umma_commit(&bar_wfree);
                }
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue: 8 warps, tile after tile
        const int e = warp - kWsEpiWarp0;
        const int lane_base = 32 * (warp & 3);
        const int col_base = (e >> 2) * 64;
        float* scratch = scratch_all + e * (32 * kWsScratchLd);
        const int r_in = lane >> 2, c4 = (lane & 3) * 4;
        const int row_img = lane_base + lane;                        // this thread's row of the image (TMEM lane)
        pdl_wait();
        int it = 0;
        for (int blk = blockIdx.x, bi = 0; blk < n_blocks; blk += gridDim.x, ++bi) {
            const int r_begin = blk * p.rows_per_cta, r_end = min(p.M, r_begin + p.rows_per_cta);
            const int n_tiles = (r_end - r_begin + 127) >> 7;
            for (int l = 0; l < L; ++l, ++it) {
                const bool relu = (p.relu_mask >> l) & 1u;
                const bool feed = l + 1 < L;
                for (int t = 0; t < n_tiles; ++t) {
                    const int m0 = r_begin + t * 128 + lane_base;
                    mbar_wait(&bar_mma[t], it & 1);
                    tc_fence_after();
                    uint8_t* img_hi = smem_raw + t * kImg;
#pragma unroll 1
                    for (int ch = 0; ch < 4; ++ch) {
                        const int c0 = col_base + ch * 16;
                        float v[16];
                        tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(t * 128 + c0), v);
                        if (!feed && ch == 3) {                      // last layer: the accumulator may be reused by the next block
                            tc_fence_before();
                            mbar_arrive(&bar_drained[t]);
                        }
#pragma unroll
                        for (int j = 0; j < 16; j += 4) {
                            const float4 bb = *reinterpret_cast<const float4*>(&s_bias[l][c0 + j]);
                            v[j] += bb.x; v[j + 1] += bb.y; v[j + 2] += bb.z; v[j + 3] += bb.w;
                        }
                        if (relu) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
                        }
                        if (feed) {                                  // next layer's A operand: row row_img, columns c0 .. c0 + 15 (two 16-byte chunks)
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const int c = c0 + h * 8;
                                const uint32_t off = (uint32_t)(c >> 6) * 16384u + (uint32_t)row_img * 128u + ((((uint32_t)(c & 63) >> 3) ^ (uint32_t)(row_img & 7)) << 4);
                                uint32_t hh[4], ll[4];
#pragma unroll
                                for (int q = 0; q < 4; ++q) {
                                    const float a = v[h * 8 + 2 * q], b2 = v[h * 8 + 2 * q + 1];
                                    hh[q] = pack_bf16(a, b2);
                                    ll[q] = pack_bf16(a - __uint_as_float(hh[q] << 16), b2 - __uint_as_float(hh[q] & 0xFFFF0000u));
                                }
                                *reinterpret_cast<uint4*>(img_hi + off) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
                                if (NSPLIT == 3) *reinterpret_cast<uint4*>(img_hi + kTile + off) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
                            }
                        }
#pragma unroll
                        for (int j = 0; j < 16; j += 4)
                            *reinterpret_cast<float4*>(scratch + lane * kWsScratchLd + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int r = j * 8 + r_in;
                            const int row = m0 + r;
                            if (row < r_end)
                                *reinterpret_cast<float4*>(p.Y[l] + (long)row * p.ldy[l] + c0 + c4) = *reinterpret_cast<const float4*>(scratch + r * kWsScratchLd + c4);
                        }
                        __syncwarp();
                    }
                    if (feed) {
                        tc_fence_before();                           // TMEM tile drained
                        fence_async_smem();                          // image writes visible to the tensor core
                        mbar_arrive(&bar_aready[t]);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------------------------------------ weight gradient
// dW[n, k] += sum_m dY[m, n] X[m, k].  MMA shape M = N_out (rows of dW, <= 128 -> padded to 128), N = K_out, K = rows m.
// Both operands MN-major, no swizzle: element (mn, k) at byte (k/8)*LBO + (mn/8)*128 + (k%8)*16 + (mn%8)*2,
// LBO = MN*16: a source row m (contiguous in mn) lands as 16-byte chunks -> conflict-free 16-byte stores.
// Sub-tiles of 64 rows (4 k-steps): both operands of a sub-tile are prefetched into registers (batched loads).
constexpr int kWgRows = 64;
constexpr int kWgIt = 4;     // 16-byte chunks per thread per batch: 64 rows x 128 columns / 8 / 256 threads

// chunk c of a [64 rows x MN] operand: 8 lanes cover 8 consecutive rows of one 8-wide column chunk.  MN/8 is a power
// of two <= 32 and a thread block advances 32 chunk columns per step, so a thread's column chunk j is constant and only
// the 8-row group kg advances.
template <bool VEC>
__device__ __forceinline__ void load_mnmajor_t(float4 (&pre)[2 * kWgIt], const float* __restrict__ src, long ld, long row0, int rows_valid, int MN,
                                               int mn_valid, int c_base) {
    const int vec_ok = VEC;
    const int n_chunks = MN >> 3, lgc = ilog2(n_chunks);
    const int r = threadIdx.x & 7, q = (c_base >> 3) + (threadIdx.x >> 3);
    const int j = q & (n_chunks - 1), kg_step = 32 >> lgc;
    int kg = q >> lgc;
    const bool col_ok = j * 8 < mn_valid, full = vec_ok && (j * 8 + 8 <= mn_valid);
    const float* g = src + (row0 + kg * 8 + r) * ld + j * 8;
    const long gstep = (long)kg_step * 8 * ld;
#pragma unroll
    for (int i = 0; i < kWgIt; ++i) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        if (kg < (kWgRows >> 3) && kg * 8 + r < rows_valid && col_ok) {
            if (full) {
                a = __ldg(reinterpret_cast<const float4*>(g));
                b = __ldg(reinterpret_cast<const float4*>(g + 4));
            } else {
                float t[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) t[e] = (j * 8 + e < mn_valid) ? __ldg(g + e) : 0.f;
                a = make_float4(t[0], t[1], t[2], t[3]);
                b = make_float4(t[4], t[5], t[6], t[7]);
            }
        }
        pre[2 * i] = a; pre[2 * i + 1] = b;
        kg += kg_step;
        g += gstep;
    }
}

__device__ __forceinline__ void load_mnmajor(float4 (&pre)[2 * kWgIt], const float* __restrict__ src, long ld, long row0, int rows_valid, int MN,
                                             int mn_valid, int c_base, int vec_ok) {
    if (vec_ok && mn_valid == MN) load_mnmajor_t<true>(pre, src, ld, row0, rows_valid, MN, mn_valid, c_base);   // all-vector fast path
    else load_mnmajor_t<false>(pre, src, ld, row0, rows_valid, MN, mn_valid, c_base);
}

template <int NSPLIT>
__device__ __forceinline__ void store_mnmajor(const float4 (&pre)[2 * kWgIt], uint8_t* hi, uint8_t* lo, int MN, int c_base, int relu, uint32_t lbo) {
    const int n_chunks = MN >> 3, lgc = ilog2(n_chunks);
    const int r = threadIdx.x & 7, q = (c_base >> 3) + (threadIdx.x >> 3);
    const int j = q & (n_chunks - 1), kg_step = 32 >> lgc;
    int kg = q >> lgc;
    uint32_t off = (uint32_t)kg * lbo + (uint32_t)j * 128u + (uint32_t)r * 16u;
#pragma unroll
    for (int i = 0; i < kWgIt; ++i) {
        if (kg < (kWgRows >> 3)) {
            float v[8] = {pre[2 * i].x, pre[2 * i].y, pre[2 * i].z, pre[2 * i].w, pre[2 * i + 1].x, pre[2 * i + 1].y, pre[2 * i + 1].z, pre[2 * i + 1].w};
            if (relu) {
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = fmaxf(v[e], 0.f);
            }
            const uint4 h = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
            *reinterpret_cast<uint4*>(hi + off) = h;
            if (NSPLIT == 3) {
                const uint32_t hh[4] = {h.x, h.y, h.z, h.w};
                uint32_t ll[4];
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    ll[e] = pack_bf16(v[2 * e] - __uint_as_float(hh[e] << 16), v[2 * e + 1] - __uint_as_float(hh[e] & 0xFFFF0000u));
                *reinterpret_cast<uint4*>(lo + off) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
            }
        }
        kg += kg_step;
        off += (uint32_t)kg_step * lbo;
    }
}

struct TcWgParams {
    const float* dY; long lddy;    // [M, N]
    const float* X; long ldx;      // [M, K]
    float* dW; long lddw;          // [N, K], accumulated with atomics
    float* db;                     // [N] bias gradient (+=) via an extra all-ones column of the X operand, or null
    long M; int N, K;
    int relu_in, dy_vec, x_vec;
    long rows_per_cta;
};

template <int NSPLIT>
__global__ void __launch_bounds__(256, 2) wgrad_tc_kernel(TcWgParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t mma_bar;
    __shared__ uint32_t tmem_slot;
    const int K = p.K;
    const int KE = p.db ? K + 16 : K;    // MMA N extent: 16 extra columns, the first one all ones -> D[:, K] = sum_m dY[m, :]
    const uint32_t a_bytes = (uint32_t)kWgRows * 128u * 2u, b_bytes = (uint32_t)kWgRows * (uint32_t)KE * 2u;
    uint8_t* a_hi = smem_raw;
    uint8_t* a_lo = a_hi + a_bytes;
    uint8_t* b_hi = smem_raw + (NSPLIT == 3 ? 2 : 1) * a_bytes;
    uint8_t* b_lo = b_hi + b_bytes;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t ncols = KE <= 32 ? 32u : (KE <= 64 ? 64u : (KE <= 128 ? 128u : 256u));
    if (warp == 0) tmem_alloc(&tmem_slot, ncols);
    if (tid == 0) mbar_init(&mma_bar, 1);
    const uint32_t a_lbo = 128u * 16u, b_lbo = (uint32_t)KE * 16u;
    if (p.db) {
        // constant part of the X operand: chunk K/8 of every row m holds [1,0,...,0], chunk K/8 + 1 holds zeros
        for (int i = tid; i < kWgRows * 2; i += 256) {
            const int m = i >> 1, jx = (K >> 3) + (i & 1);
            const uint32_t off = (uint32_t)(m >> 3) * b_lbo + (uint32_t)jx * 128u + (uint32_t)(m & 7) * 16u;
            *reinterpret_cast<uint4*>(b_hi + off) = make_uint4((i & 1) ? 0u : 0x00003F80u, 0u, 0u, 0u);   // bf16(1.0) = 0x3F80
            if (NSPLIT == 3) *reinterpret_cast<uint4*>(b_lo + off) = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t idesc = make_idesc(128, KE, 1, 1);
    const int b_batches = (kWgRows * (K >> 3) + 256 * kWgIt - 1) / (256 * kWgIt);   // 1 for K <= 128, 2 for K = 256

    const long m_begin = (long)blockIdx.x * p.rows_per_cta;
    const long m_end = min(p.M, m_begin + p.rows_per_cta);
    uint32_t phase = 0, acc = 0;
    float4 pa[2 * kWgIt], pb[2 * kWgIt];
    if (m_begin < m_end) {
        const int rows = (int)min((long)kWgRows, m_end - m_begin);
        load_mnmajor(pa, p.dY, p.lddy, m_begin, rows, 128, p.N, 0, p.dy_vec);
        load_mnmajor(pb, p.X, p.ldx, m_begin, rows, K, K, 0, p.x_vec);
    }
    for (long m0 = m_begin; m0 < m_end; m0 += kWgRows) {
        const int rows = (int)min((long)kWgRows, m_end - m0);
        if (acc) {           // previous sub-tile's MMAs must have consumed the operand buffers
            mbar_wait(&mma_bar, phase);
            phase ^= 1;
        }
        store_mnmajor<NSPLIT>(pa, a_hi, a_lo, 128, 0, 0, a_lbo);
        store_mnmajor<NSPLIT>(pb, b_hi, b_lo, K, 0, p.relu_in, b_lbo);
        for (int bb = 1; bb < b_batches; ++bb) {       // K = 256: second half of the X sub-tile
            load_mnmajor(pb, p.X, p.ldx, m0, rows, K, K, bb * 256 * kWgIt, p.x_vec);
            store_mnmajor<NSPLIT>(pb, b_hi, b_lo, K, bb * 256 * kWgIt, p.relu_in, b_lbo);
        }
        const long mn = m0 + kWgRows;
        if (mn < m_end) {    // prefetch the next sub-tile: in flight under the fence / sync / MMA issue
            const int rn = (int)min((long)kWgRows, m_end - mn);
            load_mnmajor(pa, p.dY, p.lddy, mn, rn, 128, p.N, 0, p.dy_vec);
            load_mnmajor(pb, p.X, p.ldx, mn, rn, K, K, 0, p.x_vec);
        }
        fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            const uint32_t sa_hi = smem_u32(a_hi), sa_lo = smem_u32(a_lo), sb_hi = smem_u32(b_hi), sb_lo = smem_u32(b_lo);
            for (int ks = 0; ks < kWgRows / 16; ++ks) {     // k-steps of 16 rows (2 k-groups of 8)
                const uint32_t ao = (uint32_t)ks * 2u * a_lbo, bo = (uint32_t)ks * 2u * b_lbo;
                umma_bf16(tmem, make_desc(sa_hi + ao, a_lbo, 128), make_desc(sb_hi + bo, b_lbo, 128), idesc, acc);
                acc = 1;
                if (NSPLIT == 3) {
                    umma_bf16(tmem, make_desc(sa_hi + ao, a_lbo, 128), make_desc(sb_lo + bo, b_lbo, 128), idesc, 1);
                    umma_bf16(tmem, make_desc(sa_lo + ao, a_lbo, 128), make_desc(sb_hi + bo, b_lbo, 128), idesc, 1);
                }
            }
            umma_commit(&mma_bar);
        }
        acc = 1;
    }
    if (acc) {
        mbar_wait(&mma_bar, phase);
        tc_fence_after();
        const int lane_base = 32 * (warp & 3);
        const int n = lane_base + lane;                    // row of dW
        const int split = ((K + 1) / 2 + 15) / 16 * 16;
        const int c_begin = (warp >> 2) ? split : 0, c_end = (warp >> 2) ? K : min(K, split);
        for (int c0 = c_begin; c0 < c_end; c0 += 16) {
            float v[16];
            tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)c0, v);
            if (n < p.N) {
                float* d = p.dW + (long)n * p.lddw + c0;
                if ((p.lddw & 3) == 0 && (reinterpret_cast<uintptr_t>(p.dW) & 15) == 0) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4) atomicAdd(reinterpret_cast<float4*>(d + j), make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
                } else {
                    atomic_add16(d, v);
                }
            }
        }
        if (p.db && warp < 4) {       // the ones column: D[n, K] = sum over rows of dY[:, n]
            float v[16];
            tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)K, v);
            if (n < p.N) atomicAdd(p.db + n, v[0]);
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, ncols);
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static bool pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }
static bool tc_shape_ok(int red, int out) { return pow2(red) && red >= 16 && red <= 128 && pow2(out) && out >= 16 && out <= 256; }

template <int NSPLIT>
static int launch_lin(TcLinParams& p, cudaStream_t st) {
    const size_t smem = (size_t)(NSPLIT == 3 ? 2 : 1) * (128 + p.NO) * p.KR * 2 + (size_t)(kLinThreads / 32) * 32 * kScratchLd * sizeof(float);
    static size_t reserved = 0;
    if (smem > reserved) {
        if (cudaFuncSetAttribute(linear_tc_kernel<NSPLIT, 128, 128, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(linear_tc_kernel<NSPLIT, 128, 128, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(linear_tc_kernel<NSPLIT, 128, 128, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(linear_tc_kernel<NSPLIT, 0, 0, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(linear_tc_kernel<NSPLIT, 0, 0, true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess) {
            cudaGetLastError();
            return NPF_ENOTSUP;
        }
        reserved = 220 * 1024;
    }
    if (smem > 220 * 1024) return NPF_ENOTSUP;
    p.n_tiles = (int)cdiv(p.M, 128);
    // CTAs per SM limited by shared memory; stay persistent with one CTA per resident slot
    const int per_sm = 1;   // 512 threads + ~200 KB of shared memory: one persistent CTA per SM
    int grid = kNumSMs * per_sm;
    if (grid > p.n_tiles) grid = p.n_tiles;
    // VEC: every activation / output / mask access is a 16-byte one (leading dimensions % 4 == 0, 16-byte aligned bases)
    const bool vec = p.a_vec && p.c_vec && (!p.mask || ((p.ldm & 3) == 0 && (reinterpret_cast<uintptr_t>(p.mask) & 15) == 0));
    const bool hot = vec && p.KR == 128 && p.NO == 128;
    if (hot && !(p.u && p.mask)) {
        p.rows_per_cta = (int)(cdiv(cdiv(p.M, grid), 8) * 8);
        const int ws_grid = (int)cdiv(p.M, p.rows_per_cta);
        // warp-specialised pipeline (2 operand stages + weights + epilogue scratch)
        const size_t ws_smem = (size_t)3 * (NSPLIT == 3 ? 2 : 1) * 32768 + (size_t)kWsEpiWarps * 32 * kWsScratchLd * sizeof(float);
        static bool ws_attr = false;
        if (!ws_attr) {
            bool ok = true;
#define NPF_WS_ATTR(U, MK, S) ok = ok && cudaFuncSetAttribute(linear_ws_kernel<NSPLIT, U, MK, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) == cudaSuccess
            NPF_WS_ATTR(false, false, true); NPF_WS_ATTR(true, false, true); NPF_WS_ATTR(false, true, true);
#undef NPF_WS_ATTR
            if (!ok) {
                cudaGetLastError();
                return NPF_ENOTSUP;
            }
            ws_attr = true;
        }
        if (p.u) launch_pdl(linear_ws_kernel<NSPLIT, true, false, true>, ws_grid, kWsThreads, ws_smem, st, p);
        else if (p.mask) launch_pdl(linear_ws_kernel<NSPLIT, false, true, true>, ws_grid, kWsThreads, ws_smem, st, p);
        else launch_pdl(linear_ws_kernel<NSPLIT, false, false, true>, ws_grid, kWsThreads, ws_smem, st, p);
        count_launch();
        return check_launch("linear_ws_kernel");
    }
    if (hot && !p.u && !p.mask) linear_tc_kernel<NSPLIT, 128, 128, false, false, true><<<grid, kLinThreads, smem, st>>>(p);
    else if (hot && !p.u) linear_tc_kernel<NSPLIT, 128, 128, false, true, true><<<grid, kLinThreads, smem, st>>>(p);
    else if (hot && !p.mask) linear_tc_kernel<NSPLIT, 128, 128, true, false, true><<<grid, kLinThreads, smem, st>>>(p);
    else if (vec) linear_tc_kernel<NSPLIT, 0, 0, true, true, true><<<grid, kLinThreads, smem, st>>>(p);
    else linear_tc_kernel<NSPLIT, 0, 0, true, true, false><<<grid, kLinThreads, smem, st>>>(p);
    count_launch();
    return check_launch("linear_tc_kernel");
}

int linear_fwd_tc(const float* X, int ldx, const float* W, int ldw, const float* b, float* Y, int ldy, int M, int K,
                  int N, int flags, const float* u, const float* w2, int ldw2, int precision, cudaStream_t st) {
    if (!tc_shape_ok(K, N) || (flags & NPF_ACCUM)) return NPF_ENOTSUP;
    TcLinParams p{};
    p.A = X; p.lda = ldx; p.W = W; p.ldw = ldw; p.C = Y; p.ldc = ldy; p.bias = b;
    p.u = u; p.w2 = w2; p.ldw2 = ldw2;
    p.M = M; p.KR = K; p.NO = N;
    p.relu_in = (flags & NPF_RELU_IN) ? 1 : 0; p.relu_out = (flags & NPF_RELU_OUT) ? 1 : 0;
    p.transposed_w = 0;
    p.a_vec = (ldx % 4 == 0) && aligned16(X);
    p.w_vec = (ldw % 4 == 0) && aligned16(W);
    p.c_vec = (ldy % 4 == 0) && aligned16(Y);
    return precision == NPF_PREC_BF16X3 ? launch_lin<3>(p, st) : launch_lin<1>(p, st);
}

int linear_bwd_data_tc(const float* dY, int lddy, const float* W, int ldw, float* dX, int lddx, int M, int K, int N,
                       const float* mask_src, int ldm, int flags, int precision, cudaStream_t st) {
    if (!tc_shape_ok(N, K) || (flags & NPF_ACCUM)) return NPF_ENOTSUP;
    TcLinParams p{};
    p.A = dY; p.lda = lddy; p.W = W; p.ldw = ldw; p.C = dX; p.ldc = lddx;
    p.mask = mask_src; p.ldm = ldm;
    p.M = M; p.KR = N; p.NO = K;
    p.transposed_w = 1;
    p.a_vec = (lddy % 4 == 0) && aligned16(dY);
    p.w_vec = (ldw % 4 == 0) && aligned16(W);
    p.c_vec = (lddx % 4 == 0) && aligned16(dX);
    return precision == NPF_PREC_BF16X3 ? launch_lin<3>(p, st) : launch_lin<1>(p, st);
}


// ------------------------------------------------------------------------------------------------ fused backward, 64-row tiles
// dX = (dY W) (.) (X > 0)   and   dW += dY^T X,  db += colsum(dY)   in ONE pass over dY and X (hot shape only).
// The dY and X row tiles are staged once (SW128, bf16 hi/lo) and each is read by the tensor core two ways:
//     dX^T[k, m] = sum_n W[n, k] dY[m, n]      A = W^T (MN-major view of the row-staged W),  B = dY tile (K-major),  N = 64
//     dW[n, k]  += sum_m dY[m, n] X[m, k]      A = dY^T, B = X (MN-major views of the same bytes), 4 k-steps of 16 rows
//     db        += column sums of dY, taken by the producers from the registers the tile passes through (exact fp32)
// so a separate weight-gradient kernel's second read of dY and X (2/5 of the backward traffic of a layer) is not needed and
// the relu mask comes from the staged X tile instead of a third global stream.
// Tiles are 64 rows so that the operand stage fits TWICE in shared memory (x3: 2 x 64 KB + 64 KB of weights): a 128-row
// stage fits only once, and "convert+store tile i+1" then waits for "multiply tile i" (14 k cycles per tile measured, against
// 8.7 k of HBM time).  The tensor-core M dimension is kept at 128 by computing the data gradient TRANSPOSED: the accumulator
// has k on the TMEM lanes and the tile's rows on the columns, so an epilogue thread owns ONE column k of dX and every register
// it reads is one row: a warp store covers 128 contiguous bytes without any shared-memory transpose, and the relu mask is a
// 2-byte read of the staged X tile.  Roles: 16 producer warps (TWO tiles in flight in registers), 1 MMA warp, 8 epilogue
// warps.  TMEM: [0,128) dX^T x2, [128,256) dW.
constexpr int kFbProdWarps = 16;
constexpr int kFbEpiWarp0 = 17;
constexpr int kFbThreads = (kFbEpiWarp0 + kWsEpiWarps) * 32;     // 800

struct TcFusedParams {
    const float* dY; long lddy;     // [M, 128]
    const float* X; long ldx;       // [M, 128]  layer input (post-relu activations): wgrad operand and relu mask
    const float* W; long ldw;       // [128 (n), 128 (k)]
    float* dX; long lddx;           // [M, 128]
    float* dW; long lddw;           // [128, 128]  +=
    float* db;                      // [128] += or null
    int M, n_tiles, rows_per_cta;
    int relu_x, use_mask, w_vec, dw_vec;
};

#ifndef F64_DEPTH
#define F64_DEPTH 1
#endif
constexpr int kF64Rows = 64;
#ifndef NPF_F64_AHEAD
#define NPF_F64_AHEAD 4
#endif
constexpr int kF64Ahead = NPF_F64_AHEAD;

__device__ __forceinline__ void f64_load_rows(float4 (&pre)[4], const float* __restrict__ g, long ld, int row_first, int rows_valid) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        pre[i] = (row_first + i < rows_valid) ? __ldg(reinterpret_cast<const float4*>(g)) : make_float4(0.f, 0.f, 0.f, 0.f);
        g += ld;
    }
}
__device__ __forceinline__ void f64_prefetch(const float* __restrict__ base, long ld, long row0, int rows_valid, int t) {
    // 64 rows x 512 bytes = 256 lines; threads 0..255 take dY / 256..511 are given the X tile by the caller
    const int l = t & 255, r = l >> 2;
    if (r < rows_valid) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (row0 + r) * ld + (l & 3) * 32));
}

template <int NSPLIT, bool HAS_MASK>
__global__ void __launch_bounds__(kFbThreads, 1) linear_bwd_fused64_kernel(TcFusedParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[2], bar_empty[2], bar_mask[2], bar_dwfull, bar_tfull[2], bar_tempty[2];
    __shared__ uint32_t tmem_slot;
    __shared__ float s_db[128];

    constexpr uint32_t kHalf = 64u * 128u * 2u;                    // one bf16 64 x 128 operand image: 16 KB
    constexpr uint32_t kOp = (NSPLIT == 3 ? 2u : 1u) * kHalf;      // hi [+ lo]
    constexpr uint32_t kStage = 2u * kOp;                          // dY + X
    constexpr uint32_t kWTile = 128u * 128u * 2u;                  // 32 KB
    uint8_t* w_hi = smem_raw + 2 * kStage;
    uint8_t* w_lo = w_hi + kWTile;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    if (tid == 32) {
        mbar_init(&bar_dwfull, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_full[i], kFbProdWarps * 32);
            mbar_init(&bar_empty[i], 1);
            mbar_init(&bar_mask[i], kWsEpiWarps * 32);
            mbar_init(&bar_tfull[i], 1);
            mbar_init(&bar_tempty[i], kWsEpiWarps * 32);
        }
    }
    if (tid < 128) s_db[tid] = 0.f;

    const int r_begin = blockIdx.x * p.rows_per_cta, r_end = min(p.M, r_begin + p.rows_per_cta);
    const int n_local = r_end > r_begin ? (r_end - r_begin + kF64Rows - 1) / kF64Rows : 0;
    const uint32_t pchunk = (uint32_t)(lane >> 1) & 7u;
    pdl_trigger();
    if (warp < kFbProdWarps) {          // weights: warp w stages rows 8 w .. 8 w + 7 of W (two 64-column atoms of 16 KB)
        const uint32_t woff = (uint32_t)(lane >> 4) * 16384u + (uint32_t)(warp * 8) * 128u + (uint32_t)(lane & 1) * 8u;
        float4 wv[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float* g = p.W + (long)(warp * 8 + i) * p.ldw + lane * 4;
            if (p.w_vec) wv[i] = __ldg(reinterpret_cast<const float4*>(g));
            else wv[i] = make_float4(__ldg(g), __ldg(g + 1), __ldg(g + 2), __ldg(g + 3));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) cvt_store<NSPLIT>(wv[i], w_hi, w_lo, woff + (uint32_t)i * 128u + ((pchunk ^ (uint32_t)i) << 4), 0);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    pdl_wait();

    if (warp < kFbProdWarps) {
        // ------------------------------------------------------------------ producers: warp w owns rows 4 w .. 4 w + 3 of a tile
        const int prow = warp * 4;
        const uint32_t psoff = (uint32_t)(lane >> 4) * 8192u + (uint32_t)prow * 128u + (uint32_t)(lane & 1) * 8u;
        const uint32_t rsw = (uint32_t)(prow & 7);                   // row % 8 of the warp's first row (0 or 4)
        float4 ya[4], xa[4], yb[4], xb[4];
        float4 dbs = make_float4(0.f, 0.f, 0.f, 0.f);
        auto load_tile = [&](float4 (&yy)[4], float4 (&xx)[4], int it) {
            const int row0 = r_begin + it * kF64Rows, rv = min(kF64Rows, r_end - row0);
            f64_load_rows(yy, p.dY + ((long)row0 + prow) * p.lddy + lane * 4, p.lddy, prow, rv);
            f64_load_rows(xx, p.X + ((long)row0 + prow) * p.ldx + lane * 4, p.ldx, prow, rv);
        };
        auto put_tile = [&](float4 (&yy)[4], float4 (&xx)[4], int it) {
            const int s = it & 1;
#pragma unroll
            for (int i = 0; i < 4; ++i) { dbs.x += yy[i].x; dbs.y += yy[i].y; dbs.z += yy[i].z; dbs.w += yy[i].w; }
            if (it >= 2) {
                mbar_wait(&bar_empty[s], ((it >> 1) - 1) & 1);               // the MMAs of tile it-2 have read this stage
                if (HAS_MASK) mbar_wait(&bar_mask[s], ((it >> 1) - 1) & 1);  // and the epilogue has taken its relu mask
            }
            uint8_t* y_hi = smem_raw + s * kStage;
            uint8_t* x_hi = y_hi + kOp;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint32_t off = psoff + (uint32_t)i * 128u + ((pchunk ^ (rsw + (uint32_t)i)) << 4);
                cvt_store<NSPLIT>(yy[i], y_hi, y_hi + kHalf, off, 0);
                cvt_store<NSPLIT>(xx[i], x_hi, x_hi + kHalf, off, p.relu_x);
            }
            fence_async_smem();
            mbar_arrive(&bar_full[s]);
            if (it + F64_DEPTH < n_local) load_tile(yy, xx, it + F64_DEPTH);
            if (it + kF64Ahead < n_local) {        // L2 prefetch kF64Ahead tiles ahead (2 tiles are in flight in registers)
                const int row0 = r_begin + (it + kF64Ahead) * kF64Rows, rv = min(kF64Rows, r_end - row0);
                if (tid < 256) f64_prefetch(p.dY, p.lddy, row0, rv, tid); else f64_prefetch(p.X, p.ldx, row0, rv, tid);
            }
        };
        static const int kDepth = F64_DEPTH;
        if (n_local > 0) load_tile(ya, xa, 0);
        if (kDepth == 2 && n_local > 1) load_tile(yb, xb, 1);
        for (int a = kDepth; a < kF64Ahead && a < n_local; ++a) {
            const int row0 = r_begin + a * kF64Rows, rv = min(kF64Rows, r_end - row0);
            if (tid < 256) f64_prefetch(p.dY, p.lddy, row0, rv, tid); else f64_prefetch(p.X, p.ldx, row0, rv, tid);
        }
        if (kDepth == 2) {
            for (int it = 0; it < n_local; it += 2) {
                put_tile(ya, xa, it);
                if (it + 1 < n_local) put_tile(yb, xb, it + 1);
            }
        } else {
            for (int it = 0; it < n_local; ++it) put_tile(ya, xa, it);
        }
        if (p.db) {
            atomicAdd(&s_db[lane * 4 + 0], dbs.x); atomicAdd(&s_db[lane * 4 + 1], dbs.y);
            atomicAdd(&s_db[lane * 4 + 2], dbs.z); atomicAdd(&s_db[lane * 4 + 3], dbs.w);
            asm volatile("bar.sync 1, %0;" ::"n"(kFbProdWarps * 32) : "memory");
            if (tid < 128) atomicAdd(p.db + tid, s_db[tid]);
        }
    } else if (warp == kFbProdWarps) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc_dx = make_idesc(128, 64, 1, 0);     // A = W^T (MN-major view), B = dY tile (K-major), D = dX^T [k x m]
            const uint32_t idesc_dw = make_idesc(128, 128, 1, 1);    // A = dY^T, B = X: MN-major views (reduction over the tile's rows)
            const uint32_t sw_hi = smem_u32(w_hi), sw_lo = smem_u32(w_lo);
            const uint32_t d_dw = tmem + 128u;
            for (int it = 0; it < n_local; ++it) {
                const int s = it & 1;
                const uint32_t par = (it >> 1) & 1;
                mbar_wait(&bar_full[s], par);
                mbar_wait(&bar_tempty[s], par ^ 1);
                tc_fence_after();
                const uint32_t sy_hi = smem_u32(smem_raw + s * kStage), sy_lo = sy_hi + kHalf, sx_hi = sy_hi + kOp, sx_lo = sx_hi + kHalf;
                const uint32_t d_dx = tmem + (uint32_t)s * 64u;
                // base descriptors once per tile, one add per k-slice (desc_adv): the issuing thread's instruction count is what paces the MMAs
                const uint64_t dwt_h = make_desc_sw128(sw_hi, 16384, 1024), dwt_l = make_desc_sw128(sw_lo, 16384, 1024);
                const uint64_t dyk_h = make_desc_sw128(sy_hi, 16, 1024), dyk_l = make_desc_sw128(sy_lo, 16, 1024);
                const uint64_t dym_h = make_desc_sw128(sy_hi, 8192, 1024), dym_l = make_desc_sw128(sy_lo, 8192, 1024);
                const uint64_t dxm_h = make_desc_sw128(sx_hi, 8192, 1024), dxm_l = make_desc_sw128(sx_lo, 8192, 1024);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks) {                     // reduction over n (16 per step)
                    const uint32_t bo = (uint32_t)(ks >> 2) * 8192u + (uint32_t)(ks & 3) * 32u;
                    const uint64_t a_h = desc_adv(dwt_h, ks * 2048u), b_h = desc_adv(dyk_h, bo);
                    umma_bf16(d_dx, a_h, b_h, idesc_dx, ks ? 1u : 0u);
                    if (NSPLIT == 3) {
                        umma_bf16(d_dx, a_h, desc_adv(dyk_l, bo), idesc_dx, 1);
                        umma_bf16(d_dx, desc_adv(dwt_l, ks * 2048u), b_h, idesc_dx, 1);
                    }
                }
                umma_commit(&bar_tfull[s]);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {                     // reduction over the 64 rows of the tile
                    const uint32_t acc = (it | ks) ? 1u : 0u;
                    const uint64_t a_h = desc_adv(dym_h, ks * 2048u), b_h = desc_adv(dxm_h, ks * 2048u);
                    umma_bf16(d_dw, a_h, b_h, idesc_dw, acc);
                    if (NSPLIT == 3) {
                        umma_bf16(d_dw, a_h, desc_adv(dxm_l, ks * 2048u), idesc_dw, 1);
                        umma_bf16(d_dw, desc_adv(dym_l, ks * 2048u), b_h, idesc_dw, 1);
                    }
                }
                umma_commit(&bar_empty[s]);
            }
            umma_commit(&bar_dwfull);
        }
    } else {
        // ------------------------------------------------------------------ epilogue: thread = column k of dX, 32 rows of the tile
        const int e = warp - kFbEpiWarp0;
        const int lane_base = 32 * (warp & 3);
        const int k = lane_base + lane;
        const int mh = (e >> 2) * 32;                                  // this warp's half of the tile's 64 rows
        const uint32_t xk_off = (uint32_t)(k >> 6) * 8192u + (uint32_t)(k & 7) * 2u, xk_chunk = (uint32_t)(k & 63) >> 3;
        for (int it = 0; it < n_local; ++it) {
            const int s = it & 1;
            const int row0 = r_begin + it * kF64Rows + mh;
            mbar_wait(&bar_tfull[s], (it >> 1) & 1);
            tc_fence_after();
            uint32_t mbits = 0xFFFFFFFFu;
            if (HAS_MASK) {          // relu mask of column k for the 32 rows, from the staged (relu'd) X tile: bf16 > 0 <=> int16 > 0
                const uint8_t* x_hi = smem_raw + s * kStage + kOp;
                mbits = 0u;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const uint32_t m = (uint32_t)(mh + j);
                    const short xb = *reinterpret_cast<const short*>(x_hi + xk_off + m * 128u + ((xk_chunk ^ (m & 7u)) << 4));
                    mbits |= (xb > 0 ? 1u : 0u) << j;
                }
                mbar_arrive(&bar_mask[s]);
            }
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                float v[16];
                tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(s * 64 + mh + c * 16), v);
                if (c == 1) {
                    tc_fence_before();
                    mbar_arrive(&bar_tempty[s]);
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int row = row0 + c * 16 + j;
                    if (row < r_end) p.dX[(long)row * p.lddx + k] = ((mbits >> (c * 16 + j)) & 1u) ? v[j] : 0.f;
                }
            }
        }
        // ---- flush of the CTA's weight gradient: thread = row n of dW, 64 columns per warp
        mbar_wait(&bar_dwfull, 0);
        tc_fence_after();
        const int col_base = (e >> 2) * 64;
#pragma unroll 1
        for (int ch = 0; ch < 4; ++ch) {
            const int c0 = col_base + ch * 16;
            float v[16];
            tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(128 + c0), v);
            float* d = p.dW + (long)k * p.lddw + c0;
            if (p.dw_vec) {
#pragma unroll
                for (int j = 0; j < 16; j += 4) atomicAdd(reinterpret_cast<float4*>(d + j), make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
            } else {
                atomic_add16(d, v);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

// Fused data + weight (+ bias) gradient of a 128 -> 128 layer; NPF_ENOTSUP for any other shape / alignment (the caller
// then runs the two separate kernels).
template <int NSPLIT>
static int launch_fused(TcFusedParams& p, cudaStream_t st) {
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(linear_bwd_fused64_kernel<NSPLIT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(linear_bwd_fused64_kernel<NSPLIT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024) != cudaSuccess) {
            cudaGetLastError();
            return NPF_ENOTSUP;
        }
        attr = true;
    }
    p.n_tiles = (int)cdiv(p.M, 128);
    int grid = p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs;
    p.rows_per_cta = (int)(cdiv(cdiv(p.M, grid), 8) * 8);
    grid = (int)cdiv(p.M, p.rows_per_cta);
    const size_t smem = (size_t)(NSPLIT == 3 ? 2 : 1) * (4 * 16384 + 32768);      // two 64-row dY + X stages, the weights
    if (p.use_mask) launch_pdl(linear_bwd_fused64_kernel<NSPLIT, true>, grid, kFbThreads, smem, st, p);
    else launch_pdl(linear_bwd_fused64_kernel<NSPLIT, false>, grid, kFbThreads, smem, st, p);
    count_launch();
    return check_launch("linear_bwd_fused64_kernel");
}

int linear_bwd_fused_tc(const float* dY, int lddy, const float* X, int ldx, const float* W, int ldw, float* dX, int lddx, float* dW,
                        int lddw, float* db, int M, int K, int N, int flags, int precision, cudaStream_t st) {
    if (K != 128 || N != 128 || M < 128) return NPF_ENOTSUP;
    if ((lddy | ldx | lddx) % 4 != 0 || !aligned16(dY) || !aligned16(X) || !aligned16(dX)) return NPF_ENOTSUP;
    TcFusedParams p{};
    p.dY = dY; p.lddy = lddy; p.X = X; p.ldx = ldx; p.W = W; p.ldw = ldw; p.dX = dX; p.lddx = lddx;
    p.dW = dW; p.lddw = lddw; p.db = db; p.M = M;
    p.relu_x = (flags & NPF_RELU_IN) ? 1 : 0;
    p.use_mask = (flags & NPF_MASK_X) ? 1 : 0;
    p.w_vec = (ldw % 4 == 0) && aligned16(W);
    p.dw_vec = (lddw % 4 == 0) && aligned16(dW);
    return precision == NPF_PREC_BF16X3 ? launch_fused<3>(p, st) : launch_fused<1>(p, st);
}

// ------------------------------------------------------------------------------------------------ MLP chain BACKWARD (128-wide)
// Whole backward of L consecutive Linear(128 -> 128) + ReLU layers with the pre-activation gradient kept ON CHIP between layers
// (the mirror of mlp_chain_fwd_kernel).  A CTA owns a row group of up to 256 rows = four 64-row blocks whose gradient images
// dZ_l (bf16 hi / lo, SWIZZLE_128B, row-major) stay resident in shared memory; layers are walked from the last to the first:
//     dA^T[k, m] = sum_n W_l[n, k] dZ_l[m, n]          (A = W_l^T: MN-major view of the row-staged W_l,  B = dZ block, K-major, N = 64)
//     dW_l[n, k] += sum_m dZ_l[m, n] X_l[m, k]         (A = dZ_l^T, B = X_l block: MN-major views; TMEM accumulator over the CTA's blocks,
//                                                       one flush of float4 atomics per layer, double-buffered across layers)
//     dZ_{l-1} = dA (.) (X_l > 0)                      written by the epilogue straight back into the block's image (thread = column k),
//     db_{l-1} = colsum(dZ_{l-1})                      summed in the epilogue's registers (exact fp32)
// so per layer HBM sees only the saved input X_l (read once: wgrad operand AND relu mask) -- dY is read once for the whole
// chain and only the first layer's dX is written.  Against L x npf_linear_bwd this removes L - 1 writes and L - 1 reads of an
// [M, 128] gradient (250 MB -> 117 MB for the 4-layer decoder at M = 32 768) and L - 1 launches with their fill / drain.
// Roles as in linear_bwd_fused64_kernel: 16 producer warps (dY blocks once, then W_l and the X_l blocks), 1 MMA warp, 8 epilogue
// warps.  Shared memory: 4 x 32 KB gradient images + 32 KB X stage + 64 KB weights = 224 KB (x3).
constexpr int kCbBlocks = 4;
struct ChainBwdParams {
    const float* dY; long lddy;
    const float* X[kChainMaxLayers]; long ldx[kChainMaxLayers];      // input of layer l (post-relu output of layer l - 1)
    const float* W[kChainMaxLayers]; long ldw[kChainMaxLayers];
    float* dW[kChainMaxLayers]; long lddw[kChainMaxLayers];
    float* db[kChainMaxLayers];                                       // null entries allowed
    float* dX; long lddx;                                             // gradient w.r.t. X[0]; null to skip
    int L, M, rows_per_grp, n_groups, mask0, w_vec, dw_vec;
    unsigned long long* trace;                                        // diagnostics (npf_debug_set_trace)
};

template <int NSPLIT>
__global__ void __launch_bounds__(kFbThreads, 1) mlp_chain_bwd_kernel(ChainBwdParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_wfull, bar_wfree, bar_xfull, bar_dwdone, bar_mask, bar_z0[kCbBlocks], bar_z[kCbBlocks], bar_tfull[2],
        bar_tempty[2], bar_dwfull[2], bar_dwflushed[2];
    __shared__ uint32_t tmem_slot;
    __shared__ float s_db[128];

    constexpr uint32_t kHalf = 64u * 128u * 2u;                    // one bf16 64 x 128 image: 16 KB
    constexpr uint32_t kOp = (NSPLIT == 3 ? 2u : 1u) * kHalf;      // hi [+ lo]
    constexpr uint32_t kWTile = 128u * 128u * 2u;
    uint8_t* x_hi = smem_raw + kCbBlocks * kOp;
    uint8_t* w_hi = x_hi + kOp;
    uint8_t* w_lo = w_hi + kWTile;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    if (tid == 32) {
        mbar_init(&bar_wfull, kFbProdWarps * 32);
        mbar_init(&bar_wfree, 1);
        mbar_init(&bar_xfull, kFbProdWarps * 32);
        mbar_init(&bar_dwdone, 1);
        mbar_init(&bar_mask, kWsEpiWarps * 32);
        for (int i = 0; i < kCbBlocks; ++i) {
            mbar_init(&bar_z0[i], kFbProdWarps * 32);
            mbar_init(&bar_z[i], kWsEpiWarps * 32);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_tfull[i], 1);
            mbar_init(&bar_tempty[i], kWsEpiWarps * 32);
            mbar_init(&bar_dwfull[i], 1);
            mbar_init(&bar_dwflushed[i], kWsEpiWarps * 32);
        }
    }
    if (tid < 128) s_db[tid] = 0.f;
    const int L = p.L;
    const bool need_dx = p.dX != nullptr;
    const uint32_t pchunk = (uint32_t)(lane >> 1) & 7u;
    pdl_trigger();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;

    if (warp < kFbProdWarps) {
        // ------------------------------------------------------------------ producers
        const uint32_t woff = (uint32_t)(lane >> 4) * 16384u + (uint32_t)(warp * 8) * 128u + (uint32_t)(lane & 1) * 8u;
        const int prow = warp * 4;                                     // rows 4 w .. 4 w + 3 of a 64-row block
        const uint32_t psoff = (uint32_t)(lane >> 4) * 8192u + (uint32_t)prow * 128u + (uint32_t)(lane & 1) * 8u;
        const uint32_t rsw = (uint32_t)(prow & 7);
        float4 dbs = make_float4(0.f, 0.f, 0.f, 0.f);
        int li = 0, bi = 0;
        for (int grp = blockIdx.x, gi = 0; grp < p.n_groups; grp += gridDim.x, ++gi) {
            const int r_begin = grp * p.rows_per_grp, r_end = min(p.M, r_begin + p.rows_per_grp);
            const int n_blk = (r_end - r_begin + kF64Rows - 1) / kF64Rows;
            // weights of the last layer: parameters, may be fetched before the predecessor kernel has finished
            float4 wv[8];
            auto load_w = [&](int l) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float* g = p.W[l] + (long)(warp * 8 + i) * p.ldw[l] + lane * 4;
                    if (p.w_vec) wv[i] = __ldg(reinterpret_cast<const float4*>(g));
                    else wv[i] = make_float4(__ldg(g), __ldg(g + 1), __ldg(g + 2), __ldg(g + 3));
                }
            };
            auto store_w = [&]() {
                if (li > 0) mbar_wait(&bar_wfree, (uint32_t)(li - 1) & 1u);          // the previous layer's MMAs have read the weight buffer
#pragma unroll
                for (int i = 0; i < 8; ++i) cvt_store<NSPLIT>(wv[i], w_hi, w_lo, woff + (uint32_t)i * 128u + ((pchunk ^ (uint32_t)i) << 4), 0);
                fence_async_smem();
                mbar_arrive(&bar_wfull);
            };
            // the group's rows of a saved layer input -> L2, issued one whole layer ahead of their use (the X blocks are then
            // fetched from L2 while the previous block is multiplied instead of exposing a DRAM round trip per block)
            auto prefetch_x = [&](int l) {
                const char* base = reinterpret_cast<const char*>(p.X[l] + (long)r_begin * p.ldx[l]);
                const int lines = (r_end - r_begin) * 4;                                // 512 bytes per row
                for (int i = tid; i < lines; i += kFbProdWarps * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + ((long)(i >> 2) * p.ldx[l] * 4 + (i & 3) * 128)));
            };
            load_w(L - 1);
            if (gi == 0) pdl_wait();
            {   // the group's rows of the incoming gradient -> L2 before the block-by-block register loads below
                const char* base = reinterpret_cast<const char*>(p.dY + (long)r_begin * p.lddy);
                const int lines = (r_end - r_begin) * 4;
                for (int i = tid; i < lines; i += kFbProdWarps * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + ((long)(i >> 2) * p.lddy * 4 + (i & 3) * 128)));
            }
            prefetch_x(L - 1);
            if (bi > 0) mbar_wait(&bar_dwdone, (uint32_t)(bi - 1) & 1u);            // previous group: every MMA has read its images
            for (int j = 0; j < n_blk; ++j) {                                        // the chain's incoming gradient -> resident images
                const int row0 = r_begin + j * kF64Rows, rv = min(kF64Rows, r_end - row0);
                float4 yy[4];
                f64_load_rows(yy, p.dY + ((long)row0 + prow) * p.lddy + lane * 4, p.lddy, prow, rv);
                uint8_t* z_hi = smem_raw + (uint32_t)j * kOp;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    dbs.x += yy[i].x; dbs.y += yy[i].y; dbs.z += yy[i].z; dbs.w += yy[i].w;
                    cvt_store<NSPLIT>(yy[i], z_hi, z_hi + kHalf, psoff + (uint32_t)i * 128u + ((pchunk ^ (rsw + (uint32_t)i)) << 4), 0);
                }
                fence_async_smem();
                mbar_arrive(&bar_z0[j]);
            }
            for (int l = L - 1; l >= 0; --l, ++li) {
                if (l < L - 1) load_w(l);
                if (l > 0) prefetch_x(l - 1);
                float4 xx[4];
                f64_load_rows(xx, p.X[l] + ((long)r_begin + prow) * p.ldx[l] + lane * 4, p.ldx[l], prow, min(kF64Rows, r_end - r_begin));
                store_w();
                for (int j = 0; j < n_blk; ++j, ++bi) {
                    if (tid == 0) trace_ev(p.trace, 0, 1);
                    if (bi > 0) {
                        mbar_wait(&bar_dwdone, (uint32_t)(bi - 1) & 1u);             // the wgrad MMAs of the previous block have read the X stage
                        mbar_wait(&bar_mask, (uint32_t)(bi - 1) & 1u);               // and the epilogue has taken its relu mask
                    }
                    if (tid == 0) trace_ev(p.trace, 0, 2);
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        cvt_store<NSPLIT>(xx[i], x_hi, x_hi + kHalf, psoff + (uint32_t)i * 128u + ((pchunk ^ (rsw + (uint32_t)i)) << 4), 0);
                    fence_async_smem();
                    mbar_arrive(&bar_xfull);
                    if (tid == 0) trace_ev(p.trace, 0, 3);
                    if (j + 1 < n_blk) {
                        const int row0 = r_begin + (j + 1) * kF64Rows;
                        f64_load_rows(xx, p.X[l] + ((long)row0 + prow) * p.ldx[l] + lane * 4, p.ldx[l], prow, min(kF64Rows, r_end - row0));
                    }
                }
            }
        }
        if (p.db[L - 1]) {
            atomicAdd(&s_db[lane * 4 + 0], dbs.x); atomicAdd(&s_db[lane * 4 + 1], dbs.y);
            atomicAdd(&s_db[lane * 4 + 2], dbs.z); atomicAdd(&s_db[lane * 4 + 3], dbs.w);
            asm volatile("bar.sync 1, %0;" ::"n"(kFbProdWarps * 32) : "memory");
            if (tid < 128) atomicAdd(p.db[L - 1] + tid, s_db[tid]);
        }
    } else if (warp == kFbProdWarps) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc_dx = make_idesc(128, 64, 1, 0);
            const uint32_t idesc_dw = make_idesc(128, 128, 1, 1);
            const uint32_t sw_hi = smem_u32(w_hi), sw_lo = smem_u32(w_lo);
            const uint32_t sx_hi = smem_u32(x_hi), sx_lo = sx_hi + kHalf;
            // base descriptors built once (desc_adv steps through the k-slices): W^T MN-major view, X block MN-major
            const uint64_t dwt_h = make_desc_sw128(sw_hi, 16384, 1024), dwt_l = make_desc_sw128(sw_lo, 16384, 1024);
            const uint64_t dxm_h = make_desc_sw128(sx_hi, 8192, 1024), dxm_l = make_desc_sw128(sx_lo, 8192, 1024);
            int li = 0, bi = 0, ti = 0;
            for (int grp = blockIdx.x, gi = 0; grp < p.n_groups; grp += gridDim.x, ++gi) {
                const int r_begin = grp * p.rows_per_grp, r_end = min(p.M, r_begin + p.rows_per_grp);
                const int n_blk = (r_end - r_begin + kF64Rows - 1) / kF64Rows;
                for (int l = L - 1; l >= 0; --l, ++li) {
                    const int d = li & 1;
                    const uint32_t d_dw = tmem + 128u + (uint32_t)d * 128u;
                    mbar_wait(&bar_wfull, (uint32_t)li & 1u);
                    if (li >= 2) mbar_wait(&bar_dwflushed[d], (uint32_t)((li >> 1) - 1) & 1u);
                    for (int j = 0; j < n_blk; ++j, ++bi) {
                        trace_ev(p.trace, 1, 1);
                        mbar_wait(&bar_xfull, (uint32_t)bi & 1u);
                        trace_ev(p.trace, 1, 2);
                        if (l == L - 1) mbar_wait(&bar_z0[j], (uint32_t)gi & 1u);
                        else mbar_wait(&bar_z[j], (uint32_t)(gi * (L - 1) + (L - 2 - l)) & 1u);
                        tc_fence_after();
                        const uint32_t sz_hi = smem_u32(smem_raw + (uint32_t)j * kOp), sz_lo = sz_hi + kHalf;
                        const uint64_t dzk_h = make_desc_sw128(sz_hi, 16, 1024), dzk_l = make_desc_sw128(sz_lo, 16, 1024);          // K-major (data gradient)
                        const uint64_t dzm_h = make_desc_sw128(sz_hi, 8192, 1024), dzm_l = make_desc_sw128(sz_lo, 8192, 1024);      // MN-major (weight gradient)
                        if (l > 0 || need_dx) {
                            const int a = ti & 1;
                            mbar_wait(&bar_tempty[a], (uint32_t)((ti >> 1) & 1) ^ 1u);
                            tc_fence_after();
                            const uint32_t d_dx = tmem + (uint32_t)a * 64u;
#pragma unroll
                            for (int ks = 0; ks < 8; ++ks) {
                                const uint32_t bo = (uint32_t)(ks >> 2) * 8192u + (uint32_t)(ks & 3) * 32u;
                                const uint64_t a_h = desc_adv(dwt_h, ks * 2048u), b_h = desc_adv(dzk_h, bo);
                                umma_bf16(d_dx, a_h, b_h, idesc_dx, ks ? 1u : 0u);
                                if (NSPLIT == 3) {
                                    umma_bf16(d_dx, a_h, desc_adv(dzk_l, bo), idesc_dx, 1);
                                    umma_bf16(d_dx, desc_adv(dwt_l, ks * 2048u), b_h, idesc_dx, 1);
                                }
                            }
                            umma_commit(&bar_tfull[a]);
                            ++ti;
                        }
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            const uint32_t acc = (j | ks) ? 1u : 0u;
                            const uint64_t a_h = desc_adv(dzm_h, ks * 2048u), b_h = desc_adv(dxm_h, ks * 2048u);
                            umma_bf16(d_dw, a_h, b_h, idesc_dw, acc);
                            if (NSPLIT == 3) {
                                umma_bf16(d_dw, a_h, desc_adv(dxm_l, ks * 2048u), idesc_dw, 1);
                                umma_bf16(d_dw, desc_adv(dzm_l, ks * 2048u), b_h, idesc_dw, 1);
                            }
                        }
                        umma_commit(&bar_dwdone);
                        trace_ev(p.trace, 1, 3);
                    }
                    umma_commit(&bar_wfree);
                    umma_commit(&bar_dwfull[d]);
                }
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue: thread = column k, 32 rows of a block
        const int e = warp - kFbEpiWarp0;
        const int lane_base = 32 * (warp & 3);
        const int k = lane_base + lane;
        const int mh = (e >> 2) * 32;
        const int col_base = (e >> 2) * 64;
        const uint32_t xk_off = (uint32_t)(k >> 6) * 8192u + (uint32_t)(k & 7) * 2u, xk_chunk = (uint32_t)(k & 63) >> 3;
        pdl_wait();
        int li = 0, bi = 0, ti = 0;
        for (int grp = blockIdx.x, gi = 0; grp < p.n_groups; grp += gridDim.x, ++gi) {
            const int r_begin = grp * p.rows_per_grp, r_end = min(p.M, r_begin + p.rows_per_grp);
            const int n_blk = (r_end - r_begin + kF64Rows - 1) / kF64Rows;
            for (int l = L - 1; l >= 0; --l, ++li) {
                const int d = li & 1;
                const bool masked = l > 0 || p.mask0;
                float dbacc = 0.f;
                for (int j = 0; j < n_blk; ++j, ++bi) {
                    // Every block iteration waits for the block's wgrad MMAs (bar_dwdone) BEFORE it releases the X stage (bar_mask):
                    // the producers need both to stage the next block, so neither barrier can run two phases ahead of a waiter.
                    if (!(l > 0 || need_dx)) { mbar_wait(&bar_dwdone, (uint32_t)bi & 1u); mbar_arrive(&bar_mask); continue; }
                    const int a = ti & 1;
                    if (e == 0 && lane == 0) trace_ev(p.trace, 2, 1);
                    mbar_wait(&bar_tfull[a], (uint32_t)(ti >> 1) & 1u);
                    tc_fence_after();
                    if (e == 0 && lane == 0) trace_ev(p.trace, 2, 2);
                    uint32_t mbits = 0xFFFFFFFFu;
                    if (masked) {                  // relu mask of column k for the 32 rows, from the staged X_l block: bf16 > 0 <=> int16 > 0
                        mbits = 0u;
#pragma unroll
                        for (int i = 0; i < 32; ++i) {
                            const uint32_t m = (uint32_t)(mh + i);
                            const short xb = *reinterpret_cast<const short*>(x_hi + xk_off + m * 128u + ((xk_chunk ^ (m & 7u)) << 4));
                            mbits |= (xb > 0 ? 1u : 0u) << i;
                        }
                    }
                    float v[32];
                    {
                        float v0[16], v1[16];
                        tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(a * 64 + mh), v0);
                        tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(a * 64 + mh + 16), v1);
#pragma unroll
                        for (int i = 0; i < 16; ++i) { v[i] = v0[i]; v[16 + i] = v1[i]; }
                    }
                    tc_fence_before();
                    mbar_arrive(&bar_tempty[a]);
                    ++ti;
                    if (e == 0 && lane == 0) trace_ev(p.trace, 2, 3);
                    mbar_wait(&bar_dwdone, (uint32_t)bi & 1u);           // the wgrad MMAs of this block have read image j and the X stage
                    mbar_arrive(&bar_mask);
                    if (e == 0 && lane == 0) trace_ev(p.trace, 2, 4);
                    if (l > 0) {
                        uint8_t* z_hi = smem_raw + (uint32_t)j * kOp;
#pragma unroll
                        for (int i = 0; i < 32; ++i) {
                            const uint32_t m = (uint32_t)(mh + i);
                            const float val = ((mbits >> i) & 1u) ? v[i] : 0.f;
                            dbacc += val;
                            const uint32_t off = xk_off + m * 128u + ((xk_chunk ^ (m & 7u)) << 4);
                            const __nv_bfloat16 h = __float2bfloat16_rn(val);
                            *reinterpret_cast<__nv_bfloat16*>(z_hi + off) = h;
                            if (NSPLIT == 3) *reinterpret_cast<__nv_bfloat16*>(z_hi + kHalf + off) = __float2bfloat16_rn(val - __bfloat162float(h));
                        }
                        fence_async_smem();
                        mbar_arrive(&bar_z[j]);
                        if (e == 0 && lane == 0) trace_ev(p.trace, 2, 5);
                    } else {
                        const int row0 = r_begin + j * kF64Rows + mh;
#pragma unroll
                        for (int i = 0; i < 32; ++i) {
                            const int row = row0 + i;
                            if (row < r_end) p.dX[(long)row * p.lddx + k] = ((mbits >> i) & 1u) ? v[i] : 0.f;
                        }
                    }
                }
                if (l > 0 && p.db[l - 1]) atomicAdd(p.db[l - 1] + k, dbacc);
                // ---- flush of this layer's weight gradient: thread = row n of dW, 64 columns per warp
                mbar_wait(&bar_dwfull[d], (uint32_t)(li >> 1) & 1u);
                tc_fence_after();
#pragma unroll 1
                for (int ch = 0; ch < 4; ++ch) {
                    const int c0 = col_base + ch * 16;
                    float v[16];
                    tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(128 + d * 128 + c0), v);
                    float* dst = p.dW[l] + (long)k * p.lddw[l] + c0;
                    if (p.dw_vec) {
#pragma unroll
                        for (int i = 0; i < 16; i += 4) atomicAdd(reinterpret_cast<float4*>(dst + i), make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i) atomicAdd(dst + i, v[i]);
                    }
                }
                tc_fence_before();
                mbar_arrive(&bar_dwflushed[d]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

template <int NSPLIT>
static int launch_chain_bwd(ChainBwdParams& p, cudaStream_t st) {
    const size_t smem = (size_t)(NSPLIT == 3 ? 2 : 1) * (kCbBlocks + 1) * 16384 + 65536;
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(mlp_chain_bwd_kernel<NSPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            cudaGetLastError();
            return NPF_ENOTSUP;
        }
        attr = true;
    }
    const int max_rows = kCbBlocks * kF64Rows;
    int grid = (int)cdiv(p.M, max_rows);
    if (grid <= kNumSMs) {                       // one balanced row group per CTA
        long want = cdiv(p.M, kF64Rows);          // at least one full 64-row block per group
        if (want > kNumSMs) want = kNumSMs;
        p.rows_per_grp = (int)(cdiv(cdiv(p.M, want), 8) * 8);
        if (p.rows_per_grp > max_rows) p.rows_per_grp = max_rows;
        p.n_groups = (int)cdiv(p.M, p.rows_per_grp);
        grid = p.n_groups;
    } else {                                     // persistent CTAs walk 256-row groups
        p.rows_per_grp = max_rows;
        p.n_groups = grid;
        grid = kNumSMs;
    }
    launch_pdl(mlp_chain_bwd_kernel<NSPLIT>, dim3(grid), dim3(kFbThreads), smem, st, p);
    count_launch();
    return check_launch("mlp_chain_bwd_kernel");
}

// Backward of L consecutive Linear(128 -> 128) layers (ReLU between them); NPF_ENOTSUP for other shapes / alignments / fp32.
int mlp_chain_bwd_tc(const float* dY, int lddy, const float* const* X, const float* const* W, float* dX, int lddx, float* const* dW, float* const* db,
                     int L, int M, int mask0, int precision, cudaStream_t st) {
    if (L < 2 || L > kChainMaxLayers || M < 64 || precision == NPF_PREC_FP32) return NPF_ENOTSUP;
    if (lddy % 4 != 0 || !aligned16(dY) || (dX && (lddx % 4 != 0 || !aligned16(dX)))) return NPF_ENOTSUP;
    ChainBwdParams p{};
    p.dY = dY; p.lddy = lddy; p.dX = dX; p.lddx = lddx; p.L = L; p.M = M; p.mask0 = mask0;
    p.w_vec = 1; p.dw_vec = 1;
    p.trace = trace_buffer();
    for (int l = 0; l < L; ++l) {
        if (!aligned16(X[l])) return NPF_ENOTSUP;
        p.X[l] = X[l]; p.ldx[l] = 128; p.W[l] = W[l]; p.ldw[l] = 128; p.dW[l] = dW[l]; p.lddw[l] = 128; p.db[l] = db ? db[l] : nullptr;
        if (!aligned16(W[l])) p.w_vec = 0;
        if (!aligned16(dW[l])) p.dw_vec = 0;
    }
    return precision == NPF_PREC_BF16X3 ? launch_chain_bwd<3>(p, st) : launch_chain_bwd<1>(p, st);
}

// Chain of L Linear(128 -> 128) layers with bias / ReLU epilogues, all outputs stored (saved activations).  NPF_ENOTSUP unless
// every layer is 128 x 128, rows are 16-byte aligned and M fits one wave of 256-row CTAs.
template <int NSPLIT>
static int launch_chain(ChainParams& p, cudaStream_t st) {
    const size_t smem = (size_t)3 * (NSPLIT == 3 ? 2 : 1) * 32768 + (size_t)kWsEpiWarps * 32 * kWsScratchLd * sizeof(float);
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(mlp_chain_fwd_kernel<NSPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            cudaGetLastError();
            return NPF_ENOTSUP;
        }
        attr = true;
    }
    int grid = (int)cdiv(p.M, kChainRows);
    if (grid <= kNumSMs) {                       // one balanced block per CTA
        p.rows_per_cta = (int)(cdiv(cdiv(p.M, grid), 8) * 8);
        grid = (int)cdiv(p.M, p.rows_per_cta);
    } else {                                     // persistent CTAs walk 256-row blocks (weights re-staged per block and layer from L2)
        p.rows_per_cta = kChainRows;
        grid = kNumSMs;
    }
    launch_pdl(mlp_chain_fwd_kernel<NSPLIT>, dim3(grid), dim3(kWsThreads), smem, st, p);
    count_launch();
    return check_launch("mlp_chain_fwd_kernel");
}

int mlp_chain_fwd_tc(const float* X, int ldx, const float* const* W, const int* ldw, const float* const* b, float* const* Y, const int* ldy, int L, int M,
                     int relu_in, unsigned relu_mask, int precision, cudaStream_t st) {
    if (L < 2 || L > kChainMaxLayers || M < 1 || precision == NPF_PREC_FP32) return NPF_ENOTSUP;
    if (ldx % 4 != 0 || !aligned16(X)) return NPF_ENOTSUP;
    ChainParams p{};
    p.X = X; p.ldx = ldx; p.L = L; p.M = M; p.relu_in = relu_in; p.relu_mask = relu_mask;
    for (int l = 0; l < L; ++l) {
        if (ldw[l] % 4 != 0 || !aligned16(W[l]) || ldy[l] % 4 != 0 || !aligned16(Y[l])) return NPF_ENOTSUP;
        p.W[l] = W[l]; p.ldw[l] = ldw[l]; p.b[l] = b ? b[l] : nullptr; p.Y[l] = Y[l]; p.ldy[l] = ldy[l];
    }
    return precision == NPF_PREC_BF16X3 ? launch_chain<3>(p, st) : launch_chain<1>(p, st);
}

template <int NSPLIT>
static int launch_wg(TcWgParams& p, cudaStream_t st) {
    const size_t smem = (size_t)(NSPLIT == 3 ? 2 : 1) * (kWgRows * 128 + kWgRows * (p.K + (p.db ? 16 : 0))) * 2;
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(wgrad_tc_kernel<NSPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess) {
            cudaGetLastError();
            return NPF_ENOTSUP;
        }
        attr = true;
    }
    if (smem > 220 * 1024) return NPF_ENOTSUP;
    int per_sm = (int)((220 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 2) per_sm = 2;
    long ctas = (long)kNumSMs * per_sm;
    long rows = cdiv(cdiv(p.M, ctas), kWgRows) * kWgRows;
    if (rows < kWgRows) rows = kWgRows;
    p.rows_per_cta = rows;
    const long grid = cdiv(p.M, rows);
    wgrad_tc_kernel<NSPLIT><<<(unsigned)grid, 256, smem, st>>>(p);
    count_launch();
    return check_launch("wgrad_tc_kernel");
}

int linear_bwd_weight_tc(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, float* db, int* db_done, int M,
                         int K, int N, int flags, int precision, cudaStream_t st) {
    // MMA M dimension = N (rows of dW, padded to 128), MMA N dimension = K, reduction over the M rows
    if (N > 128 || N < 8 || N % 8 != 0 || !pow2(K) || K < 16 || K > 256) return NPF_ENOTSUP;
    TcWgParams p{};
    p.dY = dY; p.lddy = lddy; p.X = X; p.ldx = ldx; p.dW = dW; p.lddw = lddw;
    p.db = (db && K + 16 <= 256) ? db : nullptr;     // fused bias gradient needs MMA N = K + 16 <= 256
    *db_done = p.db != nullptr;
    p.M = M; p.N = N; p.K = K;
    p.relu_in = (flags & NPF_RELU_IN) ? 1 : 0;
    p.dy_vec = (lddy % 4 == 0) && aligned16(dY);
    p.x_vec = (ldx % 4 == 0) && aligned16(X);
    return precision == NPF_PREC_BF16X3 ? launch_wg<3>(p, st) : launch_wg<1>(p, st);
}

}  // namespace npf
