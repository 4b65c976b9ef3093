// One kernel per direction for the 1-D pre-activation residual block of the ConvCNP CNN (upstream npf/architectures/cnn.py:204-215,
// n_conv_layers = 1, Normalization = Identity: the constructor default of ConvCNP):
//
//     O[l, :] = sum_j wdw[:, j] (.) relu(X[l + j - p, :]) + bdw + X[l, :]        depthwise k taps (zero padding) + residual
//     Y[l, :] = Wpw . O[l, :] + bpw                                               pointwise 128 -> 128
//
// The unfused path runs this as npf_dwconv_fwd + npf_linear_fwd: O makes a round trip through HBM (write 50 MB, read 50 MB
// at config 2) between two launches.  Here a persistent CTA walks 128- or 96-row tiles of one task at a time:
//   * ONE thread issues a TMA bulk copy (cp.async.bulk, 1-D: the tile's rows and their +-p halo are contiguous in the
//     channel-last layout) of the raw fp32 rows into shared memory; rows outside the task are zero-filled (padding);
//   * 16 producer warps run the depthwise conv out of that raw tile (thread = 2 channels x 16 rows, the k taps of its two
//     channels in registers for the whole kernel), add bias + residual, and write O split into bf16 hi / lo straight into the
//     SWIZZLE_128B K-major A-operand image (optionally also as fp32 rows to HBM when the caller wants O saved);
//   * 1 MMA warp multiplies by the once-staged pointwise weights (tcgen05, hi.hi + hi.lo + lo.hi, accumulator double-
//     buffered in TMEM).  The product is issued TRANSPOSED, Y^T = Wpw . O^T (both images are 128-column K-major, so they just swap
//     roles): TMEM lane = output channel, column = tile row, and the 8 epilogue warps store 32 consecutive channels of a row straight
//     from their tcgen05.ld registers -- no shared-memory transpose.  With the rows as the N extent of the MMA the tile may be 96 rows
//     high (chosen when it leaves fewer rows on the busiest CTA).
// HBM sees X once (+ 2p / 128 halo re-reads out of L2) and Y once.
#include <type_traits>

#include "tc_common.cuh"

namespace npf {

constexpr int kRbProd = 16;
constexpr int kRbMmaWarp = kRbProd;
constexpr int kRbEpiWarp0 = kRbProd + 1;
constexpr int kRbEpi = 8;
constexpr int kRbThreads = (kRbEpiWarp0 + kRbEpi) * 32;       // 800
constexpr int kRbMaxPad = 9;                                   // k <= 19
constexpr int kRbRawRows = 128 + 2 * kRbMaxPad;                // 146
constexpr uint32_t kRbTile = 128u * 128u * 2u;                 // one bf16 128 x 128 image: 32 KB

struct RbFwdParams {
    const float* X;      // [B, L, 128]
    const float* wdw;    // [128, k]
    const float* bdw;    // [128] or null
    const float* wpw;    // [128, 128]
    const float* bpw;    // [128] or null
    float* O;            // [B, L, 128] or null
    float* Y;            // [B, L, 128]
    int B, L, n_lt, n_tiles;
    unsigned long long* trace;      // diagnostics (npf_debug_set_trace)
};

__device__ __forceinline__ uint64_t rb_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return make_desc(saddr, lbo_bytes, sbo_bytes) | (2ull << 61);
}
// byte offset of element (row, col) of a [128 x 128] bf16 SWIZZLE_128B K-major image (two 64-column atoms of 16 KB)
__device__ __forceinline__ uint32_t rb_img_off(uint32_t row, uint32_t col) {
    return (col >> 6) * 16384u + row * 128u + ((((col & 63u) >> 3) ^ (row & 7u)) << 4) + (col & 7u) * 2u;
}
__device__ __forceinline__ void rb_prod_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kRbProd * 32) : "memory"); }

// TR = rows per tile: 128, or (the rows are the N extent of the MMA) 96 when that splits the tiles more
// evenly over the CTAs -- config 2: 768 tiles of 128 rows are 6 rounds on 148 SMs (768 rows on the critical CTA), 1024 tiles of 96 are 7 (672).
template <int KW, int TR>
__global__ void __launch_bounds__(kRbThreads, 1) resblock1d_fwd_kernel(RbFwdParams p) {
    constexpr int P = KW / 2;
    constexpr int RAW = TR + 2 * P;                             // raw rows of a tile: row i <-> position l0 - P + i
    constexpr int RPT = TR / 8;                                 // rows per producer thread (8 row groups x 2 channel halves = 16 warps)
    static_assert(TR == 128 || TR == 96, "tile rows");
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_raw, bar_afull, bar_aempty, bar_tfull[2], bar_tempty[2];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float s_bias[128];

    uint8_t* a_hi = smem_raw;                                   // O image (B operand of Y^T = Wpw . O^T)
    uint8_t* a_lo = a_hi + kRbTile;
    uint8_t* b_hi = smem_raw + 2 * kRbTile;                     // pointwise weights (A operand)
    uint8_t* b_lo = b_hi + kRbTile;
    float* raw = reinterpret_cast<float*>(smem_raw + 4 * kRbTile);          // [RAW][128] fp32

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    if (tid == 32) {
        mbar_init(&bar_raw, 1);
        mbar_init(&bar_afull, kRbProd * 32);
        mbar_init(&bar_aempty, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_tfull[i], 1);
            mbar_init(&bar_tempty[i], kRbEpi * 32);
        }
    }
    if (tid < 128) s_bias[tid] = p.bpw ? __ldg(p.bpw + tid) : 0.f;
    // contiguous, balanced tile ranges (tiles of one task stay together: halo rows come out of L2)
    const int per = p.n_tiles / (int)gridDim.x, rem = p.n_tiles - per * (int)gridDim.x;
    const int g0 = (int)blockIdx.x * per + min((int)blockIdx.x, rem), g1 = g0 + per + ((int)blockIdx.x < rem ? 1 : 0);
    pdl_trigger();

    // pointwise weights [128 x 128] fp32 row-major, staged once per CTA by the 16 producer warps (parameters: before pdl_wait)
    if (warp < kRbProd) {
        const uint32_t pchunk = (uint32_t)(lane >> 1) & 7u;
        const uint32_t psoff = (uint32_t)(lane >> 4) * 16384u + (uint32_t)(warp * 8) * 128u + (uint32_t)(lane & 1) * 8u;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(p.wpw + (long)(warp * 8 + i) * 128) + lane);
            const uint32_t off = psoff + (uint32_t)i * 128u + ((pchunk ^ (uint32_t)i) << 4);
            const uint32_t h01 = pack_bf16(v.x, v.y), h23 = pack_bf16(v.z, v.w);
            *reinterpret_cast<uint2*>(b_hi + off) = make_uint2(h01, h23);
            *reinterpret_cast<uint2*>(b_lo + off) = make_uint2(pack_bf16(v.x - __uint_as_float(h01 << 16), v.y - __uint_as_float(h01 & 0xFFFF0000u)),
                                                                 pack_bf16(v.z - __uint_as_float(h23 << 16), v.w - __uint_as_float(h23 & 0xFFFF0000u)));
        }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    pdl_wait();

    if (warp < kRbProd) {
        // ------------------------------------------------------------------ producers: raw tile -> depthwise -> O image
        const int cp = lane + 32 * (warp & 1);                   // channel pair: channels 2 cp, 2 cp + 1
        const int rg = warp >> 1;                                // rows 16 rg .. 16 rg + 15 of the tile
        float2 w2[KW];                                            // taps of the two channels, packed for FFMA2 (fp32 x 2 per instruction)
#pragma unroll
        for (int j = 0; j < KW; ++j) w2[j] = make_float2(__ldg(p.wdw + (2 * cp) * KW + j), __ldg(p.wdw + (2 * cp + 1) * KW + j));
        const float2 bd2 = make_float2(p.bdw ? __ldg(p.bdw + 2 * cp) : 0.f, p.bdw ? __ldg(p.bdw + 2 * cp + 1) : 0.f);

        // raw rows of tile g: TMA bulk copy of the in-task part, zero fill of the rest (issued when the raw buffer is free)
        auto fetch = [&](int g) {
            const int b = g / p.n_lt, l0 = (g - b * p.n_lt) * TR;
            const int s0 = max(0, l0 - P), e0 = min(p.L, l0 + TR + P);
            const int d0 = s0 - (l0 - P), d1 = d0 + (e0 - s0);                     // raw rows [d0, d1) come from HBM
            for (int i = tid; i < (d0 + (RAW - d1)) * 32; i += kRbProd * 32) {      // 32 float4 per row
                const int r = i >> 5, rr = r < d0 ? r : d1 + (r - d0);
                reinterpret_cast<float4*>(raw + rr * 128)[i & 31] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (tid == 0) {
                fence_async_smem();                       // the generic reads of the previous tile are ordered before the async writes
                const uint32_t bytes = (uint32_t)(e0 - s0) * 512u;
                mbar_expect_tx(&bar_raw, bytes);
                bulk_g2s(raw + d0 * 128, p.X + ((long)b * p.L + s0) * 128, bytes, &bar_raw);
            }
        };
        if (g0 < g1) fetch(g0);
        int it = 0;
        for (int g = g0; g < g1; ++g, ++it) {
            const int b = g / p.n_lt, l0 = (g - b * p.n_lt) * TR;
            const int rows_ok = min(TR, p.L - l0);
            if (tid == 0) trace_ev(p.trace, 0, 1);
            mbar_wait(&bar_raw, (uint32_t)it & 1u);
            rb_prod_sync();                                       // the zero-filled rows of this tile are visible to every producer
            if (tid == 0) trace_ev(p.trace, 0, 2);
            float2 acc2[RPT];
#pragma unroll
            for (int o = 0; o < RPT; ++o) acc2[o] = bd2;
            const float* rp = raw + (RPT * rg) * 128 + 2 * cp;
#pragma unroll
            for (int i = 0; i < RPT + 2 * P; ++i) {               // raw row RPT rg + i feeds outputs o = i - j, tap j
                const float2 v = *reinterpret_cast<const float2*>(rp + i * 128);
                const float2 r = make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f));
#pragma unroll
                for (int j = 0; j < KW; ++j) {
                    const int o = i - j;
                    if (o >= 0 && o < RPT) acc2[o] = __ffma2_rn(w2[j], r, acc2[o]);
                }
                if (i - P >= 0 && i - P < RPT) acc2[i - P] = __fadd2_rn(acc2[i - P], v);         // residual: the block input itself
            }
            float a0[RPT], a1[RPT];
#pragma unroll
            for (int o = 0; o < RPT; ++o) { a0[o] = acc2[o].x; a1[o] = acc2[o].y; }
            if (tid == 0) trace_ev(p.trace, 0, 3);
            rb_prod_sync();                                       // every producer has finished reading the raw tile
            if (g + 1 < g1) fetch(g + 1);
            if (tid == 0) trace_ev(p.trace, 0, 4);
            if (p.O) {                                            // O saved for a backward pass that does not recompute it
#pragma unroll
                for (int o = 0; o < RPT; ++o) {
                    const int row = RPT * rg + o;
                    if (row < rows_ok) *reinterpret_cast<float2*>(p.O + ((long)b * p.L + l0 + row) * 128 + 2 * cp) = make_float2(a0[o], a1[o]);
                }
            }
            if (it > 0) mbar_wait(&bar_aempty, (uint32_t)(it - 1) & 1u);        // the MMAs of the previous tile have read the image
            if (tid == 0) trace_ev(p.trace, 0, 5);
#pragma unroll
            for (int o = 0; o < RPT; ++o) {
                const uint32_t row = (uint32_t)(RPT * rg + o);
                const uint32_t off = rb_img_off(row, (uint32_t)(2 * cp));
                const uint32_t h = pack_bf16(a0[o], a1[o]);
                *reinterpret_cast<uint32_t*>(a_hi + off) = h;
                *reinterpret_cast<uint32_t*>(a_lo + off) = pack_bf16(a0[o] - __uint_as_float(h << 16), a1[o] - __uint_as_float(h & 0xFFFF0000u));
            }
            fence_async_smem();
            mbar_arrive(&bar_afull);
            if (tid == 0) trace_ev(p.trace, 0, 6);
        }
    } else if (warp == kRbMmaWarp) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc(128, TR, 0, 0);
            const uint64_t da_h = rb_desc_sw128(smem_u32(a_hi), 16, 1024), da_l = rb_desc_sw128(smem_u32(a_lo), 16, 1024);
            const uint64_t db_h = rb_desc_sw128(smem_u32(b_hi), 16, 1024), db_l = rb_desc_sw128(smem_u32(b_lo), 16, 1024);
            int it = 0;
            for (int g = g0; g < g1; ++g, ++it) {
                const int t = it & 1;
                trace_ev(p.trace, 1, 1);
                mbar_wait(&bar_afull, (uint32_t)it & 1u);
                mbar_wait(&bar_tempty[t], (uint32_t)((it >> 1) & 1) ^ 1u);
                tc_fence_after();
                trace_ev(p.trace, 1, 2);
                const uint32_t d = tmem + (uint32_t)t * 128u;
#pragma unroll
                for (int ks = 0; ks < 8; ++ks) {
                    const uint32_t ao = (uint32_t)(ks >> 2) * 16384u + (uint32_t)(ks & 3) * 32u;
                    const uint64_t a_h = desc_adv(da_h, ao), b_h = desc_adv(db_h, ao);
                    // Y^T = Wpw . O^T: both images are 128 x 128 K-major, so swapping the operands transposes the product
                    umma_bf16(d, b_h, a_h, idesc, ks ? 1u : 0u);
                    umma_bf16(d, desc_adv(db_l, ao), a_h, idesc, 1);
                    umma_bf16(d, b_h, desc_adv(da_l, ao), idesc, 1);
                }
                umma_commit(&bar_aempty);
                umma_commit(&bar_tfull[t]);
                trace_ev(p.trace, 1, 3);
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue: TMEM -> + bias -> rows of Y
        // TMEM lane = output channel, columns = the tile's rows: a warp stores 32 consecutive channels of one row
        const int e = warp - kRbEpiWarp0;
        const int lane_base = 32 * (warp & 3);
        int it = 0;
        for (int g = g0; g < g1; ++g, ++it) {
            const int t = it & 1;
            const int b = g / p.n_lt, l0 = (g - b * p.n_lt) * TR;
            if (e == 0 && lane == 0) trace_ev(p.trace, 2, 1);
            mbar_wait(&bar_tfull[t], (uint32_t)(it >> 1) & 1u);
            tc_fence_after();
            if (e == 0 && lane == 0) trace_ev(p.trace, 2, 2);
            const float bias = s_bias[lane_base + lane];
            const int rows_tile = min(TR, p.L - l0);
            float* yc = p.Y + ((long)b * p.L + l0) * 128 + lane_base + lane;
#pragma unroll 1
            for (int ch = 0; ch < TR / 32; ++ch) {              // this warp's half of the tile's rows, 16 at a time
                const int r0 = (e >> 2) * (TR / 2) + ch * 16;
                float v[16];
                tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(t * 128 + r0), v);
                if (ch == TR / 32 - 1) {
                    tc_fence_before();
                    mbar_arrive(&bar_tempty[t]);
                }
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (r0 + j < rows_tile) yc[(long)(r0 + j) * 128] = v[j] + bias;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

template <int KW, int TR>
static int launch_rb_fwd(RbFwdParams& p, cudaStream_t st) {
    const size_t smem = (size_t)4 * kRbTile + (size_t)kRbRawRows * 512;
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(resblock1d_fwd_kernel<KW, TR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            cudaGetLastError();
            return NPF_ENOTSUP;
        }
        attr = true;
    }
    const int grid = p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs;
    launch_pdl(resblock1d_fwd_kernel<KW, TR>, dim3(grid), dim3(kRbThreads), smem, st, p);
    count_launch();
    return check_launch("resblock1d_fwd_kernel");
}

// ------------------------------------------------------------------------------------------------------------------
// Backward of the same block in ONE kernel, with O RECOMPUTED (the forward then never writes it):
//     dO = dY . Wpw          dWpw += dY^T . O        dbpw += colsum(dY)
//     dX[m] = dO[m] + relu'(X[m]) sum_j wdw[j] dO[m - j + p]      dwdw[j] += sum_l dO[l] relu(X[l + j - p])      dbdw += colsum(dO)
// against npf_linear_bwd + npf_dwconv_bwd: dO (50 MB written + read at config 2) and the saved O (50 MB read, and its write
// in the forward) disappear; HBM sees dY and X once (+ halo re-reads out of L2) and dX once.
// Tiles of 64 rows of one task = 48 interior rows + the +-p halo the transposed depthwise conv needs.  As in
// linear_bwd_fused64_kernel the data gradient is computed TRANSPOSED,  dO^T[k, m] = sum_n Wpw[n, k] dY[m, n]  (A = Wpw^T: MN-major
// view of the row-staged weights, B = dY tile K-major, N = 64), so an epilogue thread owns ONE channel k and the tile's rows sit
// in its registers: the depthwise transposed conv, the filter gradient and the relu mask are register arithmetic along the row
// axis with X read from the raw tile in shared memory -- no exchange between threads.  dWpw accumulates in TMEM over the CTA's
// tiles (A = dY^T, B = O: MN-major views; O rows outside the interior are zero so that every row counts once).
// Roles: loader warp (TMA bulk copies of the raw dY / X tiles, zero fill outside the task), 16 producer warps (dY raw -> image;
// O recomputed from raw X for the 48 interior rows -> image, whose halo rows are zeroed once), 1 MMA warp, 8 epilogue warps.
// Wpw^T is the TMEM-resident A operand of the data-gradient product (written once per CTA with tcgen05.st): the 64 KB its
// shared-memory images would take hold a third raw X and a second raw dY buffer (the epilogue of tile i still reads X(i) while
// tiles i + 1, i + 2 are prepared).
// ------------------------------------------------------------------------------------------------------------------
constexpr int kRwRows = 64;
constexpr int kRwInt = 48;                                      // interior rows per tile (k = 11: 48 + 2 * 5 = 58 <= 64)
constexpr int kRwThreads = (kRbEpiWarp0 + kRbEpi + 1) * 32;   // 832: producers + MMA + epilogue + loader warp
constexpr uint32_t kRwHalf = 64u * 128u * 2u;                   // one bf16 64 x 128 image: 16 KB
constexpr int kRwNX = 3, kRwNY = 2;                             // raw X / raw dY buffers in flight

struct RbBwdParams {
    const float* dY; const float* X; const float* wdw; const float* bdw; const float* wpw;
    float* dX; float* dWdw; float* dbdw; float* dWpw; float* dbpw;
    int B, L, n_lt, n_tiles;
    unsigned long long* trace;
};

// 32 lanes x 8 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// the same load without the wait (several in flight), and the wait
__device__ __forceinline__ void tmem_ld8_issue(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// byte offset of element (row m, col c) of a [64 x 128] bf16 SWIZZLE_128B image (two 64-column atoms of 8 KB)
__device__ __forceinline__ uint32_t rw_img_off(uint32_t m, uint32_t c) {
    return (c >> 6) * 8192u + m * 128u + ((((c & 63u) >> 3) ^ (m & 7u)) << 4) + (c & 7u) * 2u;
}

// NE = 8 epilogue warps: two row groups of 24 interior rows, two 12-row sub-passes each
template <int KW, int NE>
__global__ void __launch_bounds__(kRwThreads, 1) resblock1d_bwd_kernel(RbBwdParams p) {
    constexpr int P = KW / 2;
    constexpr int kRwLoadWarp = kRbEpiWarp0 + NE;
    constexpr int NP = 2;                                       // sub-passes per epilogue thread
    constexpr int RP = 12;                                      // interior rows per sub-pass
    static_assert(NE == kRbEpi, "epilogue warps");
    static_assert((NE / 4) * NP * RP == kRwInt, "row groups must tile the interior");
    static_assert(kRwInt + 2 * P <= kRwRows, "tile too small for the halo");
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_y[2], bar_yfree[2], bar_x[3], bar_xfree[3], bar_afull, bar_aempty, bar_tfull[2], bar_tempty[2], bar_dwfull;
    __shared__ uint32_t tmem_slot;
    __shared__ float s_db[128];

    constexpr int NX = kRwNX, NY = kRwNY;
    constexpr int TILE = kRwRows * 128;                         // floats of one raw tile (32 KB)
    uint8_t* y_hi = smem_raw;                                   // dY image: hi 16 KB | lo 16 KB
    uint8_t* o_hi = smem_raw + 2 * kRwHalf;                     // O image
    float* rawY = reinterpret_cast<float*>(smem_raw + 4 * kRwHalf);   // NY x [64][128]
    float* rawX = rawY + NY * TILE;                                   // NX x [64][128]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_slot, 512);
    if (tid == 32) {
        mbar_init(&bar_afull, kRbProd * 32);
        mbar_init(&bar_aempty, 1);
        mbar_init(&bar_dwfull, 1);
        for (int i = 0; i < 3; ++i) {
            mbar_init(&bar_x[i], 1);
            mbar_init(&bar_xfree[i], kRbProd * 32 + NE * 32);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_y[i], 1);
            mbar_init(&bar_yfree[i], kRbProd * 32);
            mbar_init(&bar_tfull[i], 1);
            mbar_init(&bar_tempty[i], NE * 32);
        }
    }
    if (tid < 128) s_db[tid] = 0.f;
    for (int i = tid; i < (int)(2 * kRwHalf / 16); i += (int)blockDim.x)      // O image: its halo rows are never written again and must read as zero
        reinterpret_cast<uint4*>(o_hi)[i] = make_uint4(0u, 0u, 0u, 0u);
    const int per = p.n_tiles / (int)gridDim.x, rem = p.n_tiles - per * (int)gridDim.x;
    const int g0 = (int)blockIdx.x * per + min((int)blockIdx.x, rem), g1 = g0 + per + ((int)blockIdx.x < rem ? 1 : 0);
    pdl_trigger();
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    // Wpw^T as the TMEM-resident A operand of dO^T = Wpw^T . dY^T: lane k = input channel k holds column k of Wpw [n, k] (K-major over
    // the output channel n, two consecutive n per 32-bit column), hi at columns [256, 320), lo at [320, 384)
    if (warp < 4) {
        const float* wc = p.wpw + 32 * warp + lane;
        const uint32_t tw = tmem + ((uint32_t)(32 * warp) << 16) + 256u;
#pragma unroll 1
        for (int cc = 0; cc < 4; ++cc) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float v0 = __ldg(wc + (long)(32 * cc + 2 * i) * 128), v1 = __ldg(wc + (long)(32 * cc + 2 * i + 1) * 128);
                const uint32_t h = pack_bf16(v0, v1);
                hi[i] = h;
                lo[i] = pack_bf16(v0 - __uint_as_float(h << 16), v1 - __uint_as_float(h & 0xFFFF0000u));
            }
            tmem_st16(tw + (uint32_t)(cc * 16), hi);
            tmem_st16(tw + 64u + (uint32_t)(cc * 16), lo);
        }
        tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_wait();

    if (warp == kRwLoadWarp) {
        // ------------------------------------------------------------------ loader: raw tiles by TMA, zero rows outside the task
        auto fetch = [&](const float* src, float* dst, uint64_t* bar, int g) {
            const int b = g / p.n_lt, pos0 = (g - b * p.n_lt) * kRwInt - P;          // position of tile row 0
            const int s0 = max(0, pos0), e0 = min(p.L, pos0 + kRwRows);
            const int d0 = s0 - pos0, n = max(0, e0 - s0);
            for (int i = lane; i < (kRwRows - n) * 32; i += 32) {
                const int r = i >> 5, rr = r < d0 ? r : d0 + n + (r - d0);
                reinterpret_cast<float4*>(dst + rr * 128)[i & 31] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            __syncwarp();
            if (lane == 0) {
                fence_async_smem();
                const uint32_t bytes = (uint32_t)n * 512u;
                mbar_expect_tx(bar, bytes);
                if (bytes) bulk_g2s(dst + d0 * 128, src + ((long)b * p.L + s0) * 128, bytes, bar);
            }
            __syncwarp();
        };
        const int nt = g1 - g0;
        if (nt > 0) { fetch(p.X, rawX, &bar_x[0], g0); fetch(p.dY, rawY, &bar_y[0], g0); }
        for (int j = 1; j < NX && j < nt; ++j) fetch(p.X, rawX + j * TILE, &bar_x[j], g0 + j);
        for (int j = 1; j < NY && j < nt; ++j) fetch(p.dY, rawY + j * TILE, &bar_y[j], g0 + j);
        int xs = 0, ys = 0;
        uint32_t xph = 0, yph = 0;
        for (int it = 0; it < nt; ++it) {
            if (it + NY < nt) {                                  // raw dY of tile it consumed by the producers -> dY of tile it + NY
                mbar_wait(&bar_yfree[ys], yph);
                fetch(p.dY, rawY + ys * TILE, &bar_y[ys], g0 + it + NY);
            }
            if (it + NX < nt) {                                  // raw X buffer of tile it released by producers AND epilogue -> tile it + NX
                mbar_wait(&bar_xfree[xs], xph);
                fetch(p.X, rawX + xs * TILE, &bar_x[xs], g0 + it + NX);
            }
            if (++xs == NX) { xs = 0; xph ^= 1u; }
            if (++ys == NY) { ys = 0; yph ^= 1u; }
        }
    } else if (warp < kRbProd) {
        // ------------------------------------------------------------------ producers
        const int cp = lane + 32 * (warp & 1);                   // O: channels 2 cp, 2 cp + 1 ...
        const int rg = warp >> 1;                                // ... INTERIOR rows P + RO rg .. P + RO rg + RO - 1 (the image's halo rows stay zero)
        constexpr int RO = kRwInt / (kRbProd / 2);               // 6
        float2 w2[KW];
#pragma unroll
        for (int j = 0; j < KW; ++j) w2[j] = make_float2(__ldg(p.wdw + (2 * cp) * KW + j), __ldg(p.wdw + (2 * cp + 1) * KW + j));
        const float2 bd2 = make_float2(p.bdw ? __ldg(p.bdw + 2 * cp) : 0.f, p.bdw ? __ldg(p.bdw + 2 * cp + 1) : 0.f);
        const int prow = warp * 4;                               // dY: rows 4 w .. 4 w + 3, float4 column lane
        const uint32_t pchunk = (uint32_t)(lane >> 1) & 7u;
        const uint32_t psoff = (uint32_t)(lane >> 4) * 8192u + (uint32_t)prow * 128u + (uint32_t)(lane & 1) * 8u;
        const uint32_t rsw = (uint32_t)(prow & 7);
        float4 dbs = make_float4(0.f, 0.f, 0.f, 0.f);
        int it = 0, xs = 0, ys = 0;
        uint32_t xph = 0, yph = 0;
        for (int g = g0; g < g1; ++g, ++it) {
            const int s = xs;
            const float* rx = rawX + s * TILE;
            const float* ry = rawY + ys * TILE;
            // ---- O rows 8 rg .. 8 rg + 7 of channels 2 cp, 2 cp + 1 from the raw X tile (registers only)
            if (tid == 0) trace_ev(p.trace, 0, 1);
            mbar_wait(&bar_x[s], xph);
            if (tid == 0) trace_ev(p.trace, 0, 2);
            float2 acc2[RO];
#pragma unroll
            for (int o = 0; o < RO; ++o) acc2[o] = bd2;
            const float* rxp = rx + (RO * rg) * 128 + 2 * cp;     // tile row RO rg + i feeds outputs o = i - j (rows RO rg .. RO rg + RO + 2 P - 1 <= 57)
#pragma unroll
            for (int i = 0; i < RO + 2 * P; ++i) {
                const float2 v = *reinterpret_cast<const float2*>(rxp + i * 128);
                const float2 r = make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f));
#pragma unroll
                for (int j = 0; j < KW; ++j) {
                    const int o = i - j;
                    if (o >= 0 && o < RO) acc2[o] = __ffma2_rn(w2[j], r, acc2[o]);
                }
                if (i - P >= 0 && i - P < RO) acc2[i - P] = __fadd2_rn(acc2[i - P], v);
            }
            float a0[RO], a1[RO];
#pragma unroll
            for (int o = 0; o < RO; ++o) { a0[o] = acc2[o].x; a1[o] = acc2[o].y; }
            mbar_arrive(&bar_xfree[s]);                          // the producers' reads of this raw X buffer are done
            if (tid == 0) trace_ev(p.trace, 0, 3);
            // ---- images: wait for the previous tile's MMAs, then dY raw -> image and O -> image
            mbar_wait(&bar_y[ys], yph);
            if (it > 0) mbar_wait(&bar_aempty, (uint32_t)(it - 1) & 1u);
            if (tid == 0) trace_ev(p.trace, 0, 4);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = prow + i;
                const float4 v = *reinterpret_cast<const float4*>(ry + r * 128 + lane * 4);
                if (r >= P && r < P + kRwInt) { dbs.x += v.x; dbs.y += v.y; dbs.z += v.z; dbs.w += v.w; }
                const uint32_t off = psoff + (uint32_t)i * 128u + ((pchunk ^ (rsw + (uint32_t)i)) << 4);
                const uint32_t h01 = pack_bf16(v.x, v.y), h23 = pack_bf16(v.z, v.w);
                *reinterpret_cast<uint2*>(y_hi + off) = make_uint2(h01, h23);
                *reinterpret_cast<uint2*>(y_hi + kRwHalf + off) =
                    make_uint2(pack_bf16(v.x - __uint_as_float(h01 << 16), v.y - __uint_as_float(h01 & 0xFFFF0000u)),
                               pack_bf16(v.z - __uint_as_float(h23 << 16), v.w - __uint_as_float(h23 & 0xFFFF0000u)));
            }
            mbar_arrive(&bar_yfree[ys]);
#pragma unroll
            for (int o = 0; o < RO; ++o) {
                const uint32_t row = (uint32_t)(P + RO * rg + o);
                const float v0 = a0[o], v1 = a1[o];
                const uint32_t off = rw_img_off(row, (uint32_t)(2 * cp));
                const uint32_t h = pack_bf16(v0, v1);
                *reinterpret_cast<uint32_t*>(o_hi + off) = h;
                *reinterpret_cast<uint32_t*>(o_hi + kRwHalf + off) = pack_bf16(v0 - __uint_as_float(h << 16), v1 - __uint_as_float(h & 0xFFFF0000u));
            }
            fence_async_smem();
            mbar_arrive(&bar_afull);
            if (tid == 0) trace_ev(p.trace, 0, 5);
            if (++xs == NX) { xs = 0; xph ^= 1u; }
            if (++ys == NY) { ys = 0; yph ^= 1u; }
        }
        if (p.dbpw) {
            atomicAdd(&s_db[lane * 4 + 0], dbs.x); atomicAdd(&s_db[lane * 4 + 1], dbs.y);
            atomicAdd(&s_db[lane * 4 + 2], dbs.z); atomicAdd(&s_db[lane * 4 + 3], dbs.w);
            rb_prod_sync();
            if (tid < 128) atomicAdd(p.dbpw + tid, s_db[tid]);
        }
    } else if (warp == kRbMmaWarp) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc_dx_ts = make_idesc(128, 64, 0, 0);   // A = Wpw^T stored K-major in TMEM, B = dY tile (K-major), D = dO^T [k x m]
            const uint32_t idesc_dw = make_idesc(128, 128, 1, 1);     // A = dY^T, B = O: MN-major views (reduction over the tile's rows)
            const uint32_t sy_hi = smem_u32(y_hi), sy_lo = sy_hi + kRwHalf, so_hi = smem_u32(o_hi), so_lo = so_hi + kRwHalf;
            // base descriptors, built once: dY K-major (data gradient), dY^T / O MN-major (weight gradient)
            const uint64_t dyk_h = rb_desc_sw128(sy_hi, 16, 1024), dyk_l = rb_desc_sw128(sy_lo, 16, 1024);
            const uint64_t dym_h = rb_desc_sw128(sy_hi, 8192, 1024), dym_l = rb_desc_sw128(sy_lo, 8192, 1024);
            const uint64_t dom_h = rb_desc_sw128(so_hi, 8192, 1024), dom_l = rb_desc_sw128(so_lo, 8192, 1024);
            const uint32_t d_dw = tmem + 128u;
            int it = 0;
            for (int g = g0; g < g1; ++g, ++it) {
                const int a = it & 1;
                trace_ev(p.trace, 1, 1);
                mbar_wait(&bar_afull, (uint32_t)it & 1u);
                trace_ev(p.trace, 1, 2);
                mbar_wait(&bar_tempty[a], (uint32_t)((it >> 1) & 1) ^ 1u);
                tc_fence_after();
                trace_ev(p.trace, 1, 3);
                const uint32_t d_dx = tmem + (uint32_t)a * 64u;
#pragma unroll
                for (int ks = 0; ks < 8; ++ks) {
                    const uint32_t bo = (uint32_t)(ks >> 2) * 8192u + (uint32_t)(ks & 3) * 32u;
                    const uint64_t b_h = desc_adv(dyk_h, bo);
                    const uint32_t ta = tmem + 256u + (uint32_t)ks * 8u;    // A = Wpw^T from TMEM (8 columns per 16-wide slice of the reduction over n)
                    umma_bf16_ts(d_dx, ta, b_h, idesc_dx_ts, ks ? 1u : 0u);
                    umma_bf16_ts(d_dx, ta, desc_adv(dyk_l, bo), idesc_dx_ts, 1);
                    umma_bf16_ts(d_dx, ta + 64u, b_h, idesc_dx_ts, 1);
                }
                umma_commit(&bar_tfull[a]);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const uint32_t acc = (it | ks) ? 1u : 0u;
                    const uint64_t a_h = desc_adv(dym_h, ks * 2048u), b_h = desc_adv(dom_h, ks * 2048u);
                    umma_bf16(d_dw, a_h, b_h, idesc_dw, acc);
                    umma_bf16(d_dw, a_h, desc_adv(dom_l, ks * 2048u), idesc_dw, 1);
                    umma_bf16(d_dw, desc_adv(dym_l, ks * 2048u), b_h, idesc_dw, 1);
                }
                umma_commit(&bar_aempty);
                trace_ev(p.trace, 1, 4);
            }
            umma_commit(&bar_dwfull);
        }
    } else {
        // ------------------------------------------------------------------ epilogue: thread = channel k, half of the interior rows
        const int e = warp - kRbEpiWarp0;
        const int lane_base = 32 * (warp & 3);
        const int k = lane_base + lane;
        const int h = e >> 2;                                     // row group: interior rows [NP RP h, NP RP (h + 1))
        float wk[KW], acc[KW];
#pragma unroll
        for (int j = 0; j < KW; ++j) { wk[j] = __ldg(p.wdw + k * KW + j); acc[j] = 0.f; }
        float dbacc = 0.f;
        int it = 0, xs = 0;
        uint32_t xph = 0;
        for (int g = g0; g < g1; ++g, ++it) {
            const int a = it & 1, s = xs;
            const int b = g / p.n_lt, l0 = (g - b * p.n_lt) * kRwInt;
            const float* rx = rawX + s * TILE + k;
            if (e == 0 && lane == 0) trace_ev(p.trace, 2, 1);
            mbar_wait(&bar_x[s], xph);                            // the raw X tile (async-proxy writes) is visible to this thread too
            mbar_wait(&bar_tfull[a], (uint32_t)(it >> 1) & 1u);
            tc_fence_after();
            if (e == 0 && lane == 0) trace_ev(p.trace, 2, 2);
#pragma unroll
            for (int sp = 0; sp < NP; ++sp) {                    // sub-passes of RP interior rows: dO window of RP + 2 P rows
                const int c = (NP * RP) * h + RP * sp;           // first tile row (= accumulator column) of the window: 0, 12, 24, 36
                const int OFF = 4 * sp;                          // the window starts at d[OFF]: ...
                const int cs = c - OFF;                           // ... it is fetched from the 8-aligned column at or below it
                float d[32];
                {
                    uint32_t r[32];
#pragma unroll
                    for (int q = 0; q < 4; ++q)                  // four loads in flight, ONE wait
                        tmem_ld8_issue(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(a * 64 + cs + 8 * q), r + 8 * q);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) d[i] = __uint_as_float(r[i]);
                }
                if (sp == NP - 1) {                               // accumulator a fully read by this thread
                    tc_fence_before();
                    mbar_arrive(&bar_tempty[a]);
                    if (e == 0 && lane == 0) trace_ev(p.trace, 2, 4);
                }
                float* dxp = p.dX + ((long)b * p.L + l0 + c) * 128 + k;    // interior row t of the window <-> position l0 + c + t
                const int n_rows = p.L - l0 - c;                             // rows of this window inside the task
#pragma unroll
                for (int i = 0; i < RP + 2 * P; ++i) {            // X row of the window: tile row c + i
                    const float x = rx[(c + i) * 128];
                    const float rxv = fmaxf(x, 0.f);
#pragma unroll
                    for (int j = 0; j < KW; ++j) {                // filter gradient: interior row t = i - j meets X row i through tap j
                        const int t = i - j;
                        if (t >= 0 && t < RP) acc[j] = fmaf(d[OFF + P + t], rxv, acc[j]);
                    }
                    const int t = i - P;                          // this X row is interior row t: its data gradient
                    if (t >= 0 && t < RP) {
                        float conv = wk[0] * d[OFF + 2 * P + t];          // one chain: the kernel is bound by instruction issue, not by FMA latency
#pragma unroll
                        for (int j = 1; j < KW; ++j) conv = fmaf(wk[j], d[OFF + 2 * P + t - j], conv);
                        dbacc += d[OFF + P + t];
                        if (t < n_rows) dxp[(long)t * 128] = d[OFF + P + t] + (x > 0.f ? conv : 0.f);
                    }
                }
            }
            mbar_arrive(&bar_xfree[s]);                           // the epilogue's reads of this raw X buffer are done
            if (e == 0 && lane == 0) trace_ev(p.trace, 2, 3);
            if (++xs == NX) { xs = 0; xph ^= 1u; }
        }
#pragma unroll
        for (int j = 0; j < KW; ++j) atomicAdd(p.dWdw + k * KW + j, acc[j]);
        if (p.dbdw) atomicAdd(p.dbdw + k, dbacc);
        // ---- flush of the CTA's pointwise weight gradient: thread = row n of dWpw, 64 columns per warp
        mbar_wait(&bar_dwfull, 0);
        tc_fence_after();
        const int col_base = h * 64;                              // 128 columns over the two row groups
#pragma unroll 1
        for (int ch = 0; ch < 4; ++ch) {
            const int c0 = col_base + ch * 16;
            float v[16];
            tmem_ld16(tmem + ((uint32_t)lane_base << 16) + (uint32_t)(128 + c0), v);
            float* dst = p.dWpw + (long)k * 128 + c0;
#pragma unroll
            for (int i = 0; i < 16; i += 4) atomicAdd(reinterpret_cast<float4*>(dst + i), make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

template <int KW, int NE>
static int launch_rb_bwd(RbBwdParams& p, cudaStream_t st) {
    const size_t smem = (size_t)4 * kRwHalf + (size_t)(kRwNY + kRwNX) * kRwRows * 512;
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(resblock1d_bwd_kernel<KW, NE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            cudaGetLastError();
            return NPF_ENOTSUP;
        }
        attr = true;
    }
    const int grid = p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs;
    launch_pdl(resblock1d_bwd_kernel<KW, NE>, dim3(grid), dim3(kRwThreads), smem, st, p);
    count_launch();
    return check_launch("resblock1d_bwd_kernel");
}

static inline bool rb_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace npf

using namespace npf;

extern "C" int npf_resblock1d_fwd(const float* X, const float* wdw, const float* bdw, const float* wpw, const float* bpw, float* O, float* Y,
                                  int B, int L, int C, int k, int precision, npf_stream_t stream) {
    NPF_REQUIRE(X && wdw && wpw && Y, "npf_resblock1d_fwd: null pointer");
    NPF_REQUIRE(B >= 0 && L >= 1 && k >= 1 && (k & 1), "npf_resblock1d_fwd: bad shape (odd kernel size)");
    if (B == 0) return NPF_OK;
    if (C != 128 || precision != NPF_PREC_BF16X3 || k != 11 || !rb_aligned16(X) || !rb_aligned16(Y) || !rb_aligned16(wpw) || (O && !rb_aligned16(O))) {
        set_error("npf_resblock1d_fwd: covered: 128 channels, kernel size 11, precision bf16x3, 16-byte aligned tensors; run npf_dwconv_fwd + npf_linear_fwd otherwise");
        return NPF_ENOTSUP;
    }
    RbFwdParams p{};
    p.X = X; p.wdw = wdw; p.bdw = bdw; p.wpw = wpw; p.bpw = bpw; p.O = O; p.Y = Y; p.B = B; p.L = L;
    // rows per tile: the choice that leaves the fewest rows on the most loaded CTA
    auto critical_rows = [&](int tr) { const long nt = (long)B * ((L + tr - 1) / tr); return ((nt + kNumSMs - 1) / kNumSMs) * tr; };
    const int tr = critical_rows(96) < critical_rows(128) ? 96 : 128;
    p.n_lt = (L + tr - 1) / tr;
    p.n_tiles = B * p.n_lt;
    p.trace = trace_buffer();
    return tr == 96 ? launch_rb_fwd<11, 96>(p, as_stream(stream)) : launch_rb_fwd<11, 128>(p, as_stream(stream));
}

extern "C" int npf_resblock1d_bwd(const float* dY, const float* X, const float* wdw, const float* bdw, const float* wpw, float* dX, float* dWdw,
                                  float* dbdw, float* dWpw, float* dbpw, int B, int L, int C, int k, int precision, npf_stream_t stream) {
    NPF_REQUIRE(dY && X && wdw && wpw && dX && dWdw && dWpw, "npf_resblock1d_bwd: null pointer");
    NPF_REQUIRE(B >= 0 && L >= 1 && k >= 1 && (k & 1), "npf_resblock1d_bwd: bad shape (odd kernel size)");
    if (B == 0) return NPF_OK;
    if (C != 128 || precision != NPF_PREC_BF16X3 || k != 11 || !rb_aligned16(dY) || !rb_aligned16(X) || !rb_aligned16(dX) || !rb_aligned16(wpw) ||
        !rb_aligned16(dWpw)) {
        set_error("npf_resblock1d_bwd: covered: 128 channels, kernel size 11, precision bf16x3, 16-byte aligned tensors; run npf_linear_bwd + npf_dwconv_bwd otherwise");
        return NPF_ENOTSUP;
    }
    RbBwdParams p{};
    p.dY = dY; p.X = X; p.wdw = wdw; p.bdw = bdw; p.wpw = wpw; p.dX = dX; p.dWdw = dWdw; p.dbdw = dbdw; p.dWpw = dWpw; p.dbpw = dbpw;
    p.B = B; p.L = L;
    p.n_lt = (L + kRwInt - 1) / kRwInt;
    p.n_tiles = B * p.n_lt;
    p.trace = trace_buffer();
    return launch_rb_bwd<11, kRbEpi>(p, as_stream(stream));
}
