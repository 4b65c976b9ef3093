// Tensor-core (tcgen05 / TMEM) path of the multi-head cross-attention, head dim 16 or 32 (the "multihead" /
// "transformer" attenders: 8 heads x 16).   NPF_PREC_BF16: operands rounded to bf16; NPF_PREC_BF16X3: hi+lo split,
// 3 MMAs per product (fp32-level logits and P.V).
//
// Forward, one CTA per (task, head, 128-query block), 128 threads = 128 TMEM lanes = 128 query rows:
//   per chunk of KC = 128 or 64 keys (64: four CTAs per SM; chosen when the grid is large enough):
//                       S = Q K^T          tcgen05.mma  M=128 N=KC K=D         (accumulator: TMEM cols [0,KC))
//                       thread r reads row r of S from TMEM (tcgen05.ld), online softmax (running max / sum, exp2),
//                       writes P (bf16 hi/lo) straight into the UMMA K-major operand layout in shared memory
//                       O_c = P V          tcgen05.mma  M=128 N=Dv  K=KC       (accumulator: TMEM cols [KC,KC+Dv))
//                       thread r: O_r = O_r * alpha + O_c[r, :]   (registers)
//   The [Tq, Tk] logits / probabilities never leave the SM.
//
// Operand layouts (no swizzle, 8x8 core matrices of 128 B; see tc_common.cuh / gemm_tc.cu):
//   Q, K   K-major over d :  (d/8)*LBO + (row/8)*128 + (row%8)*16 + (d%8)*2,   LBO = rows*16
//   P      K-major over key: (key/8)*2048 + (q/8)*128 + (q%8)*16 + (key%8)*2
//   V      MN-major (N = channel c, K = key): (key/8)*LBO + (c/8)*128 + (key%8)*16 + (c%8)*2,  LBO = (Dv/8)*128
#include "tc_common.cuh"

namespace npf {

struct AttnTcParams {
    const float* Q; const float* K; const float* V; const float* O; const float* LSE; const float* dO;
    float* Oo; float* LSEo; float* dQ; float* dK; float* dV;
    int Tq, Tk, H, D, Dv;
    float scale;
};

constexpr int kQB = 128;   // query rows per CTA (= TMEM lanes)
constexpr int kKC = 128;   // keys per chunk

__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
    return make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}
__device__ __forceinline__ void split8(const float (&v)[8], float (&lo)[8]) {
#pragma unroll
    for (int i = 0; i < 8; i += 2) {     // residual against the packed bf16 pair (bf16 -> fp32 is a 16-bit shift)
        const uint32_t h = pack_bf16(v[i], v[i + 1]);
        lo[i] = v[i] - __uint_as_float(h << 16);
        lo[i + 1] = v[i + 1] - __uint_as_float(h & 0xFFFF0000u);
    }
}

// Stage `rows_valid` rows (thread = row) of a [rows, width] fp32 slice (row stride ld) as a K-major operand with `R`
// rows in the tile: chunk (w/8) at (w/8)*R*16 + (row/8)*128 + (row%8)*16.
template <int NSPLIT>
__device__ __forceinline__ void stage_rows_kmajor(uint8_t* hi, uint8_t* lo, const float* __restrict__ src, long ld, int row, bool valid, int width,
                                                  int R, uint8_t* lo2 = nullptr) {
    const uint32_t base = (uint32_t)(row >> 3) * 128u + (uint32_t)(row & 7) * 16u;
    for (int ch = 0; ch < (width >> 3); ++ch) {
        float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (valid) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(src + (long)row * ld + ch * 8));
            const float4 b = __ldg(reinterpret_cast<const float4*>(src + (long)row * ld + ch * 8 + 4));
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        }
        const uint32_t off = (uint32_t)ch * (uint32_t)R * 16u + base;
        *reinterpret_cast<uint4*>(hi + off) = pack8(v);
        if (NSPLIT == 3) {
            float l[8];
            split8(v, l);
            *reinterpret_cast<uint4*>(lo + off) = pack8(l);
            if (lo2) {   // third bf16 term: x = hi + lo + lo2 to fp32 precision (operands of the softmax logits)
                float l2[8];
                split8(l, l2);
                *reinterpret_cast<uint4*>(lo2 + off) = pack8(l2);
            }
        }
    }
}

// Logits need fp32-level accuracy (an absolute logit error is a RELATIVE error of the softmax weight, and trained
// attention has |logit| ~ 1e2): with NSPLIT == 3 the product Q K^T uses three bf16 terms per operand and the six
// cross products down to 2^-24: hh, hm, mh, mm, hl, lh.
template <int NSPLIT>
__device__ __forceinline__ void mma_logits(uint32_t d, uint32_t a_h, uint32_t a_m, uint32_t a_l, uint32_t a_lbo, uint32_t b_h, uint32_t b_m, uint32_t b_l,
                                           uint32_t b_lbo, uint32_t idesc, uint32_t acc) {
    umma_bf16(d, make_desc(a_h, a_lbo, 128), make_desc(b_h, b_lbo, 128), idesc, acc);
    if (NSPLIT == 3) {
        umma_bf16(d, make_desc(a_h, a_lbo, 128), make_desc(b_m, b_lbo, 128), idesc, 1);
        umma_bf16(d, make_desc(a_m, a_lbo, 128), make_desc(b_h, b_lbo, 128), idesc, 1);
        umma_bf16(d, make_desc(a_m, a_lbo, 128), make_desc(b_m, b_lbo, 128), idesc, 1);
        umma_bf16(d, make_desc(a_h, a_lbo, 128), make_desc(b_l, b_lbo, 128), idesc, 1);
        umma_bf16(d, make_desc(a_l, a_lbo, 128), make_desc(b_h, b_lbo, 128), idesc, 1);
    }
}

// V chunk as MN-major B operand (N = channel, K = key): thread = key row.
template <int NSPLIT>
__device__ __forceinline__ void stage_rows_mnmajor(uint8_t* hi, uint8_t* lo, const float* __restrict__ src, long ld, int row, bool valid, int width) {
    const uint32_t lbo = (uint32_t)(width >> 3) * 128u;
    const uint32_t base = (uint32_t)(row >> 3) * lbo + (uint32_t)(row & 7) * 16u;
    for (int ch = 0; ch < (width >> 3); ++ch) {
        float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (valid) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(src + (long)row * ld + ch * 8));
            const float4 b = __ldg(reinterpret_cast<const float4*>(src + (long)row * ld + ch * 8 + 4));
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        }
        const uint32_t off = base + (uint32_t)ch * 128u;
        *reinterpret_cast<uint4*>(hi + off) = pack8(v);
        if (NSPLIT == 3) {
            float l[8];
            split8(v, l);
            *reinterpret_cast<uint4*>(lo + off) = pack8(l);
        }
    }
}

// KC keys per chunk: 128, or 64 -- half the logits / probability tile, 55 KB of shared memory and 128 TMEM columns per CTA, so that FOUR
// CTAs share an SM instead of two (every phase of a CTA is serial: stage -> MMA -> softmax -> MMA; the overlap comes from the neighbours).
template <int NSPLIT, int DV, int KC>
__global__ void __launch_bounds__(128) xattn_fwd_tc_kernel(AttnTcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_s, bar_o;
    __shared__ uint32_t tmem_slot;
    const int D = p.D;
    const uint32_t q_bytes = kQB * D * 2u, k_bytes = KC * D * 2u, v_bytes = KC * DV * 2u, p_bytes = kQB * KC * 2u;
    uint8_t* q_hi = smem_raw;
    uint8_t* k_hi = q_hi + q_bytes;
    uint8_t* v_hi = k_hi + k_bytes;
    uint8_t* p_hi = v_hi + v_bytes;
    const uint32_t half = q_bytes + k_bytes + v_bytes + p_bytes;
    uint8_t* q_lo = q_hi + half; uint8_t* k_lo = k_hi + half; uint8_t* v_lo = v_hi + half; uint8_t* p_lo = p_hi + half;   // NSPLIT == 3 only
    uint8_t* q_l2 = smem_raw + 2 * half; uint8_t* k_l2 = q_l2 + q_bytes;                                                  // NSPLIT == 3 only

    const int tid = threadIdx.x, warp = tid >> 5;
    const int qb = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int q_row = qb * kQB + tid;
    const bool q_ok = q_row < p.Tq;
    const long ldq = (long)p.H * D, ldv = (long)p.H * DV;
    const float* Qb = p.Q + ((long)b * p.Tq) * ldq + h * D;
    const float* Kb = p.K + ((long)b * p.Tk) * ldq + h * D;
    const float* Vb = p.V + ((long)b * p.Tk) * ldv + h * DV;

    constexpr uint32_t kCols = KC == 128 ? 256 : 128;   // S: [0, KC), O chunk: [KC, KC + DV)
    if (warp == 0) tmem_alloc(&tmem_slot, kCols);
    if (tid == 0) { mbar_init(&bar_s, 1); mbar_init(&bar_o, 1); }
    stage_rows_kmajor<NSPLIT>(q_hi, q_lo, Qb + (long)qb * kQB * ldq, ldq, tid, q_ok, D, kQB, NSPLIT == 3 ? q_l2 : nullptr);   // tile row tid <- query row
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t t_s = tmem + ((uint32_t)(32 * warp) << 16);
    const uint32_t t_o = t_s + (uint32_t)KC;
    const uint32_t idesc_s = make_idesc(128, KC, 0, 0);
    const uint32_t idesc_o = make_idesc(128, DV, 0, 1);
    const uint32_t q_lbo = kQB * 16u, k_lbo = KC * 16u, p_lbo = kQB * 16u, v_lbo = (uint32_t)(DV >> 3) * 128u;

    const float sl2 = p.scale * 1.4426950408889634f;      // logits in log2 units: exp(x) = exp2(x * log2 e)
    float m_run = -INFINITY, l_run = 0.f;
    float o_run[DV];
#pragma unroll
    for (int c = 0; c < DV; ++c) o_run[c] = 0.f;

    uint32_t ph = 0;
    for (int k0 = 0; k0 < p.Tk; k0 += KC) {
        // stage this chunk of K and V (thread = key row); the previous chunk's MMAs have completed (bar_o waited below)
        if (KC == 128) {
            const bool k_ok = k0 + tid < p.Tk;
            stage_rows_kmajor<NSPLIT>(k_hi, k_lo, Kb + (long)k0 * ldq, ldq, tid, k_ok, D, KC, NSPLIT == 3 ? k_l2 : nullptr);
            stage_rows_mnmajor<NSPLIT>(v_hi, v_lo, Vb + (long)k0 * ldv, ldv, tid, k_ok, DV);
        } else {                                   // 64 keys: threads 0..63 stage the K rows, threads 64..127 the V rows
            const int row = tid & 63;
            const bool k_ok = k0 + row < p.Tk;
            if (tid < 64) stage_rows_kmajor<NSPLIT>(k_hi, k_lo, Kb + (long)k0 * ldq, ldq, row, k_ok, D, KC, NSPLIT == 3 ? k_l2 : nullptr);
            else stage_rows_mnmajor<NSPLIT>(v_hi, v_lo, Vb + (long)k0 * ldv, ldv, row, k_ok, DV);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            for (int ks = 0; ks < D / 16; ++ks) {
                const uint32_t oq = (uint32_t)ks * 2u * q_lbo, ok = (uint32_t)ks * 2u * k_lbo;
                mma_logits<NSPLIT>(tmem, smem_u32(q_hi) + oq, smem_u32(q_lo) + oq, smem_u32(q_l2) + oq, q_lbo, smem_u32(k_hi) + ok, smem_u32(k_lo) + ok,
                                   smem_u32(k_l2) + ok, k_lbo, idesc_s, ks > 0);
            }
            umma_commit(&bar_s);
        }
        mbar_wait(&bar_s, ph);
        tc_fence_after();

        // ---- online softmax over this chunk's 128 logits of row `tid` ----
        const int n_valid = min(KC, p.Tk - k0);
        float mx = -INFINITY;
#pragma unroll 1
        for (int c0 = 0; c0 < KC; c0 += 32) {
            float v[32];
            tmem_ld32(t_s + (uint32_t)c0, v);
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (c0 + j < n_valid) mx = fmaxf(mx, v[j] * sl2);
        }
        const float m_new = fmaxf(m_run, mx);               // finite: every chunk holds >= 1 valid key
        const float alpha = exp2f(m_run - m_new);           // first chunk: exp2(-inf) = 0
        float lsum = 0.f;
#pragma unroll 1
        for (int c0 = 0; c0 < KC; c0 += 32) {
            float v[32];
            tmem_ld32(t_s + (uint32_t)c0, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const float e = (c0 + j < n_valid) ? exp2f(fmaf(v[j], sl2, -m_new)) : 0.f;
                v[j] = e;
                lsum += e;
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float w8[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) w8[i] = v[g * 8 + i];
                const uint32_t off = (uint32_t)((c0 >> 3) + g) * p_lbo + (uint32_t)(tid >> 3) * 128u + (uint32_t)(tid & 7) * 16u;
                *reinterpret_cast<uint4*>(p_hi + off) = pack8(w8);
                if (NSPLIT == 3) {
                    float l8[8];
                    split8(w8, l8);
                    *reinterpret_cast<uint4*>(p_lo + off) = pack8(l8);
                }
            }
        }
        l_run = l_run * alpha + lsum;
        m_run = m_new;

        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            uint32_t acc = 0;
            for (int ks = 0; ks < KC / 16; ++ks) {
                const uint32_t po = (uint32_t)ks * 2u * p_lbo, vo = (uint32_t)ks * 2u * v_lbo;
                umma_bf16(tmem + (uint32_t)KC, make_desc(smem_u32(p_hi) + po, p_lbo, 128), make_desc(smem_u32(v_hi) + vo, v_lbo, 128), idesc_o, acc);
                acc = 1;
                if (NSPLIT == 3) {
                    umma_bf16(tmem + (uint32_t)KC, make_desc(smem_u32(p_hi) + po, p_lbo, 128), make_desc(smem_u32(v_lo) + vo, v_lbo, 128), idesc_o, 1);
                    umma_bf16(tmem + (uint32_t)KC, make_desc(smem_u32(p_lo) + po, p_lbo, 128), make_desc(smem_u32(v_hi) + vo, v_lbo, 128), idesc_o, 1);
                }
            }
            umma_commit(&bar_o);
        }
        mbar_wait(&bar_o, ph);
        ph ^= 1;
        tc_fence_after();
#pragma unroll
        for (int c0 = 0; c0 < DV; c0 += 16) {
            float oc[16];
            tmem_ld16(t_o + (uint32_t)c0, oc);
#pragma unroll
            for (int j = 0; j < 16; ++j) o_run[c0 + j] = fmaf(o_run[c0 + j], alpha, oc[j]);
        }
        tc_fence_before();
        __syncthreads();       // all TMEM reads of this chunk done before the next chunk's MMAs / staging
    }
    if (q_ok) {
        const float inv = 1.f / l_run;
        float* out = p.Oo + ((long)b * p.Tq + q_row) * ldv + h * DV;
#pragma unroll
        for (int c = 0; c < DV; c += 4)
            *reinterpret_cast<float4*>(out + c) = make_float4(o_run[c] * inv, o_run[c + 1] * inv, o_run[c + 2] * inv, o_run[c + 3] * inv);
        p.LSEo[((long)b * p.H + h) * p.Tq + q_row] = (m_run + log2f(l_run)) * 0.6931471805599453f;   // back to natural log
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, kCols);
}

template <int NSPLIT, int DV, int KC>
static int launch_fwd_kc(AttnTcParams& p, int B, cudaStream_t st) {
    const size_t half = (size_t)(kQB * p.D + KC * p.D + KC * DV + kQB * KC) * 2;
    const size_t smem = half * (NSPLIT == 3 ? 2 : 1) + (NSPLIT == 3 ? (size_t)(kQB + KC) * p.D * 2 : 0);
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(xattn_fwd_tc_kernel<NSPLIT, DV, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess) {
            cudaGetLastError();
            return NPF_ENOTSUP;
        }
        attr = true;
    }
    dim3 grid((unsigned)cdiv(p.Tq, kQB), (unsigned)p.H, (unsigned)B);
    xattn_fwd_tc_kernel<NSPLIT, DV, KC><<<grid, 128, smem, st>>>(p);
    count_launch();
    return check_launch("xattn_fwd_tc_kernel");
}
template <int NSPLIT, int DV>
static int launch_fwd(AttnTcParams& p, int B, cudaStream_t st) {
    // 64-key chunks when there are enough CTAs to fill four per SM and more than one chunk of keys anyway
    const long ctas = (long)cdiv(p.Tq, kQB) * p.H * B;
    const bool small = p.Tk > 64 && ctas >= 2L * kNumSMs;
    return small ? launch_fwd_kc<NSPLIT, DV, 64>(p, B, st) : launch_fwd_kc<NSPLIT, DV, 128>(p, B, st);
}

// ----------------------------------------------------------------------------------------------------------------
// Backward.  One CTA per (task, head, 128-key block); loops over 64-query blocks with the score tile TRANSPOSED (TMEM
// lane = key), so that two CTAs fit an SM: a CTA's phases (stage -> MMA -> exp -> MMA -> atomics) are strictly serial, and
// the other CTA's work fills its hand-offs.  Per 64-query block:
//   S^T = K Q^T, dP^T = V dO^T                 (M = 128 keys, N = 64 queries, K = D | Dv: every operand in its natural row-major staging)
//   thread (key r, query half) : P^T = exp2(S^T scale - lse[q]), dS^T = P^T (dP^T - Di[q]) scale      -> [128 keys x 64 q] bf16 hi / lo images
//   dV += P^T dO,  dK += dS^T Q                (A = the images as stored, K-major over q; B = dO / Q read through the transposed view)
//   dQ_blk = dS K                               (A = transposed view of the dS^T image: its M extent is the 64 queries; the MMA runs with
//                                                M = 128 and the upper 64 accumulator rows, fed by whatever follows the image, are never read)
// 94 KB of shared memory (head dim 16) and 224 TMEM columns per CTA.
// Every staged tile uses ONE physical layout: 16-byte rows of 8 consecutive columns, 8 rows = a 128-byte core matrix, row
// groups 128 B apart, column chunks rows x 16 B apart (CHK = 2048 B in the 128-row tiles, CHQ = 1024 B in the 64-row ones).
// Read with (LBO = chunk stride, SBO = 128) it is a K-major operand over its columns; read with (LBO = 128, SBO = chunk
// stride) and the MN-major flag it is the TRANSPOSED operand -- so Q, dO, K, P and dS are staged once and serve both roles.
// ----------------------------------------------------------------------------------------------------------------
template <int NSPLIT>
__device__ __forceinline__ void mma3(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t a_lbo, uint32_t a_sbo, uint32_t b_hi, uint32_t b_lo,
                                     uint32_t b_lbo, uint32_t b_sbo, uint32_t idesc, uint32_t acc) {
    umma_bf16(d, make_desc(a_hi, a_lbo, a_sbo), make_desc(b_hi, b_lbo, b_sbo), idesc, acc);
    if (NSPLIT == 3) {
        umma_bf16(d, make_desc(a_hi, a_lbo, a_sbo), make_desc(b_lo, b_lbo, b_sbo), idesc, 1);
        umma_bf16(d, make_desc(a_lo, a_lbo, a_sbo), make_desc(b_hi, b_lbo, b_sbo), idesc, 1);
    }
}

template <int NSPLIT>
__global__ void __launch_bounds__(256, 2) xattn_bwd_tc_q64_kernel(AttnTcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar1, bar2;
    __shared__ uint32_t tmem_slot;
    __shared__ float s_lse2[64], s_di[64];
    const int D = p.D, DV = p.Dv;
    constexpr uint32_t CHK = 2048u, CHQ = 1024u;                 // column-chunk strides of the 128-row and the 64-row tiles
    constexpr int QB = 64;
    const uint32_t kt_b = (uint32_t)(D >> 3) * CHK, vt_b = (uint32_t)(DV >> 3) * CHK, qt_b = (uint32_t)(D >> 3) * CHQ, dot_b = (uint32_t)(DV >> 3) * CHQ;
    constexpr uint32_t pt_b = (QB / 8) * CHK;                    // 16 KB
    uint8_t* kt = smem_raw;
    uint8_t* vt = kt + kt_b;
    uint8_t* qt = vt + vt_b;
    uint8_t* dot_ = qt + qt_b;
    uint8_t* dst = dot_ + dot_b;                                  // dS^T, then P^T: the M = 128 read of the transposed dS view runs on into P^T
    uint8_t* pt = dst + pt_b;
    const uint32_t half = kt_b + vt_b + qt_b + dot_b + 2u * pt_b;
    const uint32_t LO = half;                                     // byte offset of the "lo" copies (NSPLIT == 3)
    uint8_t* kt_l2 = smem_raw + 2 * half; uint8_t* qt_l2 = kt_l2 + kt_b;     // third bf16 term of K and Q (logits only)

    const int tid = threadIdx.x, warp = tid >> 5;
    const int r = tid & 127, qh = tid >> 7;
    const int kb = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const long ldq = (long)p.H * D, ldv = (long)p.H * DV;
    const float* Qb = p.Q + ((long)b * p.Tq) * ldq + h * D;
    const float* Kb = p.K + ((long)b * p.Tk) * ldq + h * D;
    const float* Vb = p.V + ((long)b * p.Tk) * ldv + h * DV;
    const float* Ob = p.O + ((long)b * p.Tq) * ldv + h * DV;
    const float* Gb = p.dO + ((long)b * p.Tq) * ldv + h * DV;

    if (warp == 0) tmem_alloc(&tmem_slot, 256);
    if (tid == 0) { mbar_init(&bar1, 1); mbar_init(&bar2, 1); }
    const int key0 = kb * 128;
    const bool key_ok = key0 + r < p.Tk;
    if (qh == 0) stage_rows_kmajor<NSPLIT>(kt, kt + LO, Kb + (long)key0 * ldq, ldq, r, key_ok, D, 128, NSPLIT == 3 ? kt_l2 : nullptr);
    else stage_rows_kmajor<NSPLIT>(vt, vt + LO, Vb + (long)key0 * ldv, ldv, r, key_ok, DV, 128);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
    const uint32_t T_S = 0, T_DP = 64, T_DQ = 128, T_DK = 160, T_DV = 192;
    const uint32_t idesc_sp = make_idesc(128, QB, 0, 0);
    const uint32_t idesc_dv = make_idesc(128, DV, 0, 1), idesc_dk = make_idesc(128, D, 0, 1), idesc_dq = make_idesc(128, D, 1, 1);
    const float sl2 = p.scale * 1.4426950408889634f;
    const uint32_t s_kt = smem_u32(kt), s_vt = smem_u32(vt), s_qt = smem_u32(qt), s_dot = smem_u32(dot_), s_pt = smem_u32(pt), s_dst = smem_u32(dst);

    uint32_t ph = 0, acc_kv = 0;
    for (int q0 = 0; q0 < p.Tq; q0 += QB) {
        // stage this query block: Q rows (threads 0..63), dO rows (64..127), per-row lse and Di = dO . O (128..191)
        if (tid < 64) {
            stage_rows_kmajor<NSPLIT>(qt, qt + LO, Qb + (long)q0 * ldq, ldq, tid, q0 + tid < p.Tq, D, QB, NSPLIT == 3 ? qt_l2 : nullptr);
        } else if (tid < 128) {
            stage_rows_kmajor<NSPLIT>(dot_, dot_ + LO, Gb + (long)q0 * ldv, ldv, tid - 64, q0 + tid - 64 < p.Tq, DV, QB);
        } else if (tid < 192) {
            const int q = q0 + tid - 128;
            float di = 0.f;
            if (q < p.Tq)
                for (int c = 0; c < DV; c += 4) {
                    const float4 g4 = __ldg(reinterpret_cast<const float4*>(Gb + (long)q * ldv + c)), o4 = __ldg(reinterpret_cast<const float4*>(Ob + (long)q * ldv + c));
                    di = fmaf(g4.x, o4.x, fmaf(g4.y, o4.y, fmaf(g4.z, o4.z, fmaf(g4.w, o4.w, di))));
                }
            s_di[tid - 128] = di;
            s_lse2[tid - 128] = q < p.Tq ? __ldg(p.LSE + ((long)b * p.H + h) * p.Tq + q) * 1.4426950408889634f : INFINITY;   // +inf -> P = 0
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            for (int ks = 0; ks < D / 16; ++ks)      // S^T = K Q^T : both K-major over d, fp32-level product
                mma_logits<NSPLIT>(tmem + T_S, s_kt + ks * 2 * CHK, s_kt + LO + ks * 2 * CHK, smem_u32(kt_l2) + ks * 2 * CHK, CHK, s_qt + ks * 2 * CHQ,
                                   s_qt + LO + ks * 2 * CHQ, smem_u32(qt_l2) + ks * 2 * CHQ, CHQ, idesc_sp, ks > 0);
            for (int ks = 0; ks < DV / 16; ++ks)     // dP^T = V dO^T
                mma3<NSPLIT>(tmem + T_DP, s_vt + ks * 2 * CHK, s_vt + LO + ks * 2 * CHK, CHK, 128, s_dot + ks * 2 * CHQ, s_dot + LO + ks * 2 * CHQ, CHQ, 128,
                             idesc_sp, ks > 0);
            umma_commit(&bar1);
        }
        mbar_wait(&bar1, ph);
        tc_fence_after();
        {   // P^T and dS^T of key row r, queries [32 qh, 32 qh + 32) of the block
            const int c0 = 32 * qh;
            float sv[32], dv[32];
            tmem_ld32(tmem + lane_addr + T_S + (uint32_t)c0, sv);
            tmem_ld32(tmem + lane_addr + T_DP + (uint32_t)c0, dv);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const float pj = key_ok ? exp2f(fmaf(sv[j], sl2, -s_lse2[c0 + j])) : 0.f;
                sv[j] = pj;
                dv[j] = pj * (dv[j] - s_di[c0 + j]) * p.scale;
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float a8[8], b8[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { a8[i] = sv[g * 8 + i]; b8[i] = dv[g * 8 + i]; }
                const uint32_t off = (uint32_t)((c0 >> 3) + g) * CHK + (uint32_t)(r >> 3) * 128u + (uint32_t)(r & 7) * 16u;
                *reinterpret_cast<uint4*>(pt + off) = pack8(a8);
                *reinterpret_cast<uint4*>(dst + off) = pack8(b8);
                if (NSPLIT == 3) {
                    float l8[8];
                    split8(a8, l8);
                    *reinterpret_cast<uint4*>(pt + LO + off) = pack8(l8);
                    split8(b8, l8);
                    *reinterpret_cast<uint4*>(dst + LO + off) = pack8(l8);
                }
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            for (int ks = 0; ks < QB / 16; ++ks) {   // reduction over the block's 64 queries, 16 per step
                // dV += P^T dO : A = the P^T image (K-major over q), B = dO through the transposed view (N = channel)
                mma3<NSPLIT>(tmem + T_DV, s_pt + ks * 2 * CHK, s_pt + LO + ks * 2 * CHK, CHK, 128, s_dot + ks * 256, s_dot + LO + ks * 256, 128, CHQ, idesc_dv,
                             acc_kv | (uint32_t)(ks > 0));
                // dK += dS^T Q
                mma3<NSPLIT>(tmem + T_DK, s_dst + ks * 2 * CHK, s_dst + LO + ks * 2 * CHK, CHK, 128, s_qt + ks * 256, s_qt + LO + ks * 256, 128, CHQ, idesc_dk,
                             acc_kv | (uint32_t)(ks > 0));
            }
            for (int ks = 0; ks < 8; ++ks)           // dQ_blk = dS K : reduction over the 128 keys; A = transposed view of dS^T (rows 64..127 of D: unused)
                mma3<NSPLIT>(tmem + T_DQ, s_dst + ks * 256, s_dst + LO + ks * 256, 128, CHK, s_kt + ks * 256, s_kt + LO + ks * 256, 128, CHK, idesc_dq, ks > 0);
            umma_commit(&bar2);
        }
        acc_kv = 1;
        mbar_wait(&bar2, ph);
        ph ^= 1;
        tc_fence_after();
        if (tid < QB) {                              // lanes 0..63 of the dQ accumulator = the block's queries
            const int q = q0 + tid;
            for (int c0 = 0; c0 < D; c0 += 16) {
                float v[16];
                tmem_ld16(tmem + lane_addr + T_DQ + (uint32_t)c0, v);
                if (q < p.Tq) {
                    float* d = p.dQ + ((long)b * p.Tq + q) * ldq + h * D + c0;
#pragma unroll
                    for (int j = 0; j < 16; j += 4) atomicAdd(reinterpret_cast<float4*>(d + j), make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
                }
            }
        }
        tc_fence_before();
        __syncthreads();
    }
    if (acc_kv) {
        tc_fence_after();
        const int key = key0 + r;
        if (qh == 0) {
            for (int c0 = 0; c0 < D; c0 += 16) {
                float v[16];
                tmem_ld16(tmem + lane_addr + T_DK + (uint32_t)c0, v);
                if (key < p.Tk) {
                    float* d = p.dK + ((long)b * p.Tk + key) * ldq + h * D + c0;
#pragma unroll
                    for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(d + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                }
            }
        } else {
            for (int c0 = 0; c0 < DV; c0 += 16) {
                float v[16];
                tmem_ld16(tmem + lane_addr + T_DV + (uint32_t)c0, v);
                if (key < p.Tk) {
                    float* d = p.dV + ((long)b * p.Tk + key) * ldv + h * DV + c0;
#pragma unroll
                    for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(d + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

static bool attn_tc_ok(const AttnTcParams& p) {
    auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    return (p.D == 16 || p.D == 32) && (p.Dv == 16 || p.Dv == 32) && al(p.Q) && al(p.K) && al(p.V) && p.Tk >= 1;
}

int xattn_fwd_tc(const float* Q, const float* K, const float* V, float* O, float* LSE, int B, int Tq, int Tk, int H, int D, int Dv,
                 float scale, int precision, cudaStream_t st) {
    AttnTcParams p{};
    p.Q = Q; p.K = K; p.V = V; p.Oo = O; p.LSEo = LSE;
    p.Tq = Tq; p.Tk = Tk; p.H = H; p.D = D; p.Dv = Dv; p.scale = scale;
    if (!attn_tc_ok(p) || (reinterpret_cast<uintptr_t>(O) & 15)) return NPF_ENOTSUP;
    if (precision == NPF_PREC_BF16X3) return Dv == 16 ? launch_fwd<3, 16>(p, B, st) : launch_fwd<3, 32>(p, B, st);
    return Dv == 16 ? launch_fwd<1, 16>(p, B, st) : launch_fwd<1, 32>(p, B, st);
}

int xattn_bwd_tc(const float* Q, const float* K, const float* V, const float* O, const float* LSE, const float* dO, float* dQ, float* dK,
                 float* dV, int B, int Tq, int Tk, int H, int D, int Dv, float scale, int precision, cudaStream_t st) {
    AttnTcParams p{};
    p.Q = Q; p.K = K; p.V = V; p.O = O; p.LSE = LSE; p.dO = dO; p.dQ = dQ; p.dK = dK; p.dV = dV;
    p.Tq = Tq; p.Tk = Tk; p.H = H; p.D = D; p.Dv = Dv; p.scale = scale;
    auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if (!attn_tc_ok(p) || !al(O) || !al(dO) || !al(dQ) || !al(dK) || !al(dV) || Tq < 1) return NPF_ENOTSUP;
    const bool x3 = precision == NPF_PREC_BF16X3;
    const size_t half = (size_t)(D >> 3) * 2048 + (size_t)(Dv >> 3) * 2048 + (size_t)(D >> 3) * 1024 + (size_t)(Dv >> 3) * 1024 + 2 * 16384;
    const size_t smem = half * (x3 ? 2 : 1) + (x3 ? (size_t)(D >> 3) * (2048 + 1024) : 0);
    if (smem > 200 * 1024) return NPF_ENOTSUP;
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(xattn_bwd_tc_q64_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(xattn_bwd_tc_q64_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess) {
            cudaGetLastError();
            return NPF_ENOTSUP;
        }
        attr = true;
    }
    cudaMemsetAsync(dQ, 0, sizeof(float) * (size_t)B * Tq * H * D, st);   // dQ is accumulated over key blocks with atomics
    dim3 grid((unsigned)cdiv(Tk, 128), (unsigned)H, (unsigned)B);
    if (x3) xattn_bwd_tc_q64_kernel<3><<<grid, 256, smem, st>>>(p);
    else xattn_bwd_tc_q64_kernel<1><<<grid, 256, smem, st>>>(p);
    count_launch();
    return check_launch("xattn_bwd_tc_q64_kernel");
}

}  // namespace npf
