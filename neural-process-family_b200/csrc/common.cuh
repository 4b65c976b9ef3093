// Shared helpers for libnpf_b200 (sm_100a).  Error plumbing, launch accounting, small device utilities.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/npf_b200.h"

namespace npf {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
unsigned long long* trace_buffer();     // diagnostics (npf_debug_set_trace); nullptr unless set

// timeline record of CTA 0: slot `role` (0..15) holds up to 255 (event, clock) records after a counter
__device__ __forceinline__ void trace_ev(unsigned long long* tr, int role, int event) {
    if (tr == nullptr || blockIdx.x != 0) return;
    unsigned long long* slot = tr + role * 256;
    const unsigned long long n = slot[0];
    if (n < 255) {
        const unsigned long long t = (unsigned long long)clock64();      // SM cycle counter: every role of the CTA shares it
        slot[1 + n] = ((unsigned long long)event << 56) | (t & 0x00FFFFFFFFFFFFFFull);
        slot[0] = n + 1;
    }
}

// returns NPF_OK or NPF_ECUDA after a kernel launch (no sync)
int check_launch(const char* what);

static inline cudaStream_t as_stream(npf_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

#define NPF_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            npf::set_error(__VA_ARGS__);  \
            return NPF_EINVAL;            \
        }                                 \
    } while (0)

constexpr int kNumSMs = 148;  // B200

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// softplus with the same branch structure as ATen (threshold 20): log1p(exp(x)) for x <= 20, x otherwise
__device__ __forceinline__ float softplus_f(float x) { return x > 20.f ? x : log1pf(expf(x)); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }

static inline long cdiv(long a, long b) { return (a + b - 1) / b; }

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------------------
// A kernel launched with launch_pdl may begin while its stream predecessor is still draining: its CTAs are scheduled as
// soon as every predecessor CTA has passed pdl_trigger() (or exited) and SM resources free up, so launch latency, the
// prologue that touches only parameters (TMEM allocation, barrier init, weight staging) and the predecessor's tail
// overlap.  CONTRACT: such a kernel executes pdl_wait() before its first access to anything a preceding kernel may have
// written (activations, gradients, statistics) and before its first global write; pdl_wait returns once the predecessor
// grid has completed and its memory is visible.
// The early start is requested only while the stream is being captured into a CUDA graph (GraphedStep): there the kernel
// order is the library's own, and no kernel that writes PARAMETERS (an optimizer step) can sit directly in front of a
// kernel whose pre-wait prologue reads them.  Eager launches keep plain stream order (the wait is then a no-op).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    const bool early = cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusActive;
    attr[0].val.programmaticStreamSerializationAllowed = early ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

}  // namespace npf
