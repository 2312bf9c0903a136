// MusicGen LM decode step for B200 (sm_100a).
//
// One decode step = LMModel.forward on one token per row (audiocraft/models/lm.py:221-268) + CFG mix + sampling
// (lm.py:393-418) + the delay-pattern write-back (lm.py:553-562), replayed as ONE CUDA graph per step with every
// step-dependent quantity (position, tokens) resident on the device.
//
// The step is HBM-bound in bytes (all layer weights, fp16, 3.2 GB for medium, and the KV cache are read once per step at ~rows FLOP/B)
// and LATENCY-bound in time: 11 dependent kernels per layer.  Design consequences:
//   * weights stay in the reference's [out][in] fp16 layout; a CTA's 16 (or 32) x kslice slab is fetched with TMA bulk copies BEFORE
//     griddepcontrol.wait, i.e. while the previous kernel of the graph still runs (programmatic dependent launch); a 16x32 block of W
//     is the A operand of two m16n8k16 MMAs, the activations (a few KB, L2 resident) are the B operand, so the tile is 16 output
//     features x (8*NT) rows and nothing is wasted on padding rows up to 128.
//   * every GEMM spreads its weight matrix over >= 2 CTAs per SM; small-N GEMMs split K across CTAs and the partial sums are reduced
//     (in a fixed order: bit-reproducible) by the consumer kernel, which is the residual add + LayerNorm, so that reduction costs no
//     extra pass.
//   * K/V go from the QKV GEMM epilogue straight into the cache; cross-attention K/V are computed once per generate() instead of
//     every step (the reference recomputes them, transformer.py:355-357).
//   * attention for one query token: one CTA per (row, head) streaming K and V through a cp.async ring (lm_attn2_kernel).
// Alternatives that were built and measured slower (persistent fused step, cluster split-K with LayerNorm on load, chain kernels, ...)
// are listed with their numbers in DESIGN.md section 3.1.
#include "common.cuh"
#include "lm_step.cuh"
#include <math.h>
#include <new>
#include <vector>
#include <algorithm>
#include <utility>
#include <stdio.h>
#include <stdlib.h>

// ------------------------------------------------------------------------------------------------ helpers
__device__ __forceinline__ void mma16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// Programmatic dependent launch (PDL): a kernel launched with the programmatic-stream-serialization attribute may
// start while its predecessor is still running; everything before pdl_wait() must only touch memory no earlier
// kernel of the step writes (weights, LayerNorm parameters, the cross K/V, cache positions < pos: see
// enqueue_step_kernels).  Both are no-ops for a normally launched kernel.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Debug timeline: thread 0 of every CTA writes %globaltimer (ns) into its 8-slot record.  Compiled in only with
// -DACB_TIMELINE (ACB_BUILD_TIMELINE=1 python -m audiocraft_b200.build) and armed with ACB_LM_TIMING=1: at this time
// scale even the dormant stamps cost (532 kernels x ~0.3 us measured), because every instruction line of a 3 us kernel is
// fetched cold.
#ifdef ACB_TIMELINE
__device__ __forceinline__ void tl_stamp(unsigned long long* t, int slot) {
    if (t && threadIdx.x == 0) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        t[(((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 8 + slot] = now;
    }
}
#else
__device__ __forceinline__ void tl_stamp(unsigned long long*, int) {}
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (UBLKCP in SASS). 16 B aligned, size % 16 == 0.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ float half_round(float v) { return __half2float(__float2half_rn(v)); }
__device__ __forceinline__ float gelu_erf(float v) { return 0.5f * v * (1.f + erff(v * 0.70710678118654752440f)); }

// Block reductions: every thread returns the full result; red needs >= 32 floats and may be reused right after
// the call returns only behind another barrier (callers alternate two scratch arrays).
__device__ __forceinline__ float block_sum(float v, float* red) {
    v = warp_sum(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = lane < nw ? red[lane] : 0.f;
    return warp_sum(t);
}
__device__ __forceinline__ float block_max(float v, float* red) {
    v = warp_max(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = lane < nw ? red[lane] : -INFINITY;
    return warp_max(t);
}

// ------------------------------------------------------------------------------------------------ embed + sin pos
// x[r] = sum_k emb_k[seq[b,k,pos]] + pos_scale * [cos(pos/f_i), sin(pos/f_i)]   (lm.py:244, transformer.py:70-89,701-705)
// PF (prompt prefill): the grid's rows are (token, row) pairs r = tok * rows_real + row at positions P[0] + tok.
template <bool PF>
__global__ void __launch_bounds__(256) lm_embed_kernel(const __half* __restrict__ emb, const float* __restrict__ inv_freq,
                                                       const int64_t* __restrict__ seq, const int* __restrict__ P,
                                                       float* __restrict__ x, int d, int n_q, int card, int max_seq,
                                                       int batch, float pos_scale, int rows_real) {
    pdl_trigger();
    pdl_wait();
    const int r = blockIdx.x, b = (PF ? r % rows_real : r) % batch, pos = P[0] + (PF ? r / rows_real : 0);
    __shared__ int tok[16];
    if (threadIdx.x < n_q) {
        long long t = seq[((size_t)b * n_q + threadIdx.x) * max_seq + pos];
        tok[threadIdx.x] = (int)(t < 0 ? card : (t > card ? card : t));
    }
    __syncthreads();
    const int half_d = d >> 1;
    for (int i = threadIdx.x; i < d; i += 256) {   // d % 32 == 0: a warp is entirely inside or outside the row
        float v = 0.f;
        for (int k = 0; k < n_q; ++k) v += __half2float(emb[((size_t)k * (card + 1) + tok[k]) * d + i]);
        const int j = i < half_d ? i : i - half_d;
        const float phase = (float)pos / inv_freq[j];
        v += pos_scale * (i < half_d ? cosf(phase) : sinf(phase));
        x[(size_t)r * d + i] = v;
    }
}

// ------------------------------------------------------------------------------------------------ residual + LN
// x[r] += sum_s part[s][r] (fixed order), then h16[r] = LayerNorm(x[r]) * gamma + beta  (eps 1e-5, fp32 statistics).
// One CTA per row, ONE float4 per thread (d <= 2048): no per-thread loops, so the kernel is ~300 instructions -- at this
// time scale cold instruction fetch is a first-order cost (the 4-float4-per-thread version was 1 048 instructions and
// spent 1-2 us before its first load was consumed).  gamma / beta do not depend on the previous kernel and are
// requested before griddepcontrol.wait.
constexpr int LN_THREADS = 512;
__global__ void __launch_bounds__(LN_THREADS) lm_ln_kernel(float* __restrict__ x, const float* __restrict__ part, int nsplit,
                                                           size_t split_stride, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, __half* __restrict__ out, int d,
                                                           unsigned long long* timing) {
    __shared__ float red[2][32];
    const int r = blockIdx.x, i = threadIdx.x;
    const bool live = i < (d >> 2);
    tl_stamp(timing, 0);
    float4 gm = make_float4(0.f, 0.f, 0.f, 0.f), bt = gm;
    if (live) { gm = reinterpret_cast<const float4*>(gamma)[i]; bt = reinterpret_cast<const float4*>(beta)[i]; }
    pdl_trigger();
    pdl_wait();
    tl_stamp(timing, 1);
    float4* xr = reinterpret_cast<float4*>(x + (size_t)r * d);
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live) {
        a = xr[i];
        float4 pt[ACB_LM_MAX_SPLIT];
#pragma unroll
        for (int sp = 0; sp < ACB_LM_MAX_SPLIT; ++sp)   // independent loads, all in flight together
            pt[sp] = sp < nsplit ? reinterpret_cast<const float4*>(part + sp * split_stride + (size_t)r * d)[i]
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int sp = 0; sp < ACB_LM_MAX_SPLIT; ++sp) {  // fixed summation order
            a.x += pt[sp].x; a.y += pt[sp].y; a.z += pt[sp].z; a.w += pt[sp].w;
        }
        if (nsplit) xr[i] = a;
    }
    tl_stamp(timing, 4);
    const float mean = block_sum((a.x + a.y) + (a.z + a.w), red[0]) / d;
    tl_stamp(timing, 5);
    float q = 0.f;
    if (live) {
        const float cx = a.x - mean, cy = a.y - mean, cz = a.z - mean, cw = a.w - mean;
        q = fmaf(cx, cx, q); q = fmaf(cy, cy, q); q = fmaf(cz, cz, q); q = fmaf(cw, cw, q);
    }
    const float rstd = 1.f / sqrtf(block_sum(q, red[1]) / d + 1e-5f);
    tl_stamp(timing, 6);
    if (live) {
        __half2 lo = __floats2half2_rn((a.x - mean) * rstd * gm.x + bt.x, (a.y - mean) * rstd * gm.y + bt.y);
        __half2 hi = __floats2half2_rn((a.z - mean) * rstd * gm.z + bt.z, (a.w - mean) * rstd * gm.w + bt.w);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&lo);
        pk.y = *reinterpret_cast<uint32_t*>(&hi);
        reinterpret_cast<uint2*>(out + (size_t)r * d)[i] = pk;
    }
    tl_stamp(timing, 3);
}

// ------------------------------------------------------------------------------------------------ skinny GEMM
enum { EPI_PARTIAL = 0, EPI_QKV = 1, EPI_GELU = 2, EPI_F32 = 3, EPI_CROSSKV = 4, EPI_QKV_PF = 5 };   // _PF: prompt prefill, rows are (token, row) pairs

struct GemmParams {
    const __half* W;  // [N][K] fp16, reference layout
    const __half* X;  // [8*NT][K] fp16, rows >= `rows` are zero
    int N, K, rows, kslice;                            // kslice: K elements per CTA (grid.y slices)
    float* out_f32; int ld_out; size_t split_stride;  // PARTIAL / F32
    __half* out_f16;                                   // GELU
    float* q32; __half* kc; __half* vc; int d, H, cache_len; const int* pos;  // QKV / CROSSKV
    int text_len, row0;                                                      // CROSSKV
    int rows_real;                                                           // QKV_PF: rows of the generation (GEMM row = tok * rows_real + row)
    unsigned long long* timing;                 // debug timeline
};

// CTA = 4 warps, tile = 16 output features x kslice of K.  The CTA's 16 x kslice weight slab is fetched by ONE thread
// with 16 TMA bulk copies (one per W row, padded pitch => conflict-free fragment reads) BEFORE griddepcontrol.wait, i.e.
// while the producer of the activations is still running: under PDL the weight stream of kernel n+1 overlaps kernel n.
// FT2 = feature tiles of 16 per CTA (1, 2 or 3; see pick_tiling).  Wider tiles mean fewer CTAs and therefore less
// activation traffic out of L2: every CTA reads the whole (8*NT) x kslice activation block.
// STAGED: right after griddepcontrol.wait, warp 0 copies that activation block into shared memory with one TMA bulk copy
// per row (same padded pitch as the weight slab), so the k-loop waits for ONE round trip and then reads only shared
// memory.  Without it (register loads) every warp fetches its activation fragments in dependent batches of U k-blocks:
// at 12 k-blocks per warp that was 3 batches, ~0.8 us each (profiles/r1_lm_timeline_layer0_kv1_fine.log).  Both paths
// issue the same MMAs in the same order, so their results are bit-identical.
template <int NT, int EPI, int FT2 = 1, bool STAGED = false>
__global__ void __launch_bounds__(128) lm_gemm_kernel(GemmParams p) {
#ifndef ACB_GEMM_U2
#define ACB_GEMM_U2 4   // k-blocks per batch of activation loads at <= 16 rows (experiment builds: -DACB_GEMM_U2=6)
#endif
    constexpr int U = NT <= 2 ? ACB_GEMM_U2 : (NT <= 4 ? 2 : 1);
    constexpr int RP = 8 * NT + 1;
    constexpr int FB = 16 * FT2;                     // output features per CTA
    extern __shared__ __align__(128) unsigned char gsm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, c4 = lane & 3;
    const int f0 = blockIdx.x * FB;
    const int k0 = blockIdx.y * p.kslice;
    const int ks = min(p.kslice, p.K - k0);          // elements of K this CTA reduces over
    const int pitch = p.kslice * 2 + 64;             // bytes per staged W / X row (+64: conflict-free LDS.128)
    unsigned char* xs = gsm + FB * pitch;            // STAGED: [8*NT][pitch] activation block
    uint64_t* bar = reinterpret_cast<uint64_t*>(xs + (STAGED ? 8 * NT * pitch : 0));   // [0] weights, [1] activations
    float* red = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(bar) + 16);   // [4][FB][RP]

    tl_stamp(p.timing, 0);
    if (tid == 0) {
        mbar_init(bar, 1);
        if (STAGED) mbar_init(bar + 1, 1);
    }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(bar, (uint32_t)FB * (uint32_t)ks * 2u);
#pragma unroll 1
        for (int r = 0; r < FB; ++r)
            bulk_g2s(gsm + r * pitch, p.W + (size_t)(f0 + r) * p.K + k0, (uint32_t)ks * 2u, bar);
    }
    pdl_trigger();
    pdl_wait();   // activations written by the previous kernel are visible from here on
    tl_stamp(p.timing, 1);
    if (STAGED && warp == 0) {
        if (lane == 0) mbar_expect_tx(bar + 1, 8u * NT * (uint32_t)ks * 2u);
        __syncwarp();
#pragma unroll 1
        for (int r = lane; r < 8 * NT; r += 32)
            bulk_g2s(xs + r * pitch, p.X + (size_t)r * p.K + k0, (uint32_t)ks * 2u, bar + 1);
    }
    int cache_pos = 0;
    if (EPI == EPI_QKV || EPI == EPI_QKV_PF) cache_pos = p.pos[0];   // requested now, consumed in the epilogue: off the critical path

    float c[FT2][NT][4];
#pragma unroll
    for (int ft = 0; ft < FT2; ++ft)
#pragma unroll
        for (int j = 0; j < NT; ++j) c[ft][j][0] = c[ft][j][1] = c[ft][j][2] = c[ft][j][3] = 0.f;

    const int nkb = ks >> 5;
    const int kbw = (nkb + 3) >> 2;
    const int kb0 = min(nkb, warp * kbw), kb1 = min(nkb, kb0 + kbw);
    const __half* xr = p.X + (size_t)g * p.K + k0 + 8 * c4;
    const unsigned char* wr0 = gsm + g * pitch + 16 * c4;
    const unsigned char* wr1 = wr0 + 8 * pitch;

    bool w_ready = false;
    if (STAGED) {
        mbar_wait(bar, 0);
        tl_stamp(p.timing, 4);
        mbar_wait(bar + 1, 0);
        tl_stamp(p.timing, 7);
        w_ready = true;
        const unsigned char* xg = xs + g * pitch + 16 * c4;
#pragma unroll 2
        for (int kb = kb0; kb < kb1; ++kb) {
            uint4 xv[NT];
#pragma unroll
            for (int j = 0; j < NT; ++j) xv[j] = *reinterpret_cast<const uint4*>(xg + 8 * j * pitch + kb * 64);
#pragma unroll
            for (int ft = 0; ft < FT2; ++ft) {
                const uint4 wa = *reinterpret_cast<const uint4*>(wr0 + ft * 16 * pitch + kb * 64);
                const uint4 wb = *reinterpret_cast<const uint4*>(wr1 + ft * 16 * pitch + kb * 64);
#pragma unroll
                for (int j = 0; j < NT; ++j) {
                    mma16816(c[ft][j], wa.x, wb.x, wa.y, wb.y, xv[j].x, xv[j].y);
                    mma16816(c[ft][j], wa.z, wb.z, wa.w, wb.w, xv[j].z, xv[j].w);
                }
            }
        }
    }
    for (int kb = kb0; !STAGED && kb < kb1; kb += U) {
        uint4 xv[U][NT];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int j = 0; j < NT; ++j)
                xv[u][j] = (kb + u < kb1) ? *reinterpret_cast<const uint4*>(xr + (size_t)(8 * j) * p.K + (size_t)(kb + u) * 32)
                                          : make_uint4(0, 0, 0, 0);
        if (!w_ready) { mbar_wait(bar, 0); w_ready = true; tl_stamp(p.timing, 4); }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (kb + u < kb1) {
#pragma unroll
                for (int ft = 0; ft < FT2; ++ft) {
                    const uint4 wa = *reinterpret_cast<const uint4*>(wr0 + ft * 16 * pitch + (kb + u) * 64);
                    const uint4 wb = *reinterpret_cast<const uint4*>(wr1 + ft * 16 * pitch + (kb + u) * 64);
#pragma unroll
                    for (int j = 0; j < NT; ++j) {
                        mma16816(c[ft][j], wa.x, wb.x, wa.y, wb.y, xv[u][j].x, xv[u][j].y);
                        mma16816(c[ft][j], wa.z, wb.z, wa.w, wb.w, xv[u][j].z, xv[u][j].w);
                    }
                }
            }
        }
    }
    if (!w_ready) mbar_wait(bar, 0);   // never leave with a bulk copy in flight
    tl_stamp(p.timing, 2);
    // cross-warp (split-K inside the CTA) reduction in a fixed order
#pragma unroll
    for (int ft = 0; ft < FT2; ++ft)
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            float* r0 = red + (warp * FB + ft * 16 + g) * RP + 8 * j + 2 * c4;
            r0[0] = c[ft][j][0];
            r0[1] = c[ft][j][1];
            r0[8 * RP] = c[ft][j][2];
            r0[8 * RP + 1] = c[ft][j][3];
        }
    __syncthreads();
    tl_stamp(p.timing, 5);
    for (int idx = tid; idx < FB * 8 * NT; idx += 128) {
        const int row = idx / FB, feat = idx % FB;
        if (row >= p.rows) continue;
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < 4; ++w) v += red[(w * FB + feat) * RP + row];
        const int n = f0 + feat;
        if (EPI == EPI_PARTIAL) {
            p.out_f32[blockIdx.y * p.split_stride + (size_t)row * p.ld_out + n] = v;
        } else if (EPI == EPI_F32) {
            p.out_f32[(size_t)row * p.ld_out + n] = v;
        } else if (EPI == EPI_GELU) {
            p.out_f16[(size_t)row * p.ld_out + n] = __float2half_rn(gelu_erf(half_round(v)));
        } else if (EPI == EPI_QKV) {   // q | k | v blocks of d features each (no integer division: cold code costs here)
            const int which = n >= 2 * p.d ? 2 : (n >= p.d ? 1 : 0), nn = n - which * p.d;
            if (which == 0) {
                p.q32[(size_t)row * p.d + nn] = v;
            } else {
                __half* cache = which == 2 ? p.vc : p.kc;
                cache[(((size_t)row * p.H + (nn >> 6)) * p.cache_len + cache_pos) * 64 + (nn & 63)] = __float2half_rn(v);
            }
        } else if (EPI == EPI_QKV_PF) {   // prefill: row = tok * rows_real + r -> cache row r, position pos + tok
            const int which = n >= 2 * p.d ? 2 : (n >= p.d ? 1 : 0), nn = n - which * p.d;
            if (which == 0) {
                p.q32[(size_t)row * p.d + nn] = v;
            } else {
                const int tk = row / p.rows_real, rr = row - tk * p.rows_real;
                __half* cache = which == 2 ? p.vc : p.kc;
                cache[(((size_t)rr * p.H + (nn >> 6)) * p.cache_len + cache_pos + tk) * 64 + (nn & 63)] = __float2half_rn(v);
            }
        } else {  // EPI_CROSSKV: GEMM rows are (row, text position) pairs
            const int R = p.row0 + row, r = R / p.text_len, tc = R % p.text_len;
            const int which = n / p.d, nn = n % p.d, h = nn >> 6, dd = nn & 63;
            __half* cache = which ? p.vc : p.kc;
            cache[(((size_t)r * p.H + h) * p.cache_len + tc) * 64 + dd] = __float2half_rn(v);
        }
    }
    tl_stamp(p.timing, 3);
}

// ------------------------------------------------------------------------------------------------ attention (1 query)
struct AttnParams {
    const float* q; int q_nsplit; size_t q_split_stride;  // q[s][row][d] fp32 partial sums
    const __half* kc; const __half* vc; __half* out;
    int H, d, cache_len; const int* pos; int fixed_len; float scale;
    unsigned long long* timing;   // debug timeline
    int rows_real;                // prefill (PF kernels): rows of the generation
    float* part; int* counter;    // split-KV self attention (gridDim.z > 1): partial (m, l, acc[64]) records, arrival counters
    int split_min;                // contexts shorter than this stay on the single-CTA path
};

// Self attention for one query token: CTA = (row, head[, KV third]), 8 warps, ONE pass over K and V with an online softmax.
// A warp instruction reads 4 consecutive cache positions (4 x 128 B = 512 contiguous bytes); 8 lanes share a position
// (8 dims each).  4 positions-groups x 4 unrolled iterations of K and V are in flight per lane before any is consumed.
// Split KV (gridDim.z = 3, opt-in: ACB_LM_ATT_SPLIT=3): rows x heads = 384 CTAs are 2.6 per SM, so SMs holding 3 finish ~25 % after those holding 2
// (timeline at KV 751: median CTA 16.7 us, last 22.3 us).  Once the context reaches split_min positions it is cut into
// up to 3 chunks (multiples of the CTA's 128-position stride): 1 152 CTAs = 7.8 per SM.  Every chunk CTA writes its
// (m, l, acc) record, and the LAST one to arrive (atomic counter, threadfence) merges the records in chunk order, so the
// result does not depend on arrival order.  Short contexts take the single-CTA path; the idle CTAs exit at once.
constexpr int ATT_WARPS = 8, ATT_UNROLL = 4;   // UNROLL 8 measured slower (98 regs: 2 CTAs/SM instead of 5)

struct OnlineSM { float m, l, acc[8]; };
__device__ __forceinline__ void osm_merge(OnlineSM& a, float m2, float l2, const float (&acc2)[8]) {
    const float mn = fmaxf(a.m, m2);
    const float ca = a.m == -INFINITY ? 0.f : __expf(a.m - mn), cb = m2 == -INFINITY ? 0.f : __expf(m2 - mn);
    a.l = a.l * ca + l2 * cb;
#pragma unroll
    for (int e = 0; e < 8; ++e) a.acc[e] = a.acc[e] * ca + acc2[e] * cb;
    a.m = mn;
}

// SPLIT = false (default step): none of the chunk / record / merge code is compiled in.  PF (prompt prefill): blockIdx.y is a
// (token, row) pair tok * rows_real + r; the query at position pos + tok attends to the cache of row r up to and including
// its own position (the QKV GEMM of the same pass has already appended every token of the pass: causal within the chunk).
template <bool SPLIT, bool PF = false>
__global__ void __launch_bounds__(ATT_WARPS * 32) lm_attn_kernel(AttnParams p) {
    __shared__ float wm[ATT_WARPS], wl[ATT_WARPS], wacc[ATT_WARPS][64];
    const int h = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int qrow = blockIdx.y, row = PF ? qrow % p.rows_real : qrow, tok = PF ? qrow / p.rows_real : 0;
    const int sl = lane & 7, pg = lane >> 3;
    tl_stamp(p.timing, 0);
    pdl_trigger();
    pdl_wait();
    tl_stamp(p.timing, 1);
    const int n = p.fixed_len > 0 ? p.fixed_len : p.pos[0] + tok + 1;
    int lo = 0, hi = n, nact = 1;
    if (SPLIT && gridDim.z > 1) {
        // measured: the record write + atomic + merge costs more than the balance gains below ~750 positions
        // (KV 376: 2.71 vs 2.57 ms per step; KV 751: equal; KV 1500: 3.62 vs 3.80), hence split_min (default 768)
        const int S = gridDim.z, chunk = n < p.split_min ? n : max(128, ((n + S - 1) / S + 127) & ~127);
        nact = (n + chunk - 1) / chunk;
        if ((int)blockIdx.z >= nact) return;         // CTA-uniform: nothing in this chunk
        lo = blockIdx.z * chunk;
        hi = min(n, lo + chunk);
    }

    float q[8];
    {   // (split-K query partials exist only on the cross-attention path; a rolled/unrolled split loop here cost
        //  ~1 500 instructions of cold code per launch)
        const float4* qp = reinterpret_cast<const float4*>(p.q + (size_t)qrow * p.d + h * 64 + sl * 8);
        const float4 qa = qp[0], qb = qp[1];
        q[0] = half_round(qa.x) * p.scale; q[1] = half_round(qa.y) * p.scale; q[2] = half_round(qa.z) * p.scale;
        q[3] = half_round(qa.w) * p.scale; q[4] = half_round(qb.x) * p.scale; q[5] = half_round(qb.y) * p.scale;
        q[6] = half_round(qb.z) * p.scale; q[7] = half_round(qb.w) * p.scale;
    }
    tl_stamp(p.timing, 4);   // n and q consumed
    const size_t base = ((size_t)row * p.H + h) * p.cache_len * 64 + sl * 8;
    const __half* kb = p.kc + base;
    const __half* vb = p.vc + base;

    OnlineSM st;
    st.m = -INFINITY; st.l = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) st.acc[e] = 0.f;

    // warp-uniform loop bound (the shuffles need all 32 lanes)
    for (int pb = lo + warp * 4; pb < hi; pb += ATT_WARPS * 4 * ATT_UNROLL) {
        uint4 kv[ATT_UNROLL], vv[ATT_UNROLL];
#pragma unroll
        for (int u = 0; u < ATT_UNROLL; ++u) {
            const int pp = pb + u * ATT_WARPS * 4 + pg;
            if (pp < hi) {
                kv[u] = ld_stream_u4(kb + (size_t)pp * 64);
                vv[u] = ld_stream_u4(vb + (size_t)pp * 64);
            } else {
                kv[u] = vv[u] = make_uint4(0, 0, 0, 0);
            }
        }
#pragma unroll
        for (int u = 0; u < ATT_UNROLL; ++u) {
            const int pp = pb + u * ATT_WARPS * 4 + pg;
            const __half2* k2 = reinterpret_cast<const __half2*>(&kv[u]);
            float s = 0.f;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 f = __half22float2(k2[e]);
                s = fmaf(q[2 * e], f.x, s);
                s = fmaf(q[2 * e + 1], f.y, s);
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            if (pp < hi) {
                const float mn = fmaxf(st.m, s);
                const float corr = __expf(st.m - mn);   // exp(-inf) = 0 on the first position
                const float pw = __expf(s - mn);
                st.l = st.l * corr + pw;
                const __half2* v2 = reinterpret_cast<const __half2*>(&vv[u]);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float2 f = __half22float2(v2[e]);
                    st.acc[2 * e] = fmaf(pw, f.x, st.acc[2 * e] * corr);
                    st.acc[2 * e + 1] = fmaf(pw, f.y, st.acc[2 * e + 1] * corr);
                }
                st.m = mn;
            }
        }
    }
    tl_stamp(p.timing, 2);   // position loop
    // merge the 4 position groups of the warp, then the warps
#pragma unroll
    for (int o = 8; o <= 16; o <<= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, st.m, o), l2 = __shfl_xor_sync(0xffffffffu, st.l, o);
        float a2[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) a2[e] = __shfl_xor_sync(0xffffffffu, st.acc[e], o);
        osm_merge(st, m2, l2, a2);
    }
    tl_stamp(p.timing, 5);   // lane merges
    if (pg == 0) {
        if (sl == 0) { wm[warp] = st.m; wl[warp] = st.l; }
#pragma unroll
        for (int e = 0; e < 8; ++e) wacc[warp][sl * 8 + e] = st.acc[e];
    }
    __syncthreads();
    tl_stamp(p.timing, 6);
    float mx = -INFINITY, l = 0.f, o = 0.f;
    if (tid < 64) {
        mx = wm[0];
#pragma unroll
        for (int w = 1; w < ATT_WARPS; ++w) mx = fmaxf(mx, wm[w]);
#pragma unroll
        for (int w = 0; w < ATT_WARPS; ++w) {
            const float cw = wm[w] == -INFINITY ? 0.f : __expf(wm[w] - mx);
            l = fmaf(wl[w], cw, l);
            o = fmaf(wacc[w][tid], cw, o);
        }
    }
    if (!SPLIT || nact == 1) {                       // CTA-uniform
        if (tid < 64) p.out[(size_t)qrow * p.d + h * 64 + tid] = __float2half_rn(o / l);
    } else {
        __shared__ int is_last;
        float* rec = p.part + ((size_t)row * p.H + h) * gridDim.z * 66;
        if (tid < 64) {
            rec[blockIdx.z * 66 + 2 + tid] = o;
            if (tid == 0) { rec[blockIdx.z * 66] = mx; rec[blockIdx.z * 66 + 1] = l; }
        }
        __threadfence();
        __syncthreads();
        if (tid == 0) is_last = atomicAdd(p.counter + row * p.H + h, 1) == nact - 1;
        __syncthreads();
        if (is_last) {
            __threadfence();
            if (tid < 64) {
                float M = -INFINITY;
                for (int z = 0; z < nact; ++z) M = fmaxf(M, __ldcg(rec + z * 66));
                float L = 0.f, O = 0.f;
                for (int z = 0; z < nact; ++z) {     // chunk order: independent of which CTA arrived last
                    const float cz = __expf(__ldcg(rec + z * 66) - M);
                    L = fmaf(__ldcg(rec + z * 66 + 1), cz, L);
                    O = fmaf(__ldcg(rec + z * 66 + 2 + tid), cz, O);
                }
                p.out[(size_t)row * p.d + h * 64 + tid] = __float2half_rn(O / L);
            }
            if (tid == 0) p.counter[row * p.H + h] = 0;   // ready for the next layer / step
        }
    }
    tl_stamp(p.timing, 3);
}

// Self attention for one query token, deep-prefetch variant (the default decode path since round 2; ACB_LM_ATTN=v1 keeps the kernel
// above, which also serves prefill and split-KV).  Same work split and arithmetic as lm_attn_kernel<false>: CTA = (row, head), 8 warps,
// a warp instruction covers 4 consecutive cache positions, 8 lanes share a position.  What changes is how K and V get there: every lane
// copies its 16-byte slices with cp.async into a private slot of a per-warp shared-memory ring, ATT2_DEPTH iterations deep, and reads
// them back (its own 32 bytes) one iteration at a time.  With register loads a lane had 128 bytes in flight in bursts (4 iterations
// requested, then all consumed): ~83 KB per SM at 2.6 CTAs per SM, against the ~13 MB that 6.5 TB/s x ~2 us of loaded HBM latency asks
// of the chip (88 KB per SM): 4.05 TB/s at KV 751.  The ring keeps up to 8 x 32 bytes per lane outstanding continuously, in shared
// memory instead of registers.
constexpr int ATT2_DEPTH = 8;
__global__ void __launch_bounds__(ATT_WARPS * 32) lm_attn2_kernel(AttnParams p) {
    extern __shared__ __align__(16) unsigned char att2sm[];   // [warp][depth][K | V][32 lanes][16 B]
    __shared__ float wm[ATT_WARPS], wl[ATT_WARPS], wacc[ATT_WARPS][64];
    const int h = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = blockIdx.y;
    const int sl = lane & 7, pg = lane >> 3;
    tl_stamp(p.timing, 0);
    pdl_trigger();
    // Before griddepcontrol.wait: pos and every cache position < pos are final for the whole step (see enqueue_step_kernels: the
    // step's first kernel waits for everything enqueued before it), so the first ATT2_DEPTH - 1 ring stages are filled while the
    // QKV GEMM still runs.  Position pos itself is what that GEMM writes: it is skipped here and fetched after the wait.
    const int n = p.fixed_len > 0 ? p.fixed_len : p.pos[0] + 1;
    const size_t base = ((size_t)row * p.H + h) * p.cache_len * 64 + sl * 8;
    const __half* kb = p.kc + base;
    const __half* vb = p.vc + base;
    const uint32_t ring = smem_u32(att2sm) + (uint32_t)(warp * ATT2_DEPTH * 1024 + lane * 16);
    // iteration k of this warp covers positions (k * 8 + warp) * 4 + pg
    const int n_it = (n + 31 - warp * 4) / 32 > 0 ? (n - warp * 4 + 31) / 32 : 0;   // iterations with at least one live position group
    auto issue = [&](int k, int lim) {   // copies of positions < lim; every lane commits one group per call, empty or not
        if (k < n_it) {
            const int pp = (k * ATT_WARPS + warp) * 4 + pg;
            if (pp < lim) {
                const uint32_t d = ring + (uint32_t)((k % ATT2_DEPTH) * 1024);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(kb + (size_t)pp * 64) : "memory");
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + 512u), "l"(vb + (size_t)pp * 64) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
#pragma unroll
    for (int k = 0; k < ATT2_DEPTH - 1; ++k) issue(k, n - 1);
    pdl_wait();
    tl_stamp(p.timing, 1);
    // Position n - 1: if it fell into the stages above, its 8 lanes load it now (together with q) and put it into the slot of its
    // iteration, which no copy targets until this lane's loop has read it (same thread: no barrier needed).
    const int pl = n - 1, kl = pl >> 5;
    const bool own_last = kl < ATT2_DEPTH - 1 && ((pl >> 2) & (ATT_WARPS - 1)) == warp && (pl & 3) == pg;
    uint4 lk = make_uint4(0, 0, 0, 0), lv = lk;
    if (own_last) {
        lk = *reinterpret_cast<const uint4*>(kb + (size_t)pl * 64);
        lv = *reinterpret_cast<const uint4*>(vb + (size_t)pl * 64);
    }

    float q[8];
    {
        const float4* qp = reinterpret_cast<const float4*>(p.q + (size_t)row * p.d + h * 64 + sl * 8);
        const float4 qa = qp[0], qb = qp[1];
        q[0] = half_round(qa.x) * p.scale; q[1] = half_round(qa.y) * p.scale; q[2] = half_round(qa.z) * p.scale;
        q[3] = half_round(qa.w) * p.scale; q[4] = half_round(qb.x) * p.scale; q[5] = half_round(qb.y) * p.scale;
        q[6] = half_round(qb.z) * p.scale; q[7] = half_round(qb.w) * p.scale;
    }
    if (own_last) {
        const uint32_t d = ring + (uint32_t)(kl * 1024);
        asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(d), "r"(lk.x), "r"(lk.y), "r"(lk.z), "r"(lk.w) : "memory");
        asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(d + 512u), "r"(lv.x), "r"(lv.y), "r"(lv.z), "r"(lv.w) : "memory");
    }
    tl_stamp(p.timing, 4);
    OnlineSM st;
    st.m = -INFINITY; st.l = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) st.acc[e] = 0.f;

    for (int k = 0; k < n_it; ++k) {                 // warp-uniform trip count (the shuffles need all 32 lanes)
        issue(k + ATT2_DEPTH - 1, n);
        asm volatile("cp.async.wait_group %0;" ::"n"(ATT2_DEPTH - 1) : "memory");   // iteration k's copies of this lane have landed
        const int pp = (k * ATT_WARPS + warp) * 4 + pg;
        const uint32_t sa = ring + (uint32_t)((k % ATT2_DEPTH) * 1024);
        uint4 kv = make_uint4(0, 0, 0, 0), vv = make_uint4(0, 0, 0, 0);
        if (pp < n) {
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(kv.x), "=r"(kv.y), "=r"(kv.z), "=r"(kv.w) : "r"(sa));
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(vv.x), "=r"(vv.y), "=r"(vv.z), "=r"(vv.w) : "r"(sa + 512u));
        }
        const __half2* k2 = reinterpret_cast<const __half2*>(&kv);
        float s = 0.f;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = __half22float2(k2[e]);
            s = fmaf(q[2 * e], f.x, s);
            s = fmaf(q[2 * e + 1], f.y, s);
        }
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        if (pp < n) {
            const float mn = fmaxf(st.m, s);
            const float corr = __expf(st.m - mn);   // exp(-inf) = 0 on the first position
            const float pw = __expf(s - mn);
            st.l = st.l * corr + pw;
            const __half2* v2 = reinterpret_cast<const __half2*>(&vv);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 f = __half22float2(v2[e]);
                st.acc[2 * e] = fmaf(pw, f.x, st.acc[2 * e] * corr);
                st.acc[2 * e + 1] = fmaf(pw, f.y, st.acc[2 * e + 1] * corr);
            }
            st.m = mn;
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    tl_stamp(p.timing, 2);
    // merge the 4 position groups of the warp, then the warps (as lm_attn_kernel)
#pragma unroll
    for (int o = 8; o <= 16; o <<= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, st.m, o), l2 = __shfl_xor_sync(0xffffffffu, st.l, o);
        float a2[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) a2[e] = __shfl_xor_sync(0xffffffffu, st.acc[e], o);
        osm_merge(st, m2, l2, a2);
    }
    if (pg == 0) {
        if (sl == 0) { wm[warp] = st.m; wl[warp] = st.l; }
#pragma unroll
        for (int e = 0; e < 8; ++e) wacc[warp][sl * 8 + e] = st.acc[e];
    }
    __syncthreads();
    if (tid < 64) {
        float mx = wm[0];
#pragma unroll
        for (int w = 1; w < ATT_WARPS; ++w) mx = fmaxf(mx, wm[w]);
        float l = 0.f, o = 0.f;
#pragma unroll
        for (int w = 0; w < ATT_WARPS; ++w) {
            const float cw = wm[w] == -INFINITY ? 0.f : __expf(wm[w] - mx);
            l = fmaf(wl[w], cw, l);
            o = fmaf(wacc[w][tid], cw, o);
        }
        p.out[(size_t)row * p.d + h * 64 + tid] = __float2half_rn(o / l);
    }
    tl_stamp(p.timing, 3);
}

// Cross attention over the (short) text condition: one WARP per (row, head), lane = text position for the scores,
// lane = 2 output dims for the weighted sum.  K/V were computed once per generate() (acb_lm_begin) and no kernel of a step
// writes them (see enqueue_step_kernels: the step's first kernel waits for everything enqueued before it), so the first
// chunk of 32 text positions -- K row per lane, V pair of dims per lane -- is loaded into registers BEFORE
// griddepcontrol.wait; after it only the query partials are read.  Later chunks are loaded after the wait.
template <bool PF>
__global__ void __launch_bounds__(256) lm_cross_attn_kernel(AttnParams p, int rows) {
    __shared__ float qs[8][64];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int pair = blockIdx.x * 8 + warp;          // (row, head) index
    const bool live = pair < rows * p.H;             // warp-uniform
    const int row = pair / p.H, h = pair % p.H, n = p.fixed_len;
    const size_t base = ((size_t)(PF ? row % p.rows_real : row) * p.H + h) * p.cache_len * 64;   // K / V of the generation row
    uint4 kr[8];                                     // K of text position t0 + lane
    __half2 vr[32];                                  // V[t0 + j][2 lane .. 2 lane + 1]
    auto load_chunk = [&](int t0) {
        const int t = t0 + lane;
#pragma unroll
        for (int c = 0; c < 8; ++c)
            kr[c] = t < n ? reinterpret_cast<const uint4*>(p.kc + base + (size_t)t * 64)[c] : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int j = 0; j < 32; ++j)
            vr[j] = t0 + j < n ? *reinterpret_cast<const __half2*>(p.vc + base + (size_t)(t0 + j) * 64 + lane * 2)
                               : __floats2half2_rn(0.f, 0.f);
    };
    tl_stamp(p.timing, 0);
    if (live) load_chunk(0);
    pdl_trigger();
    pdl_wait();
    tl_stamp(p.timing, 1);
    if (!live) return;
    {
        const float* qp = p.q + (size_t)row * p.d + h * 64 + lane * 2;
        float2 part[ACB_LM_MAX_SPLIT];
#pragma unroll
        for (int s = 0; s < ACB_LM_MAX_SPLIT; ++s)   // independent loads, fixed summation order
            part[s] = s < p.q_nsplit ? *reinterpret_cast<const float2*>(qp + s * p.q_split_stride) : make_float2(0.f, 0.f);
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int s = 0; s < ACB_LM_MAX_SPLIT; ++s) { a0 += part[s].x; a1 += part[s].y; }
        qs[warp][lane * 2] = half_round(a0) * p.scale;
        qs[warp][lane * 2 + 1] = half_round(a1) * p.scale;
    }
    __syncwarp();
    tl_stamp(p.timing, 4);
    float mx = -INFINITY, l = 0.f, o0 = 0.f, o1 = 0.f;
    for (int t0 = 0; t0 < n; t0 += 32) {             // chunks of 32 text positions (online softmax across chunks)
        if (t0 > 0) load_chunk(t0);
        const int t = t0 + lane;
        float s = -INFINITY;
        if (t < n) {
            s = 0.f;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const __half2* k2 = reinterpret_cast<const __half2*>(&kr[c]);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float2 f = __half22float2(k2[e]);
                    s = fmaf(qs[warp][c * 8 + 2 * e], f.x, s);
                    s = fmaf(qs[warp][c * 8 + 2 * e + 1], f.y, s);
                }
            }
        }
        tl_stamp(p.timing, 5);
        const float cm = fmaxf(mx, warp_max(s));
        const float corr = mx == -INFINITY ? 0.f : __expf(mx - cm);
        const float pw = t < n ? __expf(s - cm) : 0.f;
        l = l * corr + warp_sum(pw);
        o0 *= corr; o1 *= corr;
        tl_stamp(p.timing, 6);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const float wj = __shfl_sync(0xffffffffu, pw, j);
            if (t0 + j < n) {
                const float2 f = __half22float2(vr[j]);
                o0 = fmaf(wj, f.x, o0);
                o1 = fmaf(wj, f.y, o1);
            }
        }
        mx = cm;
    }
    tl_stamp(p.timing, 2);
    *reinterpret_cast<__half2*>(p.out + (size_t)row * p.d + h * 64 + lane * 2) = __floats2half2_rn(o0 / l, o1 / l);
    tl_stamp(p.timing, 3);
}

// ------------------------------------------------------------------------------------------------ sampling
// Philox4x32-10 (counter-based; one 4-word block per 4 candidates) -> 24-bit uniforms -> Exponential(1).
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}
__device__ __forceinline__ float exp1_noise(uint64_t seed, uint32_t step, uint32_t stream, uint32_t i) {
    uint4 r = philox4x32_10(make_uint4(i >> 2, stream, step, 0x5a17u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    uint32_t w = (i & 3) == 0 ? r.x : ((i & 3) == 1 ? r.y : ((i & 3) == 2 ? r.z : r.w));
    float u = ((float)(w >> 8) + 0.5f) * (1.0f / 16777216.0f);  // (0,1), never 0 or 1
    return -logf(u);
}

struct SampleParams {
    const float* logits;  // [rows][n_q*card]
    const float* noise;   // [batch][n_q][card] or NULL
    float* logits_out;    // [batch][n_q][card] CFG-mixed logits or NULL
    int64_t* seq; const uint8_t* seq_mask; int* pos; int max_seq;  // in-loop write-back (seq may be NULL)
    int64_t* tokens;      // [batch][n_q] stand-alone output (may be NULL)
    int batch, rows, n_q, card, NP;
    int use_sampling, top_k; float temp, top_p, cfg_coef; uint64_t seed; uint32_t step;
    float cfg_coef_beta;   // rows == 3 * batch: double CFG (lm.py:362-376)
};

// descending order, ties by ascending index
__device__ __forceinline__ bool before(float va, int ia, float vb, int ib) { return va > vb || (va == vb && ia < ib); }

__global__ void __launch_bounds__(1024) lm_sample_kernel(SampleParams p) {
    extern __shared__ float sm[];
    float* pr = sm;                 // [card] logits -> probabilities
    float* sv = pr + p.card;        // [NP] sort values
    int* si = (int*)(sv + p.NP);    // [NP] sort indices
    __shared__ float red[3][32];
    __shared__ float bestv[32];
    __shared__ int besti[32];
    __shared__ float s_scalar;
    const int k = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
    const int card = p.card;
    const bool cfg = p.rows == 2 * p.batch, cfg3 = p.rows == 3 * p.batch;   // [cond; null] or [cond; style-only; null]
    const float* lc = p.logits + ((size_t)b * p.n_q + k) * card;
    const float* lu = p.logits + ((size_t)((cfg3 ? 2 : 1) * p.batch + b) * p.n_q + k) * card;
    const float* lw = p.logits + ((size_t)(p.batch + b) * p.n_q + k) * card;
    pdl_trigger();
    pdl_wait();
    const int cur_pos = p.pos ? p.pos[0] : 0;   // read once: the last block to finish advances it (below)
    const uint32_t step = p.pos ? (uint32_t)cur_pos : p.step;

    for (int i = tid; i < card; i += nt) {
        float l = lc[i];
        if (cfg) { float u = lu[i]; l = u + (l - u) * p.cfg_coef; }   // lm.py:399
        else if (cfg3) { const float u = lu[i], w = lw[i]; l = u + p.cfg_coef * (w + p.cfg_coef_beta * (l - w) - u); }   // lm.py:372-376
        pr[i] = l;
        if (p.logits_out) p.logits_out[((size_t)b * p.n_q + k) * card + i] = l;
    }
    __syncthreads();

    const bool sampling = p.use_sampling && p.temp > 0.f;
    bool sorted_space = false;
    if (sampling) {
        float lm = -INFINITY;
        for (int i = tid; i < card; i += nt) { float l = pr[i] / p.temp; pr[i] = l; lm = fmaxf(lm, l); }
        const float m = block_max(lm, red[0]);
        float ls = 0.f;
        for (int i = tid; i < card; i += nt) { float e = expf(pr[i] - m); pr[i] = e; ls += e; }
        const float s = block_sum(ls, red[1]);
        for (int i = tid; i < card; i += nt) pr[i] = pr[i] / s;
        __syncthreads();
        const int kk = p.top_k > card ? card : p.top_k;
        if (p.top_p <= 0.f && kk > 0) {
            // utils.sample_top_k (utils/utils.py:108-122) keeps p >= the k-th largest probability and renormalises: only
            // that VALUE is needed, so instead of sorting (66 block barriers for 2048 candidates) select it exactly with
            // a 4-pass radix select on the bit patterns (non-negative floats order like their uint32 bits).
            __shared__ int hist[256];
            __shared__ int s_bin, s_rem;
            uint32_t prefix = 0u, mask = 0u;
            int remaining = kk;                     // rank (from the top) among the candidates matching prefix/mask
#pragma unroll 1
            for (int shift = 24; shift >= 0; shift -= 8) {
                for (int i = tid; i < 256; i += nt) hist[i] = 0;
                __syncthreads();
                for (int i = tid; i < card; i += nt) {
                    const uint32_t key = __float_as_uint(pr[i]);
                    if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1);
                }
                __syncthreads();
                if (tid == 0) {
                    int acc = 0, bin = 255;
                    for (; bin > 0; --bin) {
                        if (acc + hist[bin] >= remaining) break;
                        acc += hist[bin];
                    }
                    s_bin = bin; s_rem = remaining - acc;
                }
                __syncthreads();
                prefix |= (uint32_t)s_bin << shift;
                mask |= 255u << shift;
                remaining = s_rem;
            }
            const float kth = __uint_as_float(prefix);
            float ls2 = 0.f;
            for (int i = tid; i < card; i += nt) { float v = pr[i] >= kth ? pr[i] : 0.f; pr[i] = v; ls2 += v; }
            const float s2 = block_sum(ls2, red[2]);
            for (int i = tid; i < card; i += nt) pr[i] = pr[i] / s2;
            __syncthreads();
        } else if (p.top_p > 0.f || kk > 0) {
            for (int i = tid; i < p.NP; i += nt) { sv[i] = i < card ? pr[i] : -INFINITY; si[i] = i; }
            __syncthreads();
            for (int size = 2; size <= p.NP; size <<= 1)
                for (int j = size >> 1; j > 0; j >>= 1) {
                    for (int i = tid; i < p.NP; i += nt) {
                        const int l = i ^ j;
                        if (l > i) {
                            const bool fwd = (i & size) == 0;
                            float va = sv[i], vb = sv[l];
                            int ia = si[i], ib = si[l];
                            const bool ok = before(va, ia, vb, ib);
                            if (fwd ? !ok : ok) { sv[i] = vb; sv[l] = va; si[i] = ib; si[l] = ia; }
                        }
                    }
                    __syncthreads();
                }
            if (p.top_p > 0.f) {
                // utils.sample_top_p (utils/utils.py:125-141): sequential cumsum like torch's CPU kernel
                if (tid == 0) {
                    float cum = 0.f;
                    for (int i = 0; i < card; ++i) {
                        const float v = sv[i];
                        cum += v;
                        if (cum - v > p.top_p) sv[i] = 0.f;
                    }
                }
                __syncthreads();
                float ls2 = 0.f;
                for (int i = tid; i < card; i += nt) ls2 += sv[i];
                const float s2 = block_sum(ls2, red[2]);
                for (int i = tid; i < card; i += nt) pr[i] = sv[i] / s2;  // pr now lives in sorted space
                sorted_space = true;
                __syncthreads();
            } else {
                // utils.sample_top_k (utils/utils.py:108-122): keep p >= k-th largest, renormalise
                if (tid == 0) s_scalar = sv[kk - 1];
                __syncthreads();
                const float kth = s_scalar;
                float ls2 = 0.f;
                for (int i = tid; i < card; i += nt) { float v = pr[i] >= kth ? pr[i] : 0.f; pr[i] = v; ls2 += v; }
                const float s2 = block_sum(ls2, red[2]);
                for (int i = tid; i < card; i += nt) pr[i] = pr[i] / s2;
                __syncthreads();
            }
        }
        // torch.multinomial(num_samples=1): argmax_i p_i / q_i, q ~ Exponential(1)
        for (int i = tid; i < card; i += nt) {
            const float qn = p.noise ? p.noise[((size_t)b * p.n_q + k) * card + i]
                                     : exp1_noise(p.seed, step, (uint32_t)(b * p.n_q + k), (uint32_t)i);
            pr[i] = pr[i] / qn;
        }
        __syncthreads();
    }
    // first-max argmax over pr
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = tid; i < card; i += nt) {
        const float v = pr[i];
        if (v > bv || (v == bv && i < bi)) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if ((tid & 31) == 0) { bestv[tid >> 5] = bv; besti[tid >> 5] = bi; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < (nt >> 5); ++w)
            if (bestv[w] > bv || (bestv[w] == bv && besti[w] < bi)) { bv = bestv[w]; bi = besti[w]; }
        if (bi == 0x7fffffff) bi = 0;
        int tok = sorted_space ? si[bi] : bi;
        if (p.tokens) p.tokens[(size_t)b * p.n_q + k] = tok;
        if (p.seq) {
            const int off = cur_pos + 1;
            if (off < p.max_seq) {
                if (!p.seq_mask[(size_t)k * p.max_seq + off]) tok = card;            // lm.py:555-556
                int64_t* dst = p.seq + ((size_t)b * p.n_q + k) * p.max_seq + off;
                if (*dst == -1) *dst = tok;                                           // lm.py:559-562
            }
            // the last (b, k) block to get here advances the position: pos[1] counts finished blocks
            __threadfence();
            const int done = atomicAdd(p.pos + 1, 1);
            if (done == (int)(gridDim.x * gridDim.y) - 1) { p.pos[1] = 0; p.pos[0] = cur_pos + 1; }
        }
    }
}

__global__ void lm_f32_to_f16_kernel(const float* __restrict__ src, __half* __restrict__ dst, size_t n_valid, size_t n_total) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_total) dst[i] = __float2half_rn(i < n_valid ? src[i] : 0.f);
}

// ------------------------------------------------------------------------------------------------ host side
struct acb_lm {
    acb_lm_config cfg;
    acb_lm_weights w;
    acb_lm_buffers buf;
    acb_lm_sampling samp;
    cudaStream_t capture_stream = nullptr;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    int batch = 0, rows = 0, rows_pad = 0, text_len = 0, seq_len = 0, sms = 148, smem_per_sm = 228 * 1024;
    int launches = 0;
    bool has_cross = false;
    bool pdl = true;          // programmatic dependent launch between the kernels of a step
    bool attn2 = true;        // deep-prefetch self attention (cp.async ring); ACB_LM_ATTN=v1: register loads
    bool fused = false;       // ACB_LM_STEP=fused / rotary positions: the whole transformer of a step is ONE persistent kernel (lm_step.cu)
    StepLaunch step{};
    unsigned long long* trace = nullptr;   // ACB_LM_STEP_TRACE=1: per-phase %globaltimer stamps of CTA 0
    // ACB_LM_TIMING=1 (debug): in-kernel time stamps of the layer-0 GEMMs of a directly enqueued step
    unsigned long long* timing = nullptr;
    struct TimedGemm { const char* what; int ctas; };
    std::vector<TimedGemm> timed;
};
constexpr int ACB_TIMING_MAX_CTAS = 1024, ACB_TIMING_MAX_GEMMS = 16;
constexpr size_t ACB_PLAN_COUNTER_BYTES = 4096;   // first bytes of buffers.plan: arrival counters of the split-KV attention

// Launch with (optionally) the programmatic-stream-serialization attribute: the kernel may begin while its
// predecessor in the stream is still running and synchronises itself with griddepcontrol.wait.
template <typename... KArgs, typename... Args>
static cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl,
                            Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    if (pdl) {
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
    }
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#define ACB_LAUNCH(...) ACB_CHECK_CUDA(launch_k(__VA_ARGS__))

static int nt_for_rows(int rows) { return rows <= 8 ? 1 : (rows <= 16 ? 2 : (rows <= 32 ? 4 : 8)); }

static size_t gemm_smem_bytes(int nt, int kslice, int ft2, bool staged) {
    const size_t pitch = (size_t)kslice * 2 + 64;
    return 16 * ft2 * pitch + (staged ? 8 * nt * pitch : 0) + 16 + (size_t)4 * 16 * ft2 * (8 * nt + 1) * sizeof(float);
}
// Register-load tiles stay within 120 KB so that two CTAs share an SM; staged tiles may use all an SM allows one block.
constexpr int GEMM_REG_MAX_SMEM = 120 * 1024, GEMM_MAX_SMEM = 227 * 1024;

struct GemmTiling { int ft2; bool staged; };

template <int EPI, int FT2, bool STAGED>
static int launch_gemm_ft(int nt, const GemmParams& p, int nsplit, cudaStream_t s, bool pdl) {
    dim3 grid(p.N / (16 * FT2), nsplit);
    const size_t smem = gemm_smem_bytes(nt, p.kslice, FT2, STAGED);
    ACB_REQUIRE(smem <= (size_t)GEMM_MAX_SMEM && p.N % (16 * FT2) == 0, "lm_gemm: tile does not fit (N=%d kslice=%d ft2=%d staged=%d)",
                p.N, p.kslice, FT2, (int)STAGED);
    switch (nt) {
        case 1: ACB_LAUNCH((lm_gemm_kernel<1, EPI, FT2, STAGED>), grid, dim3(128), smem, s, pdl, p); break;
        case 2: ACB_LAUNCH((lm_gemm_kernel<2, EPI, FT2, STAGED>), grid, dim3(128), smem, s, pdl, p); break;
        case 4: ACB_LAUNCH((lm_gemm_kernel<4, EPI, FT2, STAGED>), grid, dim3(128), smem, s, pdl, p); break;
        default: ACB_LAUNCH((lm_gemm_kernel<8, EPI, FT2, STAGED>), grid, dim3(128), smem, s, pdl, p); break;
    }
    return ACB_OK;
}
// The cross K/V and prefill QKV epilogues are built with 16-feature register-load tiles only.
constexpr bool gemm_epi_tiled(int epi) { return epi != EPI_CROSSKV && epi != EPI_QKV_PF; }

template <int EPI>
static int launch_gemm(int nt, const GemmParams& p, int nsplit, cudaStream_t s, bool pdl, GemmTiling t = {1, false}) {
    if constexpr (gemm_epi_tiled(EPI)) {
        if (t.staged) {
            if (t.ft2 == 3) return launch_gemm_ft<EPI, 3, true>(nt, p, nsplit, s, pdl);
            if (t.ft2 == 2) return launch_gemm_ft<EPI, 2, true>(nt, p, nsplit, s, pdl);
            return launch_gemm_ft<EPI, 1, true>(nt, p, nsplit, s, pdl);
        }
        if (t.ft2 == 2) return launch_gemm_ft<EPI, 2, false>(nt, p, nsplit, s, pdl);
    } else if (t.staged || t.ft2 != 1) {
        acb_set_error("lm_gemm: this epilogue uses 16-feature register-load tiles");
        return ACB_ERR_INVALID;
    }
    return launch_gemm_ft<EPI, 1, false>(nt, p, nsplit, s, pdl);
}

template <int NT, int EPI, int FT2, bool STAGED>
static cudaError_t gemm_attr_one() {
    cudaError_t e = cudaFuncSetAttribute(lm_gemm_kernel<NT, EPI, FT2, STAGED>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_MAX_SMEM);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(lm_gemm_kernel<NT, EPI, FT2, STAGED>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
}
template <int EPI, int FT2, bool STAGED>
static cudaError_t gemm_attr_nt() {
    cudaError_t e;
    if ((e = gemm_attr_one<1, EPI, FT2, STAGED>()) != cudaSuccess) return e;
    if ((e = gemm_attr_one<2, EPI, FT2, STAGED>()) != cudaSuccess) return e;
    if ((e = gemm_attr_one<4, EPI, FT2, STAGED>()) != cudaSuccess) return e;
    return gemm_attr_one<8, EPI, FT2, STAGED>();
}
template <int EPI>
static cudaError_t gemm_attr_all() {
    cudaError_t e;
    if ((e = gemm_attr_nt<EPI, 1, false>()) != cudaSuccess) return e;
    if constexpr (gemm_epi_tiled(EPI)) {
        if ((e = gemm_attr_nt<EPI, 2, false>()) != cudaSuccess) return e;
        if ((e = gemm_attr_nt<EPI, 1, true>()) != cudaSuccess) return e;
        if ((e = gemm_attr_nt<EPI, 2, true>()) != cudaSuccess) return e;
        if ((e = gemm_attr_nt<EPI, 3, true>()) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// Tiling of one decode GEMM, from its shape and the SM's shared memory:
//  * big GEMMs (>= 2 M weights; d x d at d = 1536 qualifies) take the narrowest of the 32- and 48-feature staged tilings whose grid
//    runs in ONE wave and still covers >= 80 % of the SMs.  With the 16-row activation block staged next to the weight slab, a
//    32-feature CTA of FFN1 / FFN2 needs ~159 KB, one per SM: 192 CTAs would be 1.3 waves, their 128 48-feature CTAs are one.
//  * other GEMMs (and every GEMM with ACB_LM_FT32=0) take 16-feature staged tiles when those run in one wave;
//  * otherwise (heads at N = 8192: 256 x 159 KB or no 48-feature split; prefill's 64-row blocks) the activations are loaded
//    into registers, with 32-feature tiles for big GEMMs when the grid covers ~90 % of the SMs and two CTAs share an SM.
// Feature tiles never change a sum (same kslice, same per-warp k ranges), so every choice is bit-identical.
static GemmTiling pick_tiling(const acb_lm* lm, int N, int K, int nsplit, int kslice, int nt) {
    const char* e = getenv("ACB_LM_FT32");
    const bool wide = !(e && e[0] == '0') && (size_t)N * K >= ((size_t)2 << 20);
    auto one_wave = [&](int ft2, bool staged) {
        const size_t smem = gemm_smem_bytes(nt, kslice, ft2, staged);
        if (N % (16 * ft2) != 0 || smem > (size_t)GEMM_MAX_SMEM) return false;
        const int per_sm = (int)((size_t)lm->smem_per_sm / (smem + 1024));   // + the 1 KB the runtime reserves per block
        return (N / (16 * ft2)) * nsplit <= lm->sms * per_sm;
    };
    if (wide) {
        for (int ft2 = 2; ft2 <= 3; ++ft2)
            if (one_wave(ft2, true) && (N / (16 * ft2)) * nsplit * 10 >= lm->sms * 8) return {ft2, true};
    } else if (one_wave(1, true)) {
        return {1, true};
    }
    if (wide && N % 32 == 0 && (N / 32) * nsplit * 10 >= lm->sms * 9 &&
        gemm_smem_bytes(nt, kslice, 2, false) <= (size_t)GEMM_REG_MAX_SMEM)
        return {2, false};
    return {1, false};
}

// K-slices per GEMM: the slab a CTA stages (16 x kslice fp16) must fit ~64 KB of shared memory, and when the
// consumer can reduce partial sums (allow_split) the matrix is cut further until there are >= 2 CTAs per SM.
// Returns nsplit (grid.y) and sets *kslice (a multiple of 32 elements).
static int pick_split(int N, int K, int sms, bool allow_split, int* kslice) {
    const int nkb = K / 32, tiles = N / 16;
    int ns = 1;
    if (allow_split) {
        ns = max(acb_ceil_div(K, 1536), acb_ceil_div(2 * sms, tiles));
        ns = max(1, min(min(ns, ACB_LM_MAX_SPLIT), nkb / 2 > 0 ? nkb / 2 : 1));
    }
    int kbs = acb_ceil_div(nkb, ns);
    ns = acb_ceil_div(nkb, kbs);   // no empty slices
    *kslice = kbs * 32;
    return ns;
}

static GemmParams base_gemm(const void* W, const void* X, int N, int K, int rows, int kslice) {
    GemmParams p{};
    p.W = (const __half*)W;
    p.X = (const __half*)X;
    p.N = N; p.K = K; p.rows = rows; p.kslice = kslice;
    return p;
}

static int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return (e && e[0]) ? atoi(e) : dflt;
}

#define ACB_TRY(expr) do { int rc_ = (expr); if (rc_ != ACB_OK) return rc_; } while (0)

// ACB_DEBUG=1: synchronise and report after every launch of a directly-enqueued step (not during graph capture).
static bool acb_debug_on() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("ACB_DEBUG"); v = (e && e[0] == '1') ? 1 : 0; }
    return v == 1;
}
static int acb_dbg(cudaStream_t s, bool capturing, const char* what, int layer) {
    if (!acb_debug_on() || capturing) return ACB_OK;
    fprintf(stderr, "[acb] %s layer %d ... ", what, layer); fflush(stderr);
    cudaError_t e = cudaStreamSynchronize(s);
    fprintf(stderr, "%s\n", cudaGetErrorString(e)); fflush(stderr);
    if (e != cudaSuccess) { acb_set_error("%s (layer %d): %s", what, layer, cudaGetErrorString(e)); return ACB_ERR_CUDA; }
    return ACB_OK;
}
#define DBG(what, layer) ACB_TRY(acb_dbg(s, capturing, what, layer))

// pf_tokens > 0: PROMPT PREFILL pass (the multi-token first call of the reference, transformer.py:240-247, 413-414, lm.py:513-534):
// the same kernels run on rows * pf_tokens (token, row) pairs -- positions pos .. pos + pf_tokens - 1 of every row at once, causal
// inside the pass because the QKV GEMM appends all of them to the cache before the attention kernel runs -- and stop after the
// last layer (no logits: the next decode step consumes the last prompt position).
static int enqueue_step_kernels(acb_lm* lm, cudaStream_t s, float* logits_out, int* n_launch, bool gemms_only,
                                bool capturing, int pf_tokens = 0) {
    const acb_lm_config& c = lm->cfg;
    const acb_lm_buffers& B = lm->buf;
    const bool pf = pf_tokens > 0;
    const int rows_real = lm->rows, rows = pf ? rows_real * pf_tokens : rows_real;
    const int d = c.dim, ffn = c.ffn_dim, L = c.num_layers, H = c.num_heads, nt = nt_for_rows(rows);
    const size_t part_stride = (size_t)(pf ? 8 * nt : lm->rows_pad) * d;
    const size_t kv_layer = (size_t)c.max_rows * H * c.max_seq * 64;
    const size_t ckv_layer = (size_t)c.max_rows * H * c.max_text * 64;
    const float scale = 1.0f / sqrtf(64.f);
    const bool pdl = lm->pdl;
    int nl = 0, ks = 0;

    // The first kernel of a step (or prefill pass) is launched WITHOUT the PDL attribute, so it starts only after everything
    // enqueued before it has completed: the previous step's sampler (which advances pos), acb_lm_begin's cross K/V GEMMs,
    // a prefill pass.  Every later kernel of the step starts after it, so within the step pos is constant and so are the cache
    // positions < pos and the cross K/V -- lm_attn2_kernel and lm_cross_attn_kernel read them before griddepcontrol.wait.
    // (A graph replay starts with the same full dependency.)
    if (!gemms_only) {
        if (pf) ACB_LAUNCH(lm_embed_kernel<true>, dim3(rows), dim3(256), 0, s, false, (const __half*)lm->w.emb, lm->w.inv_freq,
                           (const int64_t*)B.seq, (const int*)B.pos, B.x, d, c.n_q, c.card, c.max_seq, lm->batch, c.pos_scale, rows_real);
        else ACB_LAUNCH(lm_embed_kernel<false>, dim3(rows), dim3(256), 0, s, false, (const __half*)lm->w.emb, lm->w.inv_freq,
                        (const int64_t*)B.seq, (const int*)B.pos, B.x, d, c.n_q, c.card, c.max_seq, lm->batch, c.pos_scale, rows);
        ++nl;
        DBG("lm_embed_kernel", -1);
    }
    // (An L2 prefetch chain -- every GEMM pulling the NEXT GEMM's weights into L2 with cp.async.bulk.prefetch.L2 -- was
    //  built and measured: 2.240 vs 2.258 ms per step, i.e. nothing: under PDL the weight slab is already in flight before
    //  the dependency resolves, weights are not on the critical path.  profiles/r1_perf_step_v5_l2prefetch_no_gain.log)
    enum { G_QKV, G_O, G_CQ, G_CO, G_FF1, G_FF2, G_HEADS };
    // split-KV self attention: records and counters live in the (otherwise chain-mode-only) plan buffer
    // OFF by default (ACB_LM_ATT_SPLIT=3 enables): measured on the 30 s workload it gains 2.8 % per step at KV 1500 and
    // 0.5 % at 1126 but the 768 extra (idle) CTAs per launch and the larger kernel cost 1-4 % per step below ~800
    // positions -- 53.0 vs 54.1 audio-s/s over the whole generation (profiles/r1_perf_step_v8_splitkv_*.log).
    int att_split = env_int("ACB_LM_ATT_SPLIT", 1);
    if (att_split < 1 || att_split > 8 || !B.plan ||
        ACB_PLAN_COUNTER_BYTES + (size_t)rows * H * att_split * 66 * sizeof(float) > ACB_LM_PLAN_BYTES ||
        (size_t)rows * H * sizeof(int) > ACB_PLAN_COUNTER_BYTES)
        att_split = 1;
    // debug timeline (ACB_LM_TIMING=1): every kernel of layer 0 of a directly enqueued step gets a stamp buffer
    if (lm->timing && !capturing) lm->timed.clear();
    auto tl = [&](const char* what, int layer, int ctas) -> unsigned long long* {
        if (!lm->timing || capturing || gemms_only || layer != 0 || (int)lm->timed.size() >= ACB_TIMING_MAX_GEMMS ||
            ctas > ACB_TIMING_MAX_CTAS)
            return nullptr;
        unsigned long long* t = lm->timing + (size_t)lm->timed.size() * ACB_TIMING_MAX_CTAS * 8;
        lm->timed.push_back({what, ctas});
        return t;
    };
    int pending = 0;  // split-K partial sums waiting to be folded into x by the next LN
    auto ln_launch = [&](const float* gamma, const float* beta, int layer) -> int {
        if (gemms_only) return ACB_OK;
        ACB_LAUNCH(lm_ln_kernel, dim3(rows), dim3(LN_THREADS), 0, s, pdl, B.x, (const float*)B.part, pending, part_stride, gamma, beta,
                   (__half*)B.h16, d, tl("ln", layer, rows));
        ++nl;
        DBG("lm_ln_kernel", layer);
        return ACB_OK;
    };
    auto partial_gemm = [&](const __half* W, const void* X, int N, int K, int layer, int id) -> int {
        const int ns = pick_split(N, K, lm->sms, true, &ks);
        GemmParams p = base_gemm(W, X, N, K, rows, ks);
        p.out_f32 = B.part; p.ld_out = N; p.split_stride = part_stride;
        const GemmTiling t = pick_tiling(lm, N, K, ns, ks, nt);
        p.timing = tl(id == G_O ? "gemm_O" : (id == G_CQ ? "gemm_CQ" : (id == G_CO ? "gemm_CO" : "gemm_FFN2")), layer, (N / (16 * t.ft2)) * ns);
        ACB_TRY(launch_gemm<EPI_PARTIAL>(nt, p, ns, s, pdl, t));
        ++nl;
        DBG("gemm_EPI_PARTIAL", layer);
        pending = ns;
        return ACB_OK;
    };
    for (int l = 0; l < L; ++l) {
        const float* ln = lm->w.ln + (size_t)l * 6 * d;
        // --- self attention
        ACB_TRY(ln_launch(ln, ln + d, l));
        {
            pick_split(3 * d, d, lm->sms, false, &ks);
            GemmParams p = base_gemm((const __half*)lm->w.w_qkv + (size_t)l * 3 * d * d, B.h16, 3 * d, d, rows, ks);
            p.q32 = B.q32; p.kc = (__half*)B.k_cache + l * kv_layer; p.vc = (__half*)B.v_cache + l * kv_layer;
            p.d = d; p.H = H; p.cache_len = c.max_seq; p.pos = B.pos; p.rows_real = rows_real;
            const GemmTiling t = pf ? GemmTiling{1, false} : pick_tiling(lm, 3 * d, d, 1, ks, nt);
            p.timing = tl("gemm_QKV", l, 3 * d / (16 * t.ft2));
            if (pf) ACB_TRY(launch_gemm<EPI_QKV_PF>(nt, p, 1, s, pdl, t));
            else ACB_TRY(launch_gemm<EPI_QKV>(nt, p, 1, s, pdl, t));
            ++nl;
            DBG("gemm_EPI_QKV", l);
        }
        if (!gemms_only) {
            AttnParams a{B.q32, 1, 0, (__half*)B.k_cache + l * kv_layer, (__half*)B.v_cache + l * kv_layer, (__half*)B.a16,
                         H, d, c.max_seq, B.pos, 0, scale};
            a.timing = tl("attn", l, H * rows * att_split);
            a.part = reinterpret_cast<float*>((unsigned char*)B.plan + ACB_PLAN_COUNTER_BYTES);
            a.counter = reinterpret_cast<int*>(B.plan);
            a.split_min = max(129, env_int("ACB_LM_ATT_SPLIT_MIN", 768));
            a.rows_real = rows_real;
            if (pf) ACB_LAUNCH((lm_attn_kernel<false, true>), dim3(H, rows), dim3(ATT_WARPS * 32), 0, s, pdl, a);
            else if (att_split <= 1 && lm->attn2)
                ACB_LAUNCH(lm_attn2_kernel, dim3(H, rows), dim3(ATT_WARPS * 32), (size_t)ATT_WARPS * ATT2_DEPTH * 1024, s, pdl, a);
            else if (att_split > 1) ACB_LAUNCH(lm_attn_kernel<true>, dim3(H, rows, att_split), dim3(ATT_WARPS * 32), 0, s, pdl, a);
            else ACB_LAUNCH(lm_attn_kernel<false>, dim3(H, rows), dim3(ATT_WARPS * 32), 0, s, pdl, a);
            ++nl;
            DBG("lm_attn_kernel", l);
        }
        ACB_TRY(partial_gemm((const __half*)lm->w.w_o + (size_t)l * d * d, B.a16, d, d, l, G_O));
        // --- cross attention
        if (lm->has_cross) {
            ACB_TRY(ln_launch(ln + 2 * d, ln + 3 * d, l));
            ACB_TRY(partial_gemm((const __half*)lm->w.w_cq + (size_t)l * d * d, B.h16, d, d, l, G_CQ));
            const int nsq = pending;
            pending = 0;   // these partials are the cross-attention queries, not a residual update
            if (!gemms_only) {
                AttnParams a{B.part, nsq, part_stride, (__half*)B.ck_cache + l * ckv_layer,
                             (__half*)B.cv_cache + l * ckv_layer, (__half*)B.a16, H, d, c.max_text, B.pos, lm->text_len,
                             scale};
                a.timing = tl("cross_attn", l, acb_ceil_div(rows * H, 8));
                a.rows_real = rows_real;
                if (pf) ACB_LAUNCH(lm_cross_attn_kernel<true>, dim3(acb_ceil_div(rows * H, 8)), dim3(256), 0, s, pdl, a, rows);
                else ACB_LAUNCH(lm_cross_attn_kernel<false>, dim3(acb_ceil_div(rows * H, 8)), dim3(256), 0, s, pdl, a, rows);
                ++nl;
                DBG("lm_cross_attn_kernel", l);
            }
            ACB_TRY(partial_gemm((const __half*)lm->w.w_co + (size_t)l * d * d, B.a16, d, d, l, G_CO));
        }
        // --- feed forward
        ACB_TRY(ln_launch(ln + 4 * d, ln + 5 * d, l));
        {
            pick_split(ffn, d, lm->sms, false, &ks);
            GemmParams p = base_gemm((const __half*)lm->w.w_ff1 + (size_t)l * ffn * d, B.h16, ffn, d, rows, ks);
            p.out_f16 = (__half*)B.f16; p.ld_out = ffn;
            const GemmTiling t = pick_tiling(lm, ffn, d, 1, ks, nt);
            p.timing = tl("gemm_FFN1", l, ffn / (16 * t.ft2));
            ACB_TRY(launch_gemm<EPI_GELU>(nt, p, 1, s, pdl, t)); ++nl;
            DBG("gemm_EPI_GELU", l);
        }
        ACB_TRY(partial_gemm((const __half*)lm->w.w_ff2 + (size_t)l * d * ffn, B.f16, d, ffn, l, G_FF2));
    }
    if (pf) {   // no output norm / heads / sampler: the pass only fills the KV cache
        if (n_launch) *n_launch = nl;
        return ACB_OK;
    }
    ACB_TRY(ln_launch(lm->w.out_norm, lm->w.out_norm + d, -1));
    {
        const int N = c.n_q * c.card;
        pick_split(N, d, lm->sms, false, &ks);
        GemmParams p = base_gemm(lm->w.heads, B.h16, N, d, rows, ks);
        p.out_f32 = B.logits; p.ld_out = N;
        ACB_TRY(launch_gemm<EPI_F32>(nt, p, 1, s, pdl, pick_tiling(lm, N, d, 1, ks, nt))); ++nl;
        DBG("gemm_EPI_F32", -1);
    }
    if (!gemms_only) {
        int NP = 1;
        while (NP < c.card) NP <<= 1;
        SampleParams sp{B.logits, lm->samp.noise_from_buffer ? B.noise : nullptr, logits_out, B.seq, B.seq_mask, B.pos,
                        c.max_seq, nullptr, lm->batch, rows, c.n_q, c.card, NP, lm->samp.use_sampling, lm->samp.top_k,
                        lm->samp.temp, lm->samp.top_p, lm->samp.cfg_coef, lm->samp.seed, 0, lm->samp.cfg_coef_beta};
        size_t smem = ((size_t)c.card + 2 * (size_t)NP) * sizeof(float);
        ACB_LAUNCH(lm_sample_kernel, dim3(c.n_q, lm->batch), dim3(1024), smem, s, pdl, sp);
        ++nl;
        DBG("lm_sample_kernel", -1);
    }
    if (n_launch) *n_launch = nl;
    return ACB_OK;
}

// Fused step: [memset of the barrier counter] -> lm_step_kernel (embed ... logits) -> lm_sample_kernel.
static int enqueue_step_fused(acb_lm* lm, cudaStream_t s, float* logits_out, int* n_launch, bool step_only, bool capturing) {
    const acb_lm_config& c = lm->cfg;
    const acb_lm_buffers& B = lm->buf;
    int nl = 0;
    ACB_TRY(lm_step_launch(lm->step, s));
    ++nl;
    DBG("lm_step_kernel", -1);
    if (!step_only) {
        int NP = 1;
        while (NP < c.card) NP <<= 1;
        SampleParams sp{B.logits, lm->samp.noise_from_buffer ? B.noise : nullptr, logits_out, B.seq, B.seq_mask, B.pos,
                        c.max_seq, nullptr, lm->batch, lm->rows, c.n_q, c.card, NP, lm->samp.use_sampling, lm->samp.top_k,
                        lm->samp.temp, lm->samp.top_p, lm->samp.cfg_coef, lm->samp.seed, 0, lm->samp.cfg_coef_beta};
        size_t smem = ((size_t)c.card + 2 * (size_t)NP) * sizeof(float);
        ACB_LAUNCH(lm_sample_kernel, dim3(c.n_q, lm->batch), dim3(1024), smem, s, false, sp);
        ++nl;
        DBG("lm_sample_kernel", -1);
    }
    if (n_launch) *n_launch = nl;
    return ACB_OK;
}

static int enqueue_step(acb_lm* lm, cudaStream_t s, float* logits_out, int* n_launch, bool gemms_only = false,
                        bool capturing = false) {
    if (lm->fused) return enqueue_step_fused(lm, s, logits_out, n_launch, gemms_only, capturing);
    return enqueue_step_kernels(lm, s, logits_out, n_launch, gemms_only, capturing);
}

extern "C" int acb_lm_create(const acb_lm_config* cfg, const acb_lm_weights* w, const acb_lm_buffers* buf, acb_lm_t** out) {
    ACB_REQUIRE(cfg && w && buf && out, "acb_lm_create: null argument");
    ACB_REQUIRE(cfg->dim % 64 == 0 && cfg->dim == cfg->num_heads * 64, "acb_lm_create: head_dim must be 64 (dim=%d heads=%d)",
                cfg->dim, cfg->num_heads);
    ACB_REQUIRE(cfg->dim <= 4 * LN_THREADS, "acb_lm_create: dim %d too large for the LayerNorm kernel", cfg->dim);
    ACB_REQUIRE(cfg->ffn_dim % 32 == 0 && cfg->card % 16 == 0 && cfg->n_q >= 1 && cfg->n_q <= 16, "acb_lm_create: bad ffn/card/n_q");
    ACB_REQUIRE(cfg->card <= 4096, "acb_lm_create: card %d > 4096 not built", cfg->card);
    ACB_REQUIRE(cfg->max_rows >= 1 && cfg->max_rows <= 64, "acb_lm_create: max_rows %d not in [1,64]", cfg->max_rows);
    ACB_REQUIRE(cfg->max_seq >= 2 && cfg->max_seq <= 12000, "acb_lm_create: max_seq %d out of range", cfg->max_seq);
    ACB_REQUIRE(cfg->dim <= 2048, "acb_lm_create: dim %d > 2048: the GEMM stages a 16 x dim weight slab per CTA", cfg->dim);
    acb_lm* lm = new (std::nothrow) acb_lm();
    ACB_REQUIRE(lm, "acb_lm_create: out of host memory");
    lm->cfg = *cfg; lm->w = *w; lm->buf = *buf;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&lm->sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&lm->smem_per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    cudaError_t e = cudaStreamCreateWithFlags(&lm->capture_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete lm; acb_set_error("acb_lm_create: cudaStreamCreate: %s", cudaGetErrorString(e)); return ACB_ERR_CUDA; }
    // the GEMMs stage up to ~210 KB of weights and activations per CTA; keep the shared-memory carve-out at its maximum for every kernel
    // of the step so that co-resident kernels (PDL) never force an L1/shared reconfiguration.
    cudaError_t ea = gemm_attr_all<EPI_PARTIAL>();
    if (ea == cudaSuccess) ea = gemm_attr_all<EPI_QKV>();
    if (ea == cudaSuccess) ea = gemm_attr_all<EPI_GELU>();
    if (ea == cudaSuccess) ea = gemm_attr_all<EPI_F32>();
    if (ea == cudaSuccess) ea = gemm_attr_all<EPI_CROSSKV>();
    if (ea == cudaSuccess) ea = gemm_attr_all<EPI_QKV_PF>();
    if (ea == cudaSuccess) ea = cudaFuncSetAttribute(lm_attn_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (ea == cudaSuccess) ea = cudaFuncSetAttribute(lm_attn_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (ea == cudaSuccess) ea = cudaFuncSetAttribute(lm_attn2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_WARPS * ATT2_DEPTH * 1024);
    if (ea == cudaSuccess) ea = cudaFuncSetAttribute(lm_attn2_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (ea == cudaSuccess) ea = cudaFuncSetAttribute(lm_cross_attn_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (ea == cudaSuccess) ea = cudaFuncSetAttribute(lm_ln_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (ea == cudaSuccess) ea = cudaFuncSetAttribute(lm_embed_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (ea == cudaSuccess) ea = cudaFuncSetAttribute(lm_sample_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (ea != cudaSuccess) {
        acb_set_error("acb_lm_create: cudaFuncSetAttribute: %s", cudaGetErrorString(ea));
        cudaStreamDestroy(lm->capture_stream);
        delete lm;
        return ACB_ERR_CUDA;
    }
    *out = lm;
    return ACB_OK;
}

static void drop_graph(acb_lm* lm) {
    if (lm->exec) { cudaGraphExecDestroy(lm->exec); lm->exec = nullptr; }
    if (lm->graph) { cudaGraphDestroy(lm->graph); lm->graph = nullptr; }
}

extern "C" int acb_lm_destroy(acb_lm_t* lm) {
    if (!lm) return ACB_OK;
    drop_graph(lm);
    if (lm->capture_stream) cudaStreamDestroy(lm->capture_stream);
    if (lm->timing) cudaFree(lm->timing);
    if (lm->trace) cudaFree(lm->trace);
    delete lm;
    return ACB_OK;
}

extern "C" int acb_lm_begin(acb_lm_t* lm, const float* cross, int batch, int rows, int text_len, int seq_len,
                            const acb_lm_sampling* sampling, void* stream) {
    ACB_REQUIRE(lm && sampling, "acb_lm_begin: null argument");
    const acb_lm_config& c = lm->cfg;
    ACB_REQUIRE(batch >= 1 && (rows == batch || rows == 2 * batch || rows == 3 * batch), "acb_lm_begin: rows must be batch, 2*batch (CFG) or 3*batch (double CFG)");
    ACB_REQUIRE(rows <= c.max_rows, "acb_lm_begin: rows %d > max_rows %d", rows, c.max_rows);
    ACB_REQUIRE(seq_len >= 2 && seq_len <= c.max_seq, "acb_lm_begin: seq_len %d > max_seq %d", seq_len, c.max_seq);
    ACB_REQUIRE(!c.cross_attention || cross, "acb_lm_begin: the model has cross attention, a condition tensor is required"
                " (the reference asserts the same, transformer.py:553-556)");
    ACB_REQUIRE(!cross || (text_len >= 1 && text_len <= c.max_text), "acb_lm_begin: text_len %d out of range", text_len);
    cudaStream_t s = (cudaStream_t)stream;
    lm->batch = batch; lm->rows = rows; lm->rows_pad = 8 * nt_for_rows(rows); lm->text_len = text_len; lm->seq_len = seq_len;
    lm->samp = *sampling;
    lm->has_cross = c.cross_attention && cross;
    const int d = c.dim, H = c.num_heads;
    // zero the padded activation rows once; kernels only ever write rows < `rows`
    ACB_CHECK_CUDA(cudaMemsetAsync(lm->buf.h16, 0, (size_t)lm->rows_pad * d * sizeof(__half), s));
    ACB_CHECK_CUDA(cudaMemsetAsync(lm->buf.a16, 0, (size_t)lm->rows_pad * d * sizeof(__half), s));
    ACB_CHECK_CUDA(cudaMemsetAsync(lm->buf.f16, 0, (size_t)lm->rows_pad * c.ffn_dim * sizeof(__half), s));
    int hp[4] = {0, 0, batch, text_len};   // pos, finished-block counter of the sampler, (info) batch, text_len
    ACB_CHECK_CUDA(cudaMemcpyAsync(lm->buf.pos, hp, sizeof(hp), cudaMemcpyHostToDevice, s));
    if (lm->has_cross) {
        const size_t M = (size_t)rows * text_len, Mpad = (M + 63) / 64 * 64;
        lm_f32_to_f16_kernel<<<(unsigned)((Mpad * d + 255) / 256), 256, 0, s>>>(cross, (__half*)lm->buf.cross16, M * d, Mpad * d);
        ACB_LAUNCH_CHECK();
        const size_t ckv_layer = (size_t)c.max_rows * H * c.max_text * 64;
        for (int l = 0; l < c.num_layers; ++l)
            for (size_t r0 = 0; r0 < M; r0 += 64) {
                int ks = 0;
                pick_split(2 * d, d, lm->sms, false, &ks);
                GemmParams p = base_gemm((const __half*)lm->w.w_ckv + (size_t)l * 2 * d * d,
                                         (const __half*)lm->buf.cross16 + r0 * d, 2 * d, d, (int)min((size_t)64, M - r0), ks);
                p.kc = (__half*)lm->buf.ck_cache + l * ckv_layer; p.vc = (__half*)lm->buf.cv_cache + l * ckv_layer;
                p.d = d; p.H = H; p.cache_len = c.max_text; p.text_len = text_len; p.row0 = (int)r0;
                ACB_TRY(launch_gemm<EPI_CROSSKV>(8, p, 1, s, false));
            }
    }
    // opt in to large dynamic shared memory where needed
    {
        int NP = 1;
        while (NP < c.card) NP <<= 1;
        size_t smem = ((size_t)c.card + 2 * (size_t)NP) * sizeof(float);
        if (smem > 48 * 1024)
            ACB_CHECK_CUDA(cudaFuncSetAttribute(lm_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    // capture one decode step (with programmatic dependent launch edges; plain edges if the driver refuses them)
    {
        const char* e = getenv("ACB_NO_PDL");
        lm->pdl = !(e && e[0] == '1');
        if (env_int("ACB_LM_TIMING", 0) && !lm->timing) {
            ACB_CHECK_CUDA(cudaMalloc(&lm->timing, (size_t)ACB_TIMING_MAX_GEMMS * ACB_TIMING_MAX_CTAS * 64));
            ACB_CHECK_CUDA(cudaMemset(lm->timing, 0, (size_t)ACB_TIMING_MAX_GEMMS * ACB_TIMING_MAX_CTAS * 64));
        }
        {
            const char* ea = getenv("ACB_LM_ATTN");
            lm->attn2 = !(ea && ea[0] == 'v' && ea[1] == '1');
        }
        const char* ev = getenv("ACB_LM_STEP");
        // The persistent fused step (lm_step.cu; needs the packed weights) is OPT-IN: ACB_LM_STEP=fused, or a model with rotary
        // positions (only built there).  Measured 3.1 ms vs 2.03 ms per step at KV length 1 for the per-phase graph below
        // (DESIGN.md section 3.1: ~2.3 us of grid barrier + skew per phase against 0.9 us per PDL kernel boundary).
        lm->fused = lm->w.wp_qkv != nullptr && ((ev && ev[0] == 'f') || c.positional_embedding != 0);
        ACB_REQUIRE(c.positional_embedding == 0 || lm->fused, "acb_lm_begin: rotary positions are built in the fused decode step only");
        if (lm->fused) {
            ACB_TRY(lm_step_prepare(c, lm->w, lm->buf, rows, batch, text_len, lm->has_cross, lm->sms, &lm->step));
            if (env_int("ACB_LM_COOP", 1) == 0) lm->step.cooperative = false;
            if (env_int("ACB_LM_STEP_TRACE", 0)) {
                if (!lm->trace) ACB_CHECK_CUDA(cudaMalloc(&lm->trace, 8192 * sizeof(unsigned long long)));
                ACB_CHECK_CUDA(cudaMemset(lm->trace, 0, 8192 * sizeof(unsigned long long)));
                ACB_REQUIRE(lm->step.n_phases + 2 <= 1024, "trace buffer too small");
            }
        }
        if (lm->buf.plan) ACB_CHECK_CUDA(cudaMemsetAsync(lm->buf.plan, 0, ACB_PLAN_COUNTER_BYTES, s));   // split-KV arrival counters
    }
    for (int attempt = 0; attempt < 2; ++attempt) {
        drop_graph(lm);
        ACB_CHECK_CUDA(cudaStreamBeginCapture(lm->capture_stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue_step(lm, lm->capture_stream, nullptr, &lm->launches, false, true);
        cudaError_t e = cudaStreamEndCapture(lm->capture_stream, &lm->graph);
        if (rc == ACB_OK && e == cudaSuccess) e = cudaGraphInstantiate(&lm->exec, lm->graph, 0);
        if (rc == ACB_OK && e == cudaSuccess && env_int("ACB_LM_GRAPH_INFO", 0)) {   // how many edges are programmatic (PDL)?
            size_t ne = 0;
            if (cudaGraphGetEdges_v2(lm->graph, nullptr, nullptr, nullptr, &ne) == cudaSuccess && ne) {
                std::vector<cudaGraphNode_t> from(ne), to(ne);
                std::vector<cudaGraphEdgeData> ed(ne);
                size_t prog = 0, port_prog = 0;
                if (cudaGraphGetEdges_v2(lm->graph, from.data(), to.data(), ed.data(), &ne) == cudaSuccess)
                    for (size_t i = 0; i < ne; ++i) {
                        prog += ed[i].type == cudaGraphDependencyTypeProgrammatic;
                        port_prog += ed[i].from_port == cudaGraphKernelNodePortProgrammatic;
                    }
                fprintf(stderr, "[acb graph] %zu edges, %zu programmatic (from_port programmatic: %zu), pdl=%d\n", ne, prog, port_prog, (int)lm->pdl);
            }
            cudaGetLastError();
        }
        if (rc == ACB_OK && e == cudaSuccess) return ACB_OK;
        cudaGetLastError();
        drop_graph(lm);
        if (lm->fused && lm->step.cooperative && attempt == 0) { lm->step.cooperative = false; continue; }   // plain launch (grid = #SMs is co-resident anyway)
        if (!lm->pdl || attempt == 1) {
            if (rc == ACB_OK) acb_set_error("acb_lm_begin: graph capture failed: %s", cudaGetErrorString(e));
            return rc != ACB_OK ? rc : ACB_ERR_CUDA;
        }
        lm->pdl = false;   // retry without programmatic edges
    }
    return ACB_OK;
}

__global__ void lm_set_pos_kernel(int* pos, int value) { pos[0] = value; }

// Prompt prefill: consume sequence positions [pos0, pos0 + n_tokens) of every row (their tokens are already in buffers.seq)
// without sampling, ACB_LM_PREFILL_ROWS / rows positions per pass.  Leaves pos = pos0 + n_tokens on the device.
extern "C" int acb_lm_prefill(acb_lm_t* lm, int pos0, int n_tokens, void* stream) {
    ACB_REQUIRE(lm && lm->rows > 0, "acb_lm_prefill: call acb_lm_begin first");
    ACB_REQUIRE(!lm->fused, "acb_lm_prefill: the prefill pass is built on the per-phase kernels");
    ACB_REQUIRE(pos0 >= 0 && n_tokens >= 0 && pos0 + n_tokens < lm->seq_len, "acb_lm_prefill: positions [%d, %d) exceed the sequence (%d)",
                pos0, pos0 + n_tokens, lm->seq_len);
    cudaStream_t s = (cudaStream_t)stream;
    const acb_lm_config& c = lm->cfg;
    const int d = c.dim, per = ACB_LM_PREFILL_ROWS / lm->rows;
    ACB_REQUIRE(per >= 1, "acb_lm_prefill: rows %d > %d", lm->rows, ACB_LM_PREFILL_ROWS);
    int done = 0;
    while (done < n_tokens) {
        const int tc = n_tokens - done < per ? n_tokens - done : per;
        const int vrows = lm->rows * tc, pad = 8 * nt_for_rows(vrows);
        lm_set_pos_kernel<<<1, 1, 0, s>>>(lm->buf.pos, pos0 + done);
        ACB_LAUNCH_CHECK();
        if (pad > vrows) {   // the GEMMs read their activation rows up to the tile height: rows >= vrows must be zero
            ACB_CHECK_CUDA(cudaMemsetAsync((__half*)lm->buf.h16 + (size_t)vrows * d, 0, (size_t)(pad - vrows) * d * sizeof(__half), s));
            ACB_CHECK_CUDA(cudaMemsetAsync((__half*)lm->buf.a16 + (size_t)vrows * d, 0, (size_t)(pad - vrows) * d * sizeof(__half), s));
            ACB_CHECK_CUDA(cudaMemsetAsync((__half*)lm->buf.f16 + (size_t)vrows * c.ffn_dim, 0, (size_t)(pad - vrows) * c.ffn_dim * sizeof(__half), s));
        }
        ACB_TRY(enqueue_step_kernels(lm, s, nullptr, nullptr, false, false, tc));
        done += tc;
    }
    lm_set_pos_kernel<<<1, 1, 0, s>>>(lm->buf.pos, pos0 + n_tokens);
    ACB_LAUNCH_CHECK();
    // back to decode: its padded rows [rows, rows_pad) must be zero again
    if (lm->rows_pad > lm->rows) {
        ACB_CHECK_CUDA(cudaMemsetAsync((__half*)lm->buf.h16 + (size_t)lm->rows * d, 0, (size_t)(lm->rows_pad - lm->rows) * d * sizeof(__half), s));
        ACB_CHECK_CUDA(cudaMemsetAsync((__half*)lm->buf.a16 + (size_t)lm->rows * d, 0, (size_t)(lm->rows_pad - lm->rows) * d * sizeof(__half), s));
        ACB_CHECK_CUDA(cudaMemsetAsync((__half*)lm->buf.f16 + (size_t)lm->rows * c.ffn_dim, 0, (size_t)(lm->rows_pad - lm->rows) * c.ffn_dim * sizeof(__half), s));
    }
    return ACB_OK;
}

extern "C" int acb_lm_uses_pdl(const acb_lm_t* lm) { return lm && lm->pdl ? 1 : 0; }

extern "C" int acb_lm_steps(acb_lm_t* lm, int n_steps, void* stream) {
    ACB_REQUIRE(lm && lm->exec, "acb_lm_steps: call acb_lm_begin first");
    ACB_REQUIRE(n_steps >= 0, "acb_lm_steps: negative step count");
    for (int i = 0; i < n_steps; ++i) ACB_CHECK_CUDA(cudaGraphLaunch(lm->exec, (cudaStream_t)stream));
    return ACB_OK;
}

// Debug timeline of the default step's layer-0 kernels (%globaltimer, ns, relative to the first CTA of the first kernel):
// CTA starts (first..last), when griddepcontrol.wait returned (median), the kernel's mid stamp (GEMM: weights + k-loop
// done; median), CTA ends (median..last).
static int report_timeline(acb_lm* lm, cudaStream_t s) {
    ACB_CHECK_CUDA(cudaStreamSynchronize(s));
    std::vector<unsigned long long> h((size_t)ACB_TIMING_MAX_CTAS * 8);
    unsigned long long t0 = 0;
    for (size_t gi = 0; gi < lm->timed.size(); ++gi) {
        const int n = lm->timed[gi].ctas;
        ACB_CHECK_CUDA(cudaMemcpy(h.data(), lm->timing + gi * ACB_TIMING_MAX_CTAS * 8, (size_t)n * 64, cudaMemcpyDeviceToHost));
        std::vector<long long> col[8];
        for (int i = 0; i < n; ++i)
            for (int sl = 0; sl < 8; ++sl)
                if (h[i * 8 + sl]) col[sl].push_back((long long)h[i * 8 + sl]);
        for (auto& v : col) std::sort(v.begin(), v.end());
        if (col[0].empty() || col[1].empty() || col[3].empty()) continue;
        if (!t0) t0 = (unsigned long long)col[0].front();
        const long long w = col[1][col[1].size() / 2];   // median wait-return
        fprintf(stderr, "[acb timeline] %-10s %4d CTAs  start %6lld..%6lld  wait-returned %6lld  end %6lld (med) %6lld (max) | after wait [ns, median]:",
                lm->timed[gi].what, n, col[0].front() - (long long)t0, col[0].back() - (long long)t0, w - (long long)t0,
                col[3][col[3].size() / 2] - (long long)t0, col[3].back() - (long long)t0);
        static const int order[6] = {4, 5, 6, 7, 2, 3};   // stamps in program order (2 = main loop done, 3 = end)
        for (int oi = 0; oi < 6; ++oi) {
            const std::vector<long long>& v = col[order[oi]];
            if (!v.empty()) fprintf(stderr, "  s%d %lld", order[oi], v[v.size() / 2] - w);
        }
        fprintf(stderr, "\n");
    }
    ACB_CHECK_CUDA(cudaMemset(lm->timing, 0, (size_t)ACB_TIMING_MAX_GEMMS * ACB_TIMING_MAX_CTAS * 64));
    return ACB_OK;
}

// ACB_LM_STEP_TRACE=1: time between consecutive grid barriers of the fused step as seen by CTA 0 (ns), summed per phase kind.
static int report_step_trace(acb_lm* lm, cudaStream_t s) {
    ACB_CHECK_CUDA(cudaStreamSynchronize(s));
    const int n = lm->step.n_phases;
    std::vector<unsigned long long> h((size_t)n + 1);
    ACB_CHECK_CUDA(cudaMemcpy(h.data(), lm->trace, ((size_t)n) * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    const bool cross = lm->has_cross;
    const int per = cross ? 12 : 8;
    static const char* names_c[12] = {"qkv", "attn", "o", "res1", "cq", "xattn", "co", "res2", "ff1", "gelu", "ff2", "res3"};
    static const char* names_n[8] = {"qkv", "attn", "o", "res1", "ff1", "gelu", "ff2", "res3"};
    double sum[12] = {0}, mx[12] = {0};
    for (int l = 0; l < lm->cfg.num_layers; ++l)
        for (int k = 0; k < per; ++k) {
            const int i = 1 + l * per + k;     // stamp i is taken after barrier i; phase k of layer l ends at barrier 1 + l*per + k + 1
            if (i + 1 >= n || !h[i] || !h[i + 1]) continue;
            const double dt = (double)(h[i + 1] - h[i]);
            sum[k] += dt; if (dt > mx[k]) mx[k] = dt;
        }
    fprintf(stderr, "[acb step trace] rows=%d pos=? total %.1f us (kernel start -> last barrier); embed %.2f us; per-layer mean (max) us:",
            lm->rows, (double)(h[n - 1] - h[0]) * 1e-3, (double)(h[1] - h[0]) * 1e-3);
    for (int k = 0; k < per; ++k)
        fprintf(stderr, "  %s %.2f (%.2f)", cross ? names_c[k] : names_n[k], sum[k] * 1e-3 / lm->cfg.num_layers, mx[k] * 1e-3);
    fprintf(stderr, "\n");
    {   // sub-steps of the GEMM phases (the CTA running item 0): ns from phase start to stats / A-load done / MMAs issued / accumulator ready / epilogue done
        std::vector<unsigned long long> f(8192);
        ACB_CHECK_CUDA(cudaMemcpy(f.data(), lm->trace, 8192 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        static const int gk_c[6] = {0, 2, 4, 6, 8, 10}, gk_n[4] = {0, 2, 4, 6};
        const int ng = cross ? 6 : 4;
        fprintf(stderr, "[acb step trace] GEMM sub-steps, mean ns after the phase's first stamp [stats, aload, mma-issued, acc-ready, epilogue]; first stamp - barrier stamp:\n");
        for (int gi = 0; gi < ng; ++gi) {
            const int k = cross ? gk_c[gi] : gk_n[gi];
            double acc[6] = {0}; int cnt = 0; double lag = 0;
            for (int l = 0; l < lm->cfg.num_layers; ++l) {
                const int ph = 1 + l * per + k;          // barrier count when the phase starts
                if (1024 + 8 * ph + 5 >= 8192) break;
                const unsigned long long* q = f.data() + 1024 + 8 * ph;
                if (!q[0] || !q[5]) continue;
                for (int j = 1; j < 6; ++j) acc[j] += q[j] ? (double)(q[j] - q[0]) : 0.0;
                lag += (double)q[0] - (double)h[ph];
                ++cnt;
            }
            if (cnt) fprintf(stderr, "    %-4s  %.0f %.0f %.0f %.0f %.0f   (start lag %.0f ns, %d layers)\n", cross ? names_c[k] : names_n[k],
                             acc[1] / cnt, acc[2] / cnt, acc[3] / cnt, acc[4] / cnt, acc[5] / cnt, lag / cnt, cnt);
        }
    }
    {   // per-K-block stamps of the layer-1 QKV and FF2 GEMMs: [loop top -> full barrier passed -> MMAs + commit issued]
        std::vector<unsigned long long> f(8192);
        ACB_CHECK_CUDA(cudaMemcpy(f.data(), lm->trace, 8192 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        for (int which = 0; which < 2; ++which) {
            const unsigned long long* q = f.data() + 6000 + which * 64;
            if (!q[0]) continue;
            fprintf(stderr, "[acb step trace] %s layer 1, per K block ns since loop start (top, data ready, issued):", which ? "ff2" : "qkv");
            for (int kb = 0; kb < 12 && q[3 * kb]; ++kb)
                fprintf(stderr, "  [%lld %lld %lld]", (long long)(q[3 * kb] - q[0]), (long long)(q[3 * kb + 1] - q[0]), (long long)(q[3 * kb + 2] - q[0]));
            fprintf(stderr, "\n");
        }
    }
    ACB_CHECK_CUDA(cudaMemset(lm->trace, 0, 8192 * sizeof(unsigned long long)));
    return ACB_OK;
}

extern "C" int acb_lm_step_logits(acb_lm_t* lm, float* logits_out, void* stream) {
    ACB_REQUIRE(lm && lm->rows > 0, "acb_lm_step_logits: call acb_lm_begin first");
    if (lm->fused && lm->trace) lm->step.p.trace = lm->trace;
    ACB_TRY(enqueue_step(lm, (cudaStream_t)stream, logits_out, nullptr));
    if (lm->fused && lm->trace) { lm->step.p.trace = nullptr; ACB_TRY(report_step_trace(lm, (cudaStream_t)stream)); }
    if (lm->fused) return ACB_OK;
    if (lm->timing) ACB_TRY(report_timeline(lm, (cudaStream_t)stream));
    return ACB_OK;
}

extern "C" int acb_lm_debug_gemms(acb_lm_t* lm, void* stream, int* n_launches) {
    ACB_REQUIRE(lm && lm->rows > 0, "acb_lm_debug_gemms: call acb_lm_begin first");
    return enqueue_step(lm, (cudaStream_t)stream, nullptr, n_launches, true);
}

extern "C" int acb_lm_debug_step_plan(const acb_lm_t* lm, int* out) {
    ACB_REQUIRE(lm && out && lm->fused, "acb_lm_debug_step_plan: the fused step is not active");
    for (int i = 0; i < ACB_STEP_GEMMS; ++i) {
        const StepGemm& g = lm->step.p.g[i];
        out[4 * i] = g.N; out[4 * i + 1] = g.K; out[4 * i + 2] = g.ksplit; out[4 * i + 3] = g.kb_per;
    }
    out[4 * ACB_STEP_GEMMS] = lm->step.p.n_stage;
    out[4 * ACB_STEP_GEMMS + 1] = lm->step.p.R;
    out[4 * ACB_STEP_GEMMS + 2] = lm->step.n_phases;
    out[4 * ACB_STEP_GEMMS + 3] = (int)lm->step.smem;
    return ACB_OK;
}

extern "C" int acb_lm_rows_pad(int rows) { return rows <= 16 ? 16 : 8 * nt_for_rows(rows); }

extern "C" int acb_lm_launches_per_step(const acb_lm_t* lm) { return lm ? lm->launches : 0; }

extern "C" int acb_sample(const float* logits, const float* noise, int64_t* tokens, int batch, int rows, int n_q, int card,
                          const acb_lm_sampling* sampling, uint64_t step, void* stream) {
    ACB_REQUIRE(logits && tokens && sampling, "acb_sample: null argument");
    ACB_REQUIRE(batch >= 1 && (rows == batch || rows == 2 * batch || rows == 3 * batch) && n_q >= 1 && card >= 2 && card <= 4096, "acb_sample: bad shape");
    int NP = 1;
    while (NP < card) NP <<= 1;
    SampleParams sp{logits, sampling->noise_from_buffer ? noise : nullptr, nullptr, nullptr, nullptr, nullptr, 0, tokens, batch, rows, n_q, card, NP,
                    sampling->use_sampling, sampling->top_k, sampling->temp, sampling->top_p, sampling->cfg_coef,
                    sampling->seed, (uint32_t)step, sampling->cfg_coef_beta};
    size_t smem = ((size_t)card + 2 * (size_t)NP) * sizeof(float);
    if (smem > 48 * 1024)
        ACB_CHECK_CUDA(cudaFuncSetAttribute(lm_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lm_sample_kernel<<<dim3(n_q, batch), 1024, smem, (cudaStream_t)stream>>>(sp);
    ACB_LAUNCH_CHECK();
    return ACB_OK;
}

// ------------------------------------------------------------------------------------------------ dependency-latency probe
// A chain of `n_kernels` dependent EMPTY kernels (grid `ctas` x `threads`, `smem` bytes of dynamic shared memory each)
// captured in one graph -- with programmatic (PDL) edges when pdl != 0 -- and replayed `reps` times: the time per
// kernel is the floor any decode step of that many dependent kernels can reach on this GPU.  Measurement aid only.
__global__ void acb_probe_kernel(int* sink) {
    pdl_trigger();
    pdl_wait();
    if (sink && threadIdx.x == 0 && blockIdx.x == 0) sink[0] += 1;   // a dependent read-modify-write through global memory
}

extern "C" int acb_debug_chain_latency(int n_kernels, int ctas, int threads, int smem, int pdl, int reps, float* us_per_kernel,
                                       void* scratch) {
    ACB_REQUIRE(n_kernels >= 1 && n_kernels <= 4096 && ctas >= 1 && threads >= 32 && threads <= 1024 && reps >= 1 && us_per_kernel,
                "acb_debug_chain_latency: bad argument");
    ACB_REQUIRE(smem >= 0 && smem <= 200 * 1024, "acb_debug_chain_latency: smem out of range");
    if (smem > 48 * 1024)
        ACB_CHECK_CUDA(cudaFuncSetAttribute(acb_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    cudaStream_t s;
    ACB_CHECK_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int rc = ACB_OK;
    cudaError_t e = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal);
    for (int i = 0; i < n_kernels && e == cudaSuccess; ++i)
        e = launch_k(acb_probe_kernel, dim3(ctas), dim3(threads), (size_t)smem, s, pdl != 0, (int*)scratch);
    cudaError_t e2 = cudaStreamEndCapture(s, &graph);
    if (e == cudaSuccess) e = e2;
    if (e == cudaSuccess) e = cudaGraphInstantiate(&exec, graph, 0);
    if (e == cudaSuccess) e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    if (e == cudaSuccess) {
        for (int i = 0; i < 3; ++i) cudaGraphLaunch(exec, s);
        cudaEventRecord(e0, s);
        for (int i = 0; i < reps; ++i) cudaGraphLaunch(exec, s);
        cudaEventRecord(e1, s);
        e = cudaStreamSynchronize(s);
        float ms = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
        *us_per_kernel = ms * 1e3f / (float)reps / (float)n_kernels;
    }
    if (e != cudaSuccess) { acb_set_error("acb_debug_chain_latency: %s", cudaGetErrorString(e)); rc = ACB_ERR_CUDA; cudaGetLastError(); }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
    cudaStreamDestroy(s);
    return rc;
}
