// rsb_bert.cu -- BERT-base query encoder forward (reference: `Contriever.forward`, contriever/src/contriever.py:17-55,
// called from src/search.py:83-96 with the model in fp16) on variable-length (un-padded) token streams.
//
//   embed_ln_kernel      word + position + token-type gather, LayerNorm(eps)                    -> H  [T,768]  f16
//   gemm_tn_pair_kernel  Y = X . W^T (+bias [+GELU | +residual]) on 5th-gen tensor cores, CTA pairs (tcgen05
//                        cta_group::2): TMA (cp.async.bulk.tensor, 128B swizzle) -> shared-memory ring -> tcgen05.mma
//                        kind::f16 (fp32 accumulate in double-buffered TMEM) -> tcgen05.ld epilogue.  One elected
//                        thread of the leader CTA issues the MMAs; warp-specialised producer / issuer / epilogue roles
//                        synchronised with mbarriers.  gemm_tn_kernel: 128 x 128 tiles, one per CTA, for N % 256 != 0.
//   attention_mma32_kernel / attention_flash_kernel   softmax(QK^T / sqrt(64)) V per (sequence, head) on mma.sync:
//                        one warp per (sequence, head) up to 32 tokens, flash-style blocks of 128 queries beyond
//                        (collect_long_kernel lists those sequences once per forward)
//   layernorm_rows_kernel  LayerNorm over 768 (fp32 statistics), persistent warps with the next row prefetched
//   pool_kernel          masked mean over the valid tokens (all tokens of an un-padded sequence) or CLS row
#include "../../include/rsb.h"

#include "rsb_internal.h"
#include "rsb_tc.cuh"

#include <cuda_fp16.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

namespace {

using namespace rsbtc;

// ---------------------------------------------------------------------------------------------------------
// GEMM  C[M,N] = A[M,K] . B[N,K]^T  (A = activations, B = nn.Linear weight: both K-major), f16 in, f32 accumulate.
// CTA tile 128 x 128, K step 64 (= one 128-byte swizzle row), 3-stage TMA ring (2 CTAs / SM co-resident so one CTA's
// epilogue overlaps the other's main loop).  192 threads: warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer,
// warps 2-5 = epilogue (warp w reads TMEM lanes 32*(w%4)..+31).
// ---------------------------------------------------------------------------------------------------------
constexpr int G_BM = 128, G_BN = 128, G_BK = 64, G_STAGES = 3, G_THREADS = 192;
constexpr int G_STAGE_BYTES = (G_BM + G_BN) * G_BK * 2;                 // 32 KB
constexpr int G_SMEM = G_STAGES * G_STAGE_BYTES + 1024 /*align*/ + 256; // ring + barriers

enum { EPI_BIAS = 0, EPI_BIAS_GELU = 1, EPI_BIAS_RESIDUAL = 2 };

// HF BERT's "gelu": 0.5 x (1 + erf(x / sqrt 2)).  erf by Abramowitz-Stegun 7.1.26 with the hardware reciprocal /
// exp2: |error| <= 5e-7 absolute -- below fp16 resolution of the output everywhere except the ~1e-6-sized negative
// tail -- at about half the instructions of CUDA's erff.  The FFN1 epilogue is bound by its instruction issue rate
// (ncu: 64 % issue-active at 33 % tensor-active with erff, profiles/r02_encoder_epilogue.md).  -DRSB_EXACT_ERF: erff.
__device__ __forceinline__ float gelu_erf(float x) {
#ifndef RSB_EXACT_ERF
    const float z = fabsf(x) * 0.70710678118654752f;
    const float t = __fdividef(1.f, fmaf(0.3275911f, z, 1.f));
    float p = fmaf(1.061405429f, t, -1.453152027f);
    p = fmaf(p, t, 1.421413741f);
    p = fmaf(p, t, -0.284496736f);
    p = fmaf(p, t, 0.254829592f);
    const float e = 1.f - p * t * __expf(-z * z);
    return 0.5f * x * (1.f + copysignf(e, x));
#else
    return 0.5f * x * (1.f + erff(x * 0.70710678118654752f));
#endif
}

// sm_100's packed fp32 pair instructions (FFMA2 / FMUL2 / FADD2: one issue slot per two lanes of work), used by the
// GELU / bias epilogue of the pair GEMM below.
__device__ __forceinline__ unsigned long long f2pack(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2unpack(unsigned long long v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long f2fma(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ unsigned long long f2mul(unsigned long long a, unsigned long long b) {
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
template <int EPI>
__global__ __launch_bounds__(G_THREADS)
void gemm_tn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    __half* __restrict__ C, const __half* __restrict__ bias, const __half* __restrict__ residual,
                    int M, int N, int K) {
    extern __shared__ unsigned char smem_dyn[];
    // 1024-byte alignment required by the 128B swizzle atom
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + G_STAGES * G_STAGE_BYTES);
    uint64_t* empty = full + G_STAGES;
    uint64_t* tmem_full = empty + G_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.y * G_BM, n0 = blockIdx.x * G_BN;
    const int nk = K / G_BK;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
        for (int s = 0; s < G_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, G_BN);   // 128 fp32 accumulator columns
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            for (int kb = 0; kb < nk; ++kb) {
                const int s = kb % G_STAGES;
                if (kb >= G_STAGES) mbar_wait(&empty[s], ((kb / G_STAGES) - 1) & 1);
                unsigned char* a_dst = smem + s * G_STAGE_BYTES;
                unsigned char* b_dst = a_dst + G_BM * G_BK * 2;
                mbar_expect_tx(&full[s], G_STAGE_BYTES);
                tma_load_2d(a_dst, &tmA, &full[s], kb * G_BK, m0);
                tma_load_2d(b_dst, &tmB, &full[s], kb * G_BK, n0);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // InstrDescriptor: c_format F32 (1<<4) | a,b F16 (0) | K-major both | N>>3 at [17,23) | M>>4 at [24,29)
            const uint32_t idesc = (1u << 4) | ((uint32_t)(G_BN >> 3) << 17) | ((uint32_t)(G_BM >> 4) << 24);
            for (int kb = 0; kb < nk; ++kb) {
                const int s = kb % G_STAGES;
                mbar_wait(&full[s], (kb / G_STAGES) & 1);
                tc_fence_after();
                const uint32_t a_addr = smem_u32(smem + s * G_STAGE_BYTES);
                const uint32_t b_addr = a_addr + G_BM * G_BK * 2;
                const uint64_t adesc = make_sw128_kmajor_desc(a_addr);
                const uint64_t bdesc = make_sw128_kmajor_desc(b_addr);
#pragma unroll
                for (int k4 = 0; k4 < G_BK / 16; ++k4) {
                    // advance 16 K-elements = 32 bytes inside the swizzle row: +2 in the (addr >> 4) field
                    umma_f16(tmem_base, adesc + (uint64_t)(k4 * 2), bdesc + (uint64_t)(k4 * 2), idesc, (kb | k4) ? 1u : 0u);
                }
                umma_commit(&empty[s]);                 // frees the smem stage when these MMAs retire
                if (kb == nk - 1) umma_commit(tmem_full);  // accumulator complete
            }
        }
    } else {
        // ===== epilogue: TMEM -> registers -> (+bias, GELU | residual) -> f16 -> global
        const int q = warp & 3;                 // TMEM lane quarter this warp may access
        const int row = m0 + q * 32 + lane;
        mbar_wait(tmem_full, 0);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < G_BN; c += 32) {
            uint32_t r[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c, r);
            if (row < M) {
                const int col0 = n0 + c;
                __half* dst = C + (size_t)row * N + col0;
                const __half* res = EPI == EPI_BIAS_RESIDUAL ? residual + (size_t)row * N + col0 : nullptr;
#pragma unroll
                for (int v = 0; v < 4; ++v) {   // 4 x (8 halves = 16 bytes)
                    const uint4 bv = *reinterpret_cast<const uint4*>(bias + col0 + v * 8);
                    const __half2* b2 = reinterpret_cast<const __half2*>(&bv);
                    uint4 rv = make_uint4(0, 0, 0, 0);
                    if (EPI == EPI_BIAS_RESIDUAL) rv = *reinterpret_cast<const uint4*>(res + v * 8);
                    const __half2* r2 = reinterpret_cast<const __half2*>(&rv);
                    uint4 ov;
                    __half2* o2 = reinterpret_cast<__half2*>(&ov);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float x0 = __uint_as_float(r[v * 8 + e * 2]) + __low2float(b2[e]);
                        float x1 = __uint_as_float(r[v * 8 + e * 2 + 1]) + __high2float(b2[e]);
                        if (EPI == EPI_BIAS_GELU) {
                            x0 = gelu_erf(x0);
                            x1 = gelu_erf(x1);
                        }
                        if (EPI == EPI_BIAS_RESIDUAL) { x0 += __low2float(r2[e]); x1 += __high2float(r2[e]); }
                        o2[e] = __floats2half2_rn(x0, x1);
                    }
                    *reinterpret_cast<uint4*>(dst + v * 8) = ov;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, G_BN);
}

// ---------------------------------------------------------------------------------------------------------
// Epilogue of the persistent kernels.  After tcgen05.ld every lane holds 32 fp32 accumulators of ONE row; a lane
// writes them as two 256-bit stores (sm_100 STG.256: whole 32-byte sectors, measured 52.8 -> 46.4 ms per 10k queries
// against 128-bit stores, profiles/r02_ab_round1_leftovers.txt).  A shared-memory transpose that makes each store
// instruction cover 8 rows x 64 contiguous bytes was measured SLOWER (51.3 ms, profiles/r02_encoder_epilogue.md): the
// epilogue is bound by its instruction count and the latency of its loads, not by L2 write transactions.  So the
// residual of chunk i+1 is requested before chunk i is processed (its ~1 us L2 round trip used to sit in front of every
// chunk of the attention-output GEMM), and the TMEM load of a chunk is issued before those requests and waited on after.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldg256(uint32_t (&v)[8], const void* p) {
    asm volatile("ld.global.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "l"(p));
}
__device__ __forceinline__ void stg256(void* p, const uint32_t (&v)[8]) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]),
                 "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------------------
// Epilogue of the pair GEMM (the first form -- residual prefetched one chunk ahead, fp16 bias, GELU with copysign -- and a
// 16-warp variant were measured against it and removed: profiles/r02_encoder_epilogue.md):
//  * the whole residual row segment of a warp (its 64 or 128 columns) is requested BEFORE the warp waits for the
//    accumulator, so the L2 round trip overlaps the tile's MMA phase instead of the first chunks of the epilogue;
//  * tcgen05.ld of chunk i+1 is in flight while chunk i is processed (two register buffers);
//  * the accumulator stage is handed back to the MMA warp as soon as the last tcgen05.ld has landed, before the last
//    chunk is processed and stored;
//  * bias as fp32 in shared memory, added with packed pair adds; residual added in half precision after rounding the
//    dense output to half, which is also the order of HF BertSelfOutput / BertOutput (dense -> fp16, then + input);
//  * GELU restated as relu(x) + 0.5|x| (erf(|x|/sqrt 2) - 1): one packed multiply-add onto max(x, 0) instead of
//    1 - p, copysign and 0.5 x (1 + e); with z' = |x| sqrt(log2(e)/2) the exponent is just -z'^2 (negation folded into
//    the MUFU operand) and every scale factor is folded into the polynomial's coefficients: 16 instead of 18
//    instructions per pair, and no cancellation for x < 0 (numpy restatement: max 1 fp16 ulp from the fp64 erf form).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long f2add(unsigned long long a, unsigned long long b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ unsigned long long f2splat(float v) { return f2pack(v, v); }

__device__ __forceinline__ unsigned long long gelu_erf_pair(unsigned long long X) {
    float x0, x1;
    f2unpack(X, x0, x1);
#ifdef RSB_EXACT_ERF
    return f2pack(gelu_erf(x0), gelu_erf(x1));
#else
    const unsigned long long Z = f2mul(f2pack(fabsf(x0), fabsf(x1)), f2splat(0.8493218003f));   // |x| sqrt(log2(e) / 2)
    float d0, d1;
    f2unpack(f2fma(Z, f2splat(0.2727374809f), f2splat(1.f)), d0, d1);                          // 1 + 0.3275911 |x| / sqrt 2
    float t0, t1;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(d0));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(d1));
    const unsigned long long T = f2pack(t0, t1);
    // -(0.5 / 0.8493218) (a1 t + ... + a5 t^5), Abramowitz-Stegun 7.1.26
    unsigned long long P = f2fma(T, f2splat(-0.624854695f), f2splat(0.8554778804f));
    P = f2fma(P, T, f2splat(-0.8367933924f));
    P = f2fma(P, T, f2splat(0.1674846542f));
    P = f2fma(P, T, f2splat(-0.1500194578f));
    P = f2mul(f2mul(P, T), Z);                                                                 // 0.5 |x| (erf - 1) e^{+z^2}
    float a0, a1;
    f2unpack(f2mul(Z, Z), a0, a1);
    float e0, e1;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(-a0));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(-a1));
    return f2fma(P, f2pack(e0, e1), f2pack(fmaxf(x0, 0.f), fmaxf(x1, 0.f)));
#endif
}

// one row (this lane's) x 32 columns; bias_c: fp32 in shared memory (same address in every lane: broadcast)
template <int EPI>
__device__ __forceinline__ void epilogue_store_chunk(const uint32_t (&r)[32], const uint32_t (&rr)[2][8], __half* dst,
                                                        uint32_t bias_c /* shared-window address */) {
#pragma unroll
    for (int w = 0; w < 2; ++w) {
        uint32_t o[8];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            float4 b;                                     // explicit ld.shared: the generic pointer would compile to LD
            asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                : "r"(bias_c + (uint32_t)((w * 16 + v * 4) * 4)));
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int j = w * 16 + v * 4 + e * 2;
                unsigned long long X = f2add(f2pack(__uint_as_float(r[j]), __uint_as_float(r[j + 1])),
                                             e ? f2pack(b.z, b.w) : f2pack(b.x, b.y));
                if (EPI == EPI_BIAS_GELU) X = gelu_erf_pair(X);
                float x0, x1;
                f2unpack(X, x0, x1);
                __half2 h = __floats2half2_rn(x0, x1);
                if (EPI == EPI_BIAS_RESIDUAL) h = __hadd2(h, *reinterpret_cast<const __half2*>(&rr[w][v * 2 + e]));
                o[v * 2 + e] = *reinterpret_cast<const uint32_t*>(&h);
            }
        }
        stg256(dst + w * 16, o);
    }
}

// all NCH chunks of one tile for this warp.  `release()` hands the accumulator stage back (called by every lane).
template <int EPI, int NCH, class Release>
__device__ __forceinline__ void epilogue_tile(uint32_t tmem_row_base, int acc_col0, int c_lo, int row, int M, int N, int n0,
                                                 __half* __restrict__ C, const float* __restrict__ bias_f,
                                                 const __half* __restrict__ residual, uint64_t* full_bar, uint32_t parity,
                                                 Release release) {
    const bool live = row < M;
    const __half* res_row = residual + (size_t)(live ? row : 0) * N + n0 + c_lo;
    __half* dst_row = C + (size_t)(live ? row : 0) * N + n0 + c_lo;
    const uint32_t bias_sa = smem_u32(bias_f + n0 + c_lo);
    uint32_t rr[NCH][2][8];
    if (EPI == EPI_BIAS_RESIDUAL && live) {
#pragma unroll
        for (int i = 0; i < NCH; ++i) { ldg256(rr[i][0], res_row + i * 32); ldg256(rr[i][1], res_row + i * 32 + 16); }
    }
    mbar_wait(full_bar, parity);
    tc_fence_after();
    uint32_t r[2][32];
    tmem_ld32_issue(tmem_row_base + (uint32_t)(acc_col0 + c_lo), r[0]);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; ++j) asm volatile("" : "+r"(r[0][j]));
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
        if (i + 1 < NCH) tmem_ld32_issue(tmem_row_base + (uint32_t)(acc_col0 + c_lo + (i + 1) * 32), r[(i + 1) & 1]);
        else release();                                   // every tcgen05.ld of this warp has completed
        if (live) epilogue_store_chunk<EPI>(r[i & 1], rr[i], dst_row + i * 32, bias_sa + (uint32_t)(i * 32 * 4));
        if (i + 1 < NCH) {
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) asm volatile("" : "+r"(r[(i + 1) & 1][j]));
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Tile constants of the pair GEMM below.  (Round 2 also had a "v2": one CTA per 128 x 256 tile, persistent, double-buffered
// TMEM -- 62-64 % of the MMA rate at best because an SM then receives 48 KB of operands per k-block; removed in favour of
// the pair kernel, measurements in profiles/r02_encoder_epilogue.md.)
// ---------------------------------------------------------------------------------------------------------
constexpr int H_BM = 128, H_BN = 256, H_BK = 64;
constexpr int H_EPI_WARPS = 8;                       // 2 warps per TMEM lane quarter, 128 accumulator columns each
constexpr int H_THREADS = 64 + 32 * H_EPI_WARPS;     // warp 0 TMA, warp 1 MMA, warps 2.. epilogue
constexpr int H_BIAS_MAX = 4096;                     // bias vector staged in shared memory as fp32 (N <= 4096)

// ---------------------------------------------------------------------------------------------------------
// cluster helpers (pair GEMM below).  Round 2 also measured a "v3": v2 plus 2-CTA clusters whose CTAs each fetched half
// of the shared weight tile and multicast it (tcgen05 cta_group::1): +-1 % (profiles/r02_ab_round1_leftovers.txt,
// r02_encoder_epilogue.md) -- multicast does not reduce what each SM receives -- and was removed in favour of the pair kernel.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t num_clusters_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------------
// Pair GEMM: CTA PAIRS (tcgen05 cta_group::2).  Why: the single-CTA 128x256 kernel pulls 48 KB of operands into its SM per
// 512-cycle k-block = 96 B/clk, the SM's L2 port delivers ~64 B/clk, and the K = 768 / K = 3072 GEMMs sat at 62-64 % of
// the MMA rate whatever the epilogue did (profiles/r02_encoder_epilogue.md); multicasting the weight tile (v3) does not
// change what each SM has to RECEIVE, which is why it measured +-1 %.  A pair of CTAs computes one 256 x 256 tile with
// 2-SM MMAs: each CTA stages only its 128 activation rows and HALF of the weight tile (32 KB per k-block = 64 B/clk), the
// tensor cores of both SMs read the two halves of B from both shared memories, and each CTA ends up with its 128 x 256
// accumulator in its own TMEM.  The leader CTA (cluster rank 0) issues every MMA; both CTAs' TMA loads signal the
// leader's "full" barrier (2CTA form, peer bit of the barrier address cleared), the leader's commits are multicast to
// both CTAs' "empty" / "accumulator full" barriers, and both CTAs' epilogue warps release the accumulator on the
// leader's barrier (remote arrive).  6-stage ring of 32 KB.
// ---------------------------------------------------------------------------------------------------------
constexpr int P_STAGES = 6;
constexpr int P_A_BYTES = 128 * H_BK * 2, P_B_BYTES = 128 * H_BK * 2;     // 16 KB + 16 KB
constexpr int P_STAGE_BYTES = P_A_BYTES + P_B_BYTES;
constexpr int P_SMEM = P_STAGES * P_STAGE_BYTES + 1024 + 256 + H_BIAS_MAX * 4;    // fp32 bias (second epilogue form)

__device__ __forceinline__ void tma_load_2d_2cta(void* smem_dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* local_bar, uint32_t cta_rank) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(local_bar)), "r"(cta_rank));
    // default semantics (as CUTLASS' ClusterBarrier::arrive): the ".release.cluster" form compiles to MEMBAR.ALL.GPU +
    // ERRBAR in front of the arrive, i.e. every epilogue warp waited for its global stores of the tile to drain before it
    // could hand the accumulator back (ncu: "membar" = 18-24 % of the stall samples of the K = 768 GEMMs).  What the
    // barrier orders here are tcgen05.ld completions, which tcgen05.wait::ld + tcgen05.fence::before_thread_sync cover.
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

template <int EPI>
__global__ __cluster_dims__(2, 1, 1) __launch_bounds__(H_THREADS, 1)
void gemm_tn_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB128,
                         __half* __restrict__ C, const __half* __restrict__ bias, const __half* __restrict__ residual,
                         int M, int N, int K, int m_rev) {
    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + P_STAGES * P_STAGE_BYTES);
    uint64_t* empty = full + P_STAGES;
    uint64_t* tmem_full = empty + P_STAGES;      // [2]
    uint64_t* tmem_empty = tmem_full + 2;        // [2]  (the leader's collects both CTAs' epilogue warps)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();                 // 0 = leader: rows 0-127 of the pair's tile, columns 0-127 of B
    const int tiles_n = N / H_BN;
    const int pairs_m = ((M + H_BM - 1) / H_BM + 1) / 2;
    const int npairs = pairs_m * tiles_n;
    const int nk = K / H_BK;
    const int pair0 = (int)cluster_id_x(), pair_step = (int)num_clusters_x();

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB128)) : "memory");
        for (int s = 0; s < P_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 2 * H_EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == 1) {                                          // one warp of EACH CTA of the pair
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
    }
    float* bias_f = reinterpret_cast<float*>(smem + P_STAGES * P_STAGE_BYTES + 256);
    for (int i = threadIdx.x; i < N; i += H_THREADS) bias_f[i] = __half2float(bias[i]);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                       // both CTAs' barriers and TMEM exist before anything remote arrives
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int it = 0;
            for (int pair = pair0; pair < npairs; pair += pair_step) {
                const int m0 = ((m_rev ? pairs_m - 1 - pair / tiles_n : pair / tiles_n) * 2 + rank) * H_BM, n0 = (pair % tiles_n) * H_BN + rank * 128;
                for (int kb = 0; kb < nk; ++kb, ++it) {
                    const int s = it % P_STAGES;
                    mbar_wait(&empty[s], ((it / P_STAGES) & 1) ^ 1);   // the leader's MMAs have consumed this slot in BOTH CTAs
                    unsigned char* a_dst = smem + s * P_STAGE_BYTES;
                    const uint32_t leader_bar = smem_u32(&full[s]) & 0xFEFFFFFFu;   // same offset in the rank-0 CTA
                    if (rank == 0) mbar_expect_tx(&full[s], 2 * P_STAGE_BYTES);     // this CTA's 32 KB + the peer's 32 KB
                    tma_load_2d_2cta(a_dst, &tmA, leader_bar, kb * H_BK, m0);      // rows past M are zero-filled by TMA
                    tma_load_2d_2cta(a_dst + P_A_BYTES, &tmB128, leader_bar, kb * H_BK, n0);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && rank == 0) {
            // c_format F32 | a,b F16 | K-major | N = 256 | M = 256 (the pair's rows)
            const uint32_t idesc = (1u << 4) | ((uint32_t)(H_BN >> 3) << 17) | ((uint32_t)((2 * H_BM) >> 4) << 24);
            int it = 0, lt = 0;
            for (int pair = pair0; pair < npairs; pair += pair_step, ++lt) {
                const int acc = lt & 1;
                mbar_wait(&tmem_empty[acc], ((lt >> 1) & 1) ^ 1);      // both CTAs' epilogues have drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * H_BN);
                for (int kb = 0; kb < nk; ++kb, ++it) {
                    const int s = it % P_STAGES;
                    mbar_wait(&full[s], (it / P_STAGES) & 1);          // both CTAs' tiles of this k-block have landed
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(smem + s * P_STAGE_BYTES);
                    const uint64_t adesc = make_sw128_kmajor_desc(a_addr);
                    const uint64_t bdesc = make_sw128_kmajor_desc(a_addr + P_A_BYTES);
#pragma unroll
                    for (int k4 = 0; k4 < H_BK / 16; ++k4)
                        umma_f16_2cta(d_tmem, adesc + (uint64_t)(k4 * 2), bdesc + (uint64_t)(k4 * 2), idesc, (kb | k4) ? 1u : 0u);
                    umma_commit_2cta(&empty[s], (uint16_t)0x3);       // frees the slot in both CTAs
                }
                umma_commit_2cta(&tmem_full[acc], (uint16_t)0x3);     // both CTAs' epilogues may read their halves
            }
        }
    } else {
        const int q = warp & 3;
        constexpr int COLS = H_BN / (H_EPI_WARPS / 4);       // this warp's share of the columns: 128
        const int c_lo = ((warp - 2) >> 2) * COLS;
        int lt = 0;
        for (int pair = pair0; pair < npairs; pair += pair_step, ++lt) {
            const int acc = lt & 1;
            const int m0 = ((m_rev ? pairs_m - 1 - pair / tiles_n : pair / tiles_n) * 2 + rank) * H_BM, n0 = (pair % tiles_n) * H_BN;
            epilogue_tile<EPI, COLS / 32>(tmem_base + ((uint32_t)(q * 32) << 16), acc * H_BN, c_lo, m0 + q * 32 + lane, M, N, n0, C,
                                          bias_f, residual, &tmem_full[acc], (uint32_t)((lt >> 1) & 1), [&]() {
                                              tc_fence_before();
                                              __syncwarp();
                                              if (lane == 0) mbar_arrive_cluster(&tmem_empty[acc], 0u);   // the leader's barrier counts both CTAs' warps
                                          });
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                       // no CTA leaves (or frees TMEM) while its peer may still use it
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

// ---------------------------------------------------------------------------------------------------------
// small kernels
// ---------------------------------------------------------------------------------------------------------
constexpr int HID = 768;  // one warp per row: 24 values per lane = 3 x (8 halves)

__device__ __forceinline__ void warp_layernorm_store(float (&x)[24], const __half* gamma, const __half* beta, float eps,
                                                     __half* out, int lane) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) s += x[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    // __fmul_rn: the mean is rounded before it is subtracted.  A plain multiply was contracted into x - s * (1/768) as
    // one FFMA, which for a constant row (s = 768 x exactly) leaves -x * 2^-25 instead of 0.  Next to eps = 1e-12 that
    // residue is not small: the row came out as up to beta -+ gamma instead of beta.
    const float mean = __fmul_rn(s, 1.f / HID);
    float v = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) { const float dlt = x[i] - mean; v = fmaf(dlt, dlt, v); }
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const float rstd = rsqrtf(v * (1.f / HID) + eps);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int col = c * 256 + lane * 8;
        const uint4 gv = *reinterpret_cast<const uint4*>(gamma + col);
        const uint4 bv = *reinterpret_cast<const uint4*>(beta + col);
        const __half2* g2 = reinterpret_cast<const __half2*>(&gv);
        const __half2* b2 = reinterpret_cast<const __half2*>(&bv);
        uint4 ov;
        __half2* o2 = reinterpret_cast<__half2*>(&ov);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float y0 = (x[c * 8 + e * 2] - mean) * rstd * __low2float(g2[e]) + __low2float(b2[e]);
            const float y1 = (x[c * 8 + e * 2 + 1] - mean) * rstd * __high2float(g2[e]) + __high2float(b2[e]);
            o2[e] = __floats2half2_rn(y0, y1);
        }
        *reinterpret_cast<uint4*>(out + col) = ov;
    }
}

__device__ __forceinline__ void load_row24(const __half* row, int lane, float (&x)[24], bool accumulate) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const uint4 v = *reinterpret_cast<const uint4*>(row + c * 256 + lane * 8);
        const __half2* h2 = reinterpret_cast<const __half2*>(&v);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = __half22float2(h2[e]);
            if (accumulate) { x[c * 8 + e * 2] += f.x; x[c * 8 + e * 2 + 1] += f.y; }
            else { x[c * 8 + e * 2] = f.x; x[c * 8 + e * 2 + 1] = f.y; }
        }
    }
}

__global__ void embed_ln_kernel(const int* __restrict__ input_ids, const int* __restrict__ type_ids,
                                const int* __restrict__ cu_seqlens, int B, int T, const __half* __restrict__ word,
                                const __half* __restrict__ pos, const __half* __restrict__ type,
                                const __half* __restrict__ gamma, const __half* __restrict__ beta, float eps,
                                int vocab, int max_pos, __half* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (t >= T) return;
    int lo = 0, hi = B;   // sequence b with cu[b] <= t < cu[b+1]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (cu_seqlens[mid] <= t) lo = mid; else hi = mid;
    }
    int p = t - cu_seqlens[lo];
    p = p < max_pos ? p : max_pos - 1;
    int id = input_ids[t];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    const int tt = type_ids ? (type_ids[t] != 0) : 0;
    float x[24];
    load_row24(word + (size_t)id * HID, lane, x, false);
    load_row24(type + (size_t)tt * HID, lane, x, true);
    load_row24(pos + (size_t)p * HID, lane, x, true);
    warp_layernorm_store(x, gamma, beta, eps, out + (size_t)t * HID, lane);
}

__global__ void layernorm_kernel(const __half* __restrict__ in, int T, const __half* __restrict__ gamma,
                                 const __half* __restrict__ beta, float eps, __half* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (t >= T) return;
    float x[24];
    load_row24(in + (size_t)t * HID, lane, x, false);
    warp_layernorm_store(x, gamma, beta, eps, out + (size_t)t * HID, lane);
}

// Persistent form for the two LayerNorms of a layer: a warp walks rows gw, gw + nw, ... with the raw 1.5 KB of its NEXT
// row already requested while it reduces and stores the current one.  Inside a forward
// the one-row-per-warp kernel ran 28-31 us against 21.5 us in isolation (RSB_BERT_PROFILE): after a GEMM the SM clock
// sits at ~1.45 GHz under the power cap, and a warp that loads, reduces and stores one row and exits is bound by its own
// latency chain, not by HBM.  Same arithmetic, same order of operations per row (RSB_LN_V1=1: the first form, A/B).
__global__ __launch_bounds__(256, 3)
void layernorm_rows_kernel(const __half* __restrict__ in, int T, const __half* __restrict__ gamma,
                           const __half* __restrict__ beta, float eps, __half* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    if (gw >= T) return;
    uint4 cur[3], nxt[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        cur[c] = *reinterpret_cast<const uint4*>(in + (size_t)gw * HID + c * 256 + lane * 8);
        nxt[c] = cur[c];
    }
    for (int t = gw; t < T; t += nw) {
        if (t + nw < T) {
#pragma unroll
            for (int c = 0; c < 3; ++c) nxt[c] = *reinterpret_cast<const uint4*>(in + (size_t)(t + nw) * HID + c * 256 + lane * 8);
        }
        float x[24];
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const __half2* h2 = reinterpret_cast<const __half2*>(&cur[c]);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 f = __half22float2(h2[e]);
                x[c * 8 + e * 2] = f.x;
                x[c * 8 + e * 2 + 1] = f.y;
            }
        }
#pragma unroll
        for (int i = 0; i < 24; ++i) s += x[i];
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        const float mean = __fmul_rn(s, 1.f / HID);     // rounded before the subtraction, as in warp_layernorm_store
        float v = 0.f;
#pragma unroll
        for (int i = 0; i < 24; ++i) { const float dlt = x[i] - mean; v = fmaf(dlt, dlt, v); }
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        const float rstd = rsqrtf(v * (1.f / HID) + eps);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const uint4 gv = *reinterpret_cast<const uint4*>(gamma + c * 256 + lane * 8);   // L1-resident after the first row
            const uint4 bv = *reinterpret_cast<const uint4*>(beta + c * 256 + lane * 8);
            const __half2* g2 = reinterpret_cast<const __half2*>(&gv);
            const __half2* b2 = reinterpret_cast<const __half2*>(&bv);
            uint4 ov;
            __half2* o2 = reinterpret_cast<__half2*>(&ov);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float y0 = (x[c * 8 + e * 2] - mean) * rstd * __low2float(g2[e]) + __low2float(b2[e]);
                const float y1 = (x[c * 8 + e * 2 + 1] - mean) * rstd * __high2float(g2[e]) + __high2float(b2[e]);
                o2[e] = __floats2half2_rn(y0, y1);
            }
            *reinterpret_cast<uint4*>(out + (size_t)t * HID + c * 256 + lane * 8) = ov;
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) cur[c] = nxt[c];
    }
}

constexpr int ATT_HD = 64, ATT_PADH = 72, ATT_MAXS = 512;

// ---------------------------------------------------------------------------------------------------------
// attention for query-length sequences (S <= 32): ONE WARP per (sequence, head), QK^T and PV on the tensor cores
// with mma.sync.m16n8k16 (a 32x32x64 problem is far too small for a tcgen05 tile), softmax on the accumulator
// fragments in registers.  Q and K fragments are read straight from global memory as 32-bit words (row-major
// [token, 64] slices are exactly the A / "col" B fragment layouts); V is staged per warp in shared memory and
// read with ldmatrix.trans.  ~64 MMAs per (sequence, head) instead of ~10k scalar instructions.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_16816(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&h);
}

constexpr int ATT32_WARP_BYTES = 3 * 32 * ATT_PADH * 2;      // Q, K, V tiles of one (sequence, head)

__global__ __launch_bounds__(128)
void attention_mma32_kernel(const __half* __restrict__ qkv, const int* __restrict__ cu_seqlens, __half* __restrict__ ctx,
                            float scale, int heads, int B, int rev) {
    extern __shared__ __align__(16) unsigned char att32_smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    // blocks run last sequence first: the QKV tensor (188 MB at 41k tokens) is larger than the L2 and the GEMM wrote its
    // last rows most recently
    const int w = (rev ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x) * 4 + wib;
    if (w >= B * heads) return;                         // warp-uniform
    const int b = w / heads, h = w % heads;
    const int t0 = cu_seqlens[b];
    const int S = cu_seqlens[b + 1] - t0;
    if (S > 32 || S <= 0) return;                        // longer sequences belong to attention_flash_kernel
    const int g = lane >> 2, t = lane & 3;
    const __half* base = qkv + (size_t)t0 * (3 * HID) + h * ATT_HD;   // Q of token 0; K at +HID, V at +2*HID
    typedef __half (*Tile)[ATT_PADH];
    Tile Qs = reinterpret_cast<Tile>(att32_smem + wib * ATT32_WARP_BYTES);
    Tile Ks = Qs + 32, Vs = Qs + 64;

    // (A persistent variant that prefetched the next item's tiles with cp.async into a second buffer was measured and
    // dropped: 81 vs 74 us per layer -- the double buffer halves the resident warps and the kernel is bound by the
    // dependent-instruction latency of each warp, profiles/r02_ncu_summary_scan_attention.md.)
    // stage Q, K, V (rows >= S zero-filled): 8 lanes cover one 128-byte row, a warp instruction covers 4 whole rows --
    // every sector that is fetched is used (the 32-bit fragment loads straight from global memory of the first version
    // touched 32 sectors per instruction for 128 useful bytes; the kernel ran at half of the HBM rate)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int idx = lane + 32 * i, j = idx >> 3, c = idx & 7;
        uint4 qv = make_uint4(0, 0, 0, 0), kv = qv, vv = qv;
        if (j < S) {
            const __half* src = base + (size_t)j * (3 * HID) + c * 8;
            qv = *reinterpret_cast<const uint4*>(src);
            kv = *reinterpret_cast<const uint4*>(src + HID);
            vv = *reinterpret_cast<const uint4*>(src + 2 * HID);
        }
        *reinterpret_cast<uint4*>(&Qs[j][c * 8]) = qv;
        *reinterpret_cast<uint4*>(&Ks[j][c * 8]) = kv;
        *reinterpret_cast<uint4*>(&Vs[j][c * 8]) = vv;
    }
    __syncwarp();

    // S = Q K^T (fp32 accumulators): 2 m-tiles (query rows 0-15, 16-31) x 4 n-tiles (keys 8 each).  Fragments come from
    // ldmatrix.x4: one instruction per Q m-tile and per PAIR of key tiles (row stride 144 B: the 8 rows of a matrix fall
    // in 8 disjoint groups of 4 banks).
    const int ntm = (S + 7) >> 3;                        // key tiles of 8 that hold at least one valid key (NQ queries: 3 of 4)
    float sacc[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
            for (int e = 0; e < 4; ++e) sacc[mt][nt][e] = 0.f;
    // lane -> row/column of the 8x8 matrix whose row address it supplies
    const uint32_t q_lane = smem_u32(&Qs[(lane & 7) + ((lane >> 3) & 1) * 8][(lane >> 4) * 8]);   // A: (r, k), (r+8, k), (r, k+8), (r+8, k+8)
    const uint32_t k_lane = smem_u32(&Ks[(lane & 7) + ((lane >> 4) & 1) * 8][((lane >> 3) & 1) * 8]); // B: tile nt (k, k+8), tile nt+1 (k, k+8)
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        uint32_t qa[2][4], kb[4][2];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
            asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                         : "=r"(qa[mt][0]), "=r"(qa[mt][1]), "=r"(qa[mt][2]), "=r"(qa[mt][3])
                         : "r"(q_lane + (uint32_t)((mt * 16 * ATT_PADH + ks * 16) * 2)));
#pragma unroll
        for (int np = 0; np < 2; ++np) {
            if (np * 2 < ntm) {                          // warp-uniform: key tiles past the sequence end are skipped
                asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                             : "=r"(kb[np * 2][0]), "=r"(kb[np * 2][1]), "=r"(kb[np * 2 + 1][0]), "=r"(kb[np * 2 + 1][1])
                             : "r"(k_lane + (uint32_t)((np * 16 * ATT_PADH + ks * 16) * 2)));
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) mma_16816(sacc[mt][np * 2], qa[mt], kb[np * 2]);
                if (np * 2 + 1 < ntm) {
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) mma_16816(sacc[mt][np * 2 + 1], qa[mt], kb[np * 2 + 1]);
                }
            }
        }
    }

    // softmax over keys: thread holds rows (mt*16 + g) [elements 0,1] and (mt*16 + g + 8) [elements 2,3], key columns
    // nt*8 + 2t + {0,1}; a row is spread over the 4 lanes of a quad.  exp((s - max) scale) = 2^(s c - max c) with
    // c = scale log2(e): one FFMA + one MUFU per element.  Every row sees at least one valid key (S >= 1), so the row
    // maximum is finite and the sum positive.  The probabilities are normalised BEFORE they are rounded to half -- the
    // order of HF BERT (softmax -> fp16 probabilities -> P V) -- which also halves the scaling work (32 instead of 64
    // multiplies per lane).
    const float cexp = scale * 1.4426950408889634f;
    uint32_t pa[2][2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            if (nt < ntm) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int col = nt * 8 + 2 * t + (e & 1);
                    const float s = col < S ? sacc[mt][nt][e] : -INFINITY;
                    sacc[mt][nt][e] = s;
                    if (e < 2) mx0 = fmaxf(mx0, s); else mx1 = fmaxf(mx1, s);
                }
            }
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float m0c = -mx0 * cexp, m1c = -mx1 * cexp;
        float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            if (nt < ntm) {                              // skipped tiles keep their zeros = probability 0
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float p;
                    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p) : "f"(fmaf(sacc[mt][nt][e], cexp, e < 2 ? m0c : m1c)));   // 2^(-inf) = 0
                    sacc[mt][nt][e] = p;
                    if (e < 2) sum0 += p; else sum1 += p;
                }
            }
        }
        sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
        sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
        const float inv0 = __fdividef(1.f, sum0), inv1 = __fdividef(1.f, sum1);
        // probabilities as the A operand of P.V: k-step kk covers keys 16kk..16kk+15 = n-tiles 2kk, 2kk+1
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
            pa[mt][kk][0] = pack_half2(sacc[mt][2 * kk][0] * inv0, sacc[mt][2 * kk][1] * inv0);
            pa[mt][kk][1] = pack_half2(sacc[mt][2 * kk][2] * inv1, sacc[mt][2 * kk][3] * inv1);
            pa[mt][kk][2] = pack_half2(sacc[mt][2 * kk + 1][0] * inv0, sacc[mt][2 * kk + 1][1] * inv0);
            pa[mt][kk][3] = pack_half2(sacc[mt][2 * kk + 1][2] * inv1, sacc[mt][2 * kk + 1][3] * inv1);
        }
    }
    // O = P V : 2 m-tiles x 8 n-tiles (head dims 8 each); V^T fragments of both 16-key steps through ONE ldmatrix.x4.trans
    // (rows = keys 0..31 of this lane, zero-filled past the sequence end)
    const uint32_t v_lane = smem_u32(&Vs[lane][0]);
    const bool two_steps = S > 16;                       // warp-uniform: a 16-key step without valid keys adds nothing
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        float o[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
        uint32_t vb[2][2];
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(vb[0][0]), "=r"(vb[0][1]), "=r"(vb[1][0]), "=r"(vb[1][1])
                     : "r"(v_lane + (uint32_t)(nt * 8 * 2)));
        mma_16816(o[0], pa[0][0], vb[0]);
        mma_16816(o[1], pa[1][0], vb[0]);
        if (two_steps) {
            mma_16816(o[0], pa[0][1], vb[1]);
            mma_16816(o[1], pa[1][1], vb[1]);
        }
        // the output tile goes back through this warp's Q tile (all Q fragments were consumed before the first P.V
        // MMA; program order inside the warp + the __syncwarp below make the reuse safe) so that it can be written
        // with whole 128-byte rows instead of 4-byte pieces
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const int r0 = mt * 16 + g, col = nt * 8 + 2 * t;
            *reinterpret_cast<__half2*>(&Qs[r0][col]) = __floats2half2_rn(o[mt][0], o[mt][1]);
            *reinterpret_cast<__half2*>(&Qs[r0 + 8][col]) = __floats2half2_rn(o[mt][2], o[mt][3]);
        }
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int idx = lane + 32 * i, j = idx >> 3, c = idx & 7;
        if (j < S)
            *reinterpret_cast<uint4*>(ctx + (size_t)(t0 + j) * HID + h * ATT_HD + c * 8) = *reinterpret_cast<const uint4*>(&Qs[j][c * 8]);
    }
}


// sequences longer than `threshold` tokens -> list (order irrelevant) + count; once per forward
__global__ void collect_long_kernel(const int* __restrict__ cu_seqlens, int B, int threshold, int* __restrict__ list,
                                    int* __restrict__ count) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x)
        if (cu_seqlens[b + 1] - cu_seqlens[b] > threshold) list[atomicAdd(count, 1)] = b;
}

// ---------------------------------------------------------------------------------------------------------
// attention for longer sequences (33..512 tokens: the passage side, reference src/embed.py:24-94 at batch 512):
// flash-style on the tensor cores.  One block = 4 warps = 128 consecutive query rows of one (sequence, head); a warp
// owns 32 query rows (Q fragments stay in registers) and walks the keys in blocks of 32 that the whole block stages
// in shared memory once: S = Q K^T with mma.sync.m16n8k16, online softmax on the accumulator fragments (running row
// maximum / sum, output rescaled when the maximum moves), O += P V with V^T fragments through ldmatrix.trans.
// Same arithmetic as attention_mma32_kernel for a single key block.
// ---------------------------------------------------------------------------------------------------------
__global__ __launch_bounds__(128)
void attention_flash_kernel(const __half* __restrict__ qkv, const int* __restrict__ cu_seqlens, __half* __restrict__ ctx,
                            float scale, const int* __restrict__ long_list, const int* __restrict__ long_count, int heads,
                            int nqb) {
    __shared__ __align__(16) __half Ks[32][ATT_PADH];
    __shared__ __align__(16) __half Vs[32][ATT_PADH];
    // work items (long sequence, head, block of 128 queries) in a grid-stride loop over the list that collect_long_kernel
    // wrote once for this forward.  A batch of queries holds one or two sequences beyond 32 tokens: walking all
    // B x heads x nqb candidates every layer kept the side stream busy for 36 us and slowed the short-sequence kernel it
    // overlaps with (attention 74 -> 120 us per layer inside a forward, RSB_BERT_PROFILE).
    const int n_items = *long_count * heads * nqb;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int qblk = item % nqb, h = (item / nqb) % heads, b = long_list[item / (nqb * heads)];
    const int t0 = cu_seqlens[b];
    const int S = cu_seqlens[b + 1] - t0;
    const int q0 = qblk * 128;
    if (q0 >= S) continue;                               // block-uniform
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int qw = q0 + wib * 32;                        // first query row of this warp
    const bool active = qw < S;                          // warp-uniform; idle warps still stage K / V and hit the barriers
    const __half* base = qkv + (size_t)t0 * (3 * HID) + h * ATT_HD;

    uint32_t qa[4][2][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const int r0 = qw + mt * 16 + g, c = ks * 16 + 2 * t;
            const __half* p0 = base + (size_t)r0 * (3 * HID) + c;
            const __half* p1 = base + (size_t)(r0 + 8) * (3 * HID) + c;
            qa[ks][mt][0] = r0 < S ? *reinterpret_cast<const uint32_t*>(p0) : 0u;
            qa[ks][mt][1] = r0 + 8 < S ? *reinterpret_cast<const uint32_t*>(p1) : 0u;
            qa[ks][mt][2] = r0 < S ? *reinterpret_cast<const uint32_t*>(p0 + 8) : 0u;
            qa[ks][mt][3] = r0 + 8 < S ? *reinterpret_cast<const uint32_t*>(p1 + 8) : 0u;
        }
    float o[2][8][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int e = 0; e < 4; ++e) o[mt][nt][e] = 0.f;
    float m_run[2][2] = {{-INFINITY, -INFINITY}, {-INFINITY, -INFINITY}};
    float l_run[2][2] = {{0.f, 0.f}, {0.f, 0.f}};       // per-lane partial row sums (quad-reduced at the end)

    const int nkb = (S + 31) >> 5;
    for (int kb = 0; kb < nkb; ++kb) {
        __syncthreads();                                 // the previous key block has been consumed by every warp
#pragma unroll
        for (int i = 0; i < 2; ++i) {                    // 32 rows x 8 uint4 for K and for V: 2 + 2 per thread
            const int idx = threadIdx.x + 128 * i, j = idx >> 3, c = idx & 7;
            const int key = kb * 32 + j;
            uint4 kv = make_uint4(0, 0, 0, 0), vv = make_uint4(0, 0, 0, 0);
            if (key < S) {
                const __half* src = base + (size_t)key * (3 * HID) + c * 8;
                kv = *reinterpret_cast<const uint4*>(src + HID);
                vv = *reinterpret_cast<const uint4*>(src + 2 * HID);
            }
            *reinterpret_cast<uint4*>(&Ks[j][c * 8]) = kv;
            *reinterpret_cast<uint4*>(&Vs[j][c * 8]) = vv;
        }
        __syncthreads();
        if (!active) continue;
        float sacc[2][4][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) sacc[mt][nt][e] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            uint32_t kbf[4][2];
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                const int j = nt * 8 + g, c = ks * 16 + 2 * t;
                kbf[nt][0] = *reinterpret_cast<const uint32_t*>(&Ks[j][c]);
                kbf[nt][1] = *reinterpret_cast<const uint32_t*>(&Ks[j][c + 8]);
            }
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) mma_16816(sacc[mt][nt], qa[ks][mt], kbf[nt]);
        }
        uint32_t pa[2][2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int col = kb * 32 + nt * 8 + 2 * t + (e & 1);
                    const float sv = col < S ? sacc[mt][nt][e] * scale : -INFINITY;
                    sacc[mt][nt][e] = sv;
                    if (e < 2) mx0 = fmaxf(mx0, sv); else mx1 = fmaxf(mx1, sv);
                }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
            // every key block holds at least one valid key, so the new maxima are finite
            const float mn0 = fmaxf(m_run[mt][0], mx0), mn1 = fmaxf(m_run[mt][1], mx1);
            const float cr0 = __expf(m_run[mt][0] - mn0), cr1 = __expf(m_run[mt][1] - mn1);   // exp(-inf) = 0 on the first block
            m_run[mt][0] = mn0; m_run[mt][1] = mn1;
            float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
            for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float sv = sacc[mt][nt][e];
                    const float pv = (sv == -INFINITY) ? 0.f : __expf(sv - (e < 2 ? mn0 : mn1));
                    sacc[mt][nt][e] = pv;
                    if (e < 2) sum0 += pv; else sum1 += pv;
                }
            l_run[mt][0] = l_run[mt][0] * cr0 + sum0;
            l_run[mt][1] = l_run[mt][1] * cr1 + sum1;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                o[mt][nt][0] *= cr0; o[mt][nt][1] *= cr0;
                o[mt][nt][2] *= cr1; o[mt][nt][3] *= cr1;
            }
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                pa[mt][kk][0] = pack_half2(sacc[mt][2 * kk][0], sacc[mt][2 * kk][1]);
                pa[mt][kk][1] = pack_half2(sacc[mt][2 * kk][2], sacc[mt][2 * kk][3]);
                pa[mt][kk][2] = pack_half2(sacc[mt][2 * kk + 1][0], sacc[mt][2 * kk + 1][1]);
                pa[mt][kk][3] = pack_half2(sacc[mt][2 * kk + 1][2], sacc[mt][2 * kk + 1][3]);
            }
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                uint32_t vb[2];
                const uint32_t addr = smem_u32(&Vs[kk * 16 + (lane & 15)][nt * 8]);
                asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(vb[0]), "=r"(vb[1]) : "r"(addr));
                mma_16816(o[0][nt], pa[0][kk], vb);
                mma_16816(o[1][nt], pa[1][kk], vb);
            }
    }
    if (active) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        float l0 = l_run[mt][0], l1 = l_run[mt][1];
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        const float i0 = l0 > 0.f ? 1.f / l0 : 0.f, i1 = l1 > 0.f ? 1.f / l1 : 0.f;
        const int r0 = qw + mt * 16 + g;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int col = h * ATT_HD + nt * 8 + 2 * t;
            if (r0 < S)
                *reinterpret_cast<__half2*>(ctx + (size_t)(t0 + r0) * HID + col) = __floats2half2_rn(o[mt][nt][0] * i0, o[mt][nt][1] * i0);
            if (r0 + 8 < S)
                *reinterpret_cast<__half2*>(ctx + (size_t)(t0 + r0 + 8) * HID + col) = __floats2half2_rn(o[mt][nt][2] * i1, o[mt][nt][3] * i1);
        }
    }
    }
    __syncthreads();                                     // K / V tiles are re-staged by the next item
    }
}

// pooling: one block per sequence; mode 0 = mean over tokens (contriever.py:45-49), 1 = CLS row (:50-51)
__global__ void pool_kernel(const __half* __restrict__ H, const int* __restrict__ cu_seqlens, int mode,
                            __half* __restrict__ out) {
    const int b = blockIdx.x;
    const int t0 = cu_seqlens[b], t1 = cu_seqlens[b + 1];
    for (int c = threadIdx.x; c < HID; c += blockDim.x) {
        float s = 0.f;
        if (mode == 1 || t1 <= t0) {
            s = t1 > t0 ? __half2float(H[(size_t)t0 * HID + c]) : 0.f;
        } else {
            for (int t = t0; t < t1; ++t) s += __half2float(H[(size_t)t * HID + c]);
            s /= (float)(t1 - t0);
        }
        out[(size_t)b * HID + c] = __float2half_rn(s);
    }
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
thread_local std::string g_berr;
int bfail(int code, const char* fmt, const char* a = "", long b = 0) {
    char buf[512];
    snprintf(buf, sizeof buf, fmt, a, b);
    g_berr = buf;
    return code;
}

bool make_map(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
    return rsbtc::make_map_2d(m, base, rows, cols, box_rows, 2);
}

struct Linear {
    __half* w = nullptr;   // [N, K]
    __half* b = nullptr;   // [N]
    int N = 0, K = 0;
    CUtensorMap map;       // box 128 rows (v1 tiles)
    bool map_ok = false, pair_ok = false;   // pair_ok: N a multiple of 256 and the fp32 bias fits its shared-memory slot
};

struct Layer {
    Linear qkv, attn_out, ffn1, ffn2;
    __half *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
};

}  // namespace

struct rsb_bert {
    int hidden = 768, layers = 12, heads = 12, inter = 3072, vocab = 30522, max_pos = 512, type_vocab = 2;
    float eps = 1e-12f;
    __half *word = nullptr, *pos = nullptr, *type = nullptr, *emb_g = nullptr, *emb_b = nullptr;
    std::vector<Layer> L;
    long launches = 0;
    // the two attention kernels of a layer work on disjoint sequences (<= 32 tokens / longer): the long-sequence one runs
    // on a side stream so that it overlaps the other instead of adding its latency to every layer
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int* long_list = nullptr;                            // sequences > 32 tokens of the current forward; [long_cap] = their count
    int long_cap = 0;
};

namespace {

int alloc_linear(Linear& l, int N, int K) {
    l.N = N; l.K = K;
    if (cudaMalloc(&l.w, (size_t)N * K * 2) != cudaSuccess) return RSB_ERR_OOM;
    if (cudaMalloc(&l.b, (size_t)N * 2) != cudaSuccess) return RSB_ERR_OOM;
    cudaMemset(l.w, 0, (size_t)N * K * 2);
    cudaMemset(l.b, 0, (size_t)N * 2);
    l.map_ok = make_map(&l.map, l.w, N, K, G_BN);
    l.pair_ok = (N % H_BN == 0) && N <= H_BIAS_MAX;
    return l.map_ok ? RSB_OK : RSB_ERR_CUDA;
}
void free_linear(Linear& l) { cudaFree(l.w); cudaFree(l.b); }

// m_rev: visit the row tiles last-to-first.  The FFN intermediate (251 MB at 41k tokens) is twice the L2: FFN2 starts with the
// rows FFN1 wrote last, which are still cached (RSB_NO_SNAKE=1 disables, A/B).
template <int EPI>
int launch_gemm(const __half* A, int M, const Linear& lin, __half* C, const __half* residual, cudaStream_t st, bool m_rev = false) {
    CUtensorMap tmA;
    if (!make_map(&tmA, A, (uint64_t)M, (uint64_t)lin.K, G_BM)) return RSB_ERR_CUDA;
    static rsb::PerDeviceFlag configured;                    // attributes are per (function, device)
    if (configured.first()) {
        cudaFuncSetAttribute(gemm_tn_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, G_SMEM);
        cudaFuncSetAttribute(gemm_tn_pair_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM);
    }
    const int sms = rsb::device_num_sms();
    static const bool v1 = getenv("RSB_GEMM_V1") != nullptr;       // A/B: 128 x 128 tiles, one tile per CTA
    if (!v1 && lin.pair_ok && lin.map_ok) {                      // CTA pairs, 2-SM MMAs (N a multiple of 256)
        const int npairs = (lin.N / H_BN) * (((M + H_BM - 1) / H_BM + 1) / 2);
        const int clusters = std::max(1, std::min(npairs, sms / 2));
        static const bool no_snake = getenv("RSB_NO_SNAKE") != nullptr;
        gemm_tn_pair_kernel<EPI><<<2 * clusters, H_THREADS, P_SMEM, st>>>(tmA, lin.map, C, lin.b, residual, M, lin.N, lin.K,
                                                                          (m_rev && !no_snake) ? 1 : 0);
        return RSB_OK;
    }
    dim3 grid(lin.N / G_BN, (M + G_BM - 1) / G_BM);                // N not a multiple of 256 (or forced): 128 x 128 tiles
    gemm_tn_kernel<EPI><<<grid, G_THREADS, G_SMEM, st>>>(tmA, lin.map, C, lin.b, residual, M, lin.N, lin.K);
    return RSB_OK;
}

// LayerNorm over 768 of T rows (one launch), shared by the forward and rsb_bert_layernorm
void launch_layernorm(const rsb_bert* h, const __half* x, int T, const __half* g, const __half* b, __half* out, cudaStream_t st) {
    static const bool ln_v1 = getenv("RSB_LN_V1") != nullptr;
    const int rows_per_block = 8;   // 256 threads = 8 warps = 8 rows
    const int ln_grid = (T + rows_per_block - 1) / rows_per_block;
    const int ln_rows_grid = std::min(ln_grid, 3 * rsb::device_num_sms());   // 24 warps per SM, ~12 rows per warp at 41k tokens
    if (ln_v1) layernorm_kernel<<<ln_grid, 256, 0, st>>>(x, T, g, b, h->eps, out);
    else layernorm_rows_kernel<<<ln_rows_grid, 256, 0, st>>>(x, T, g, b, h->eps, out);
}

// The list of sequences longer than 32 tokens that the flash kernel takes, written once per forward (one launch when
// max_seqlen > 32, none otherwise; the count of launches is returned through *launches).
int prepare_attention(rsb_bert* h, const int* cu_seqlens, int B, int max_seqlen, cudaStream_t st, long* launches) {
    static rsb::PerDeviceFlag att_configured;
    if (att_configured.first())
        cudaFuncSetAttribute(attention_mma32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * ATT32_WARP_BYTES);
    if (!h->side) {
        cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking);
        cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
    }
    if (max_seqlen <= 32) return RSB_OK;
    if (h->long_cap < B) {
        cudaFree(h->long_list);
        h->long_list = nullptr;
        h->long_cap = 0;
        if (cudaMalloc(&h->long_list, ((size_t)B + 1) * sizeof(int)) != cudaSuccess) return RSB_ERR_OOM;
        h->long_cap = B;
    }
    cudaMemsetAsync(h->long_list + h->long_cap, 0, sizeof(int), st);          // the count lives behind the list
    collect_long_kernel<<<(B + 255) / 256, 256, 0, st>>>(cu_seqlens, B, 32, h->long_list, h->long_list + h->long_cap);
    ++*launches;
    return RSB_OK;
}

// softmax(Q K^T / 8) V of every (sequence, head) of the un-padded [T, 3 x 768] QKV into ctx [T, 768] (after
// prepare_attention for the same cu_seqlens / max_seqlen).  Sequences of <= 32 tokens (queries): warp-per-(sequence,
// head) tensor-core kernel; longer ones (passages, the odd long query): flash-style kernel on a side stream -- the two
// work on disjoint sequences of the same buffers.
void launch_attention(rsb_bert* h, const __half* qkv, const int* cu_seqlens, int B, int max_seqlen, __half* ctx,
                      cudaStream_t st, long* launches) {
    const bool have_long = max_seqlen > 32;
    if (have_long) {
        cudaEventRecord(h->ev_fork, st);
        cudaStreamWaitEvent(h->side, h->ev_fork, 0);
        const int nqb = (max_seqlen + 127) / 128;
        const long items = (long)B * h->heads * nqb;
        const int fgrid = (int)std::min<long>(items, 2L * rsb::device_num_sms());   // 194 registers: two resident blocks per SM
        attention_flash_kernel<<<fgrid, 128, 0, h->side>>>(qkv, cu_seqlens, ctx, 0.125f, h->long_list, h->long_list + h->long_cap,
                                                           h->heads, nqb);
        cudaEventRecord(h->ev_join, h->side);
        ++*launches;
    }
    const int nwarps = B * h->heads;
    static const bool no_snake = getenv("RSB_NO_SNAKE") != nullptr;
    attention_mma32_kernel<<<(nwarps + 3) / 4, 128, 4 * ATT32_WARP_BYTES, st>>>(qkv, cu_seqlens, ctx, 0.125f, h->heads, B,
                                                                               no_snake ? 0 : 1);
    ++*launches;
    if (have_long) cudaStreamWaitEvent(st, h->ev_join, 0);   // join before the attention-output GEMM
}

}  // namespace

extern "C" const char* rsb_bert_last_error(void) { return g_berr.c_str(); }

extern "C" int rsb_bert_create(int hidden, int layers, int heads, int inter, int vocab, int max_pos, int type_vocab,
                               float ln_eps, rsb_bert_t** out) {
    if (!out) return bfail(RSB_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (hidden != 768 || heads != 12 || inter % G_BN || inter % G_BK || layers <= 0 || vocab <= 0 || max_pos <= 0 || type_vocab <= 0)
        return bfail(RSB_ERR_UNSUPPORTED, "only BERT-base geometry (hidden 768, 12 heads, FFN multiple of 128) is implemented");
    if (!get_encode()) return bfail(RSB_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    rsb_bert* h = new rsb_bert();
    h->hidden = hidden; h->layers = layers; h->heads = heads; h->inter = inter; h->vocab = vocab;
    h->max_pos = max_pos; h->type_vocab = type_vocab; h->eps = ln_eps;
    bool ok = true;
    ok &= cudaMalloc(&h->word, (size_t)vocab * hidden * 2) == cudaSuccess;
    ok &= cudaMalloc(&h->pos, (size_t)max_pos * hidden * 2) == cudaSuccess;
    ok &= cudaMalloc(&h->type, (size_t)std::max(type_vocab, 2) * hidden * 2) == cudaSuccess;
    ok &= cudaMalloc(&h->emb_g, hidden * 2) == cudaSuccess;
    ok &= cudaMalloc(&h->emb_b, hidden * 2) == cudaSuccess;
    if (ok) cudaMemset(h->type, 0, (size_t)std::max(type_vocab, 2) * hidden * 2);
    h->L.resize(layers);
    for (auto& l : h->L) {
        ok &= alloc_linear(l.qkv, 3 * hidden, hidden) == RSB_OK;
        ok &= alloc_linear(l.attn_out, hidden, hidden) == RSB_OK;
        ok &= alloc_linear(l.ffn1, inter, hidden) == RSB_OK;
        ok &= alloc_linear(l.ffn2, hidden, inter) == RSB_OK;
        ok &= cudaMalloc(&l.ln1_g, hidden * 2) == cudaSuccess;
        ok &= cudaMalloc(&l.ln1_b, hidden * 2) == cudaSuccess;
        ok &= cudaMalloc(&l.ln2_g, hidden * 2) == cudaSuccess;
        ok &= cudaMalloc(&l.ln2_b, hidden * 2) == cudaSuccess;
    }
    if (!ok) { rsb_bert_free(h); return bfail(RSB_ERR_OOM, "allocating encoder weights failed"); }
    *out = h;
    return RSB_OK;
}

extern "C" int rsb_bert_free(rsb_bert_t* h) {
    if (!h) return RSB_OK;
    cudaFree(h->word); cudaFree(h->pos); cudaFree(h->type); cudaFree(h->emb_g); cudaFree(h->emb_b);
    if (h->side) cudaStreamDestroy(h->side);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    cudaFree(h->long_list);
    for (auto& l : h->L) {
        free_linear(l.qkv); free_linear(l.attn_out); free_linear(l.ffn1); free_linear(l.ffn2);
        cudaFree(l.ln1_g); cudaFree(l.ln1_b); cudaFree(l.ln2_g); cudaFree(l.ln2_b);
    }
    delete h;
    return RSB_OK;
}

// name = HF BertModel state_dict key (SURVEY.md App. B), data = fp16 device pointer, n = element count.
extern "C" int rsb_bert_load(rsb_bert_t* h, const char* name, const void* dev_ptr, int64_t n, rsb_stream_t stream) {
    if (!h || !name || !dev_ptr) return bfail(RSB_ERR_INVALID, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int H = h->hidden;
    auto put = [&](void* dst, int64_t expect) -> int {
        if (n != expect) return bfail(RSB_ERR_INVALID, "weight %s has the wrong size (%ld elements)", name, (long)n);
        return cudaMemcpyAsync(dst, dev_ptr, (size_t)n * 2, cudaMemcpyDeviceToDevice, st) == cudaSuccess
                   ? RSB_OK : bfail(RSB_ERR_CUDA, "copy of %s failed", name);
    };
    std::string s(name);
    if (s == "embeddings.word_embeddings.weight") return put(h->word, (int64_t)h->vocab * H);
    if (s == "embeddings.position_embeddings.weight") return put(h->pos, (int64_t)h->max_pos * H);
    if (s == "embeddings.token_type_embeddings.weight") return put(h->type, (int64_t)h->type_vocab * H);
    if (s == "embeddings.LayerNorm.weight") return put(h->emb_g, H);
    if (s == "embeddings.LayerNorm.bias") return put(h->emb_b, H);
    int li = -1;
    char rest[128] = {0};
    if (sscanf(name, "encoder.layer.%d.%127s", &li, rest) == 2 && li >= 0 && li < h->layers) {
        Layer& l = h->L[li];
        std::string r(rest);
        const int64_t HH = (int64_t)H * H;
        if (r == "attention.self.query.weight") return put(l.qkv.w, HH);
        if (r == "attention.self.key.weight") return put(l.qkv.w + HH, HH);
        if (r == "attention.self.value.weight") return put(l.qkv.w + 2 * HH, HH);
        if (r == "attention.self.query.bias") return put(l.qkv.b, H);
        if (r == "attention.self.key.bias") return put(l.qkv.b + H, H);
        if (r == "attention.self.value.bias") return put(l.qkv.b + 2 * H, H);
        if (r == "attention.output.dense.weight") return put(l.attn_out.w, HH);
        if (r == "attention.output.dense.bias") return put(l.attn_out.b, H);
        if (r == "attention.output.LayerNorm.weight") return put(l.ln1_g, H);
        if (r == "attention.output.LayerNorm.bias") return put(l.ln1_b, H);
        if (r == "intermediate.dense.weight") return put(l.ffn1.w, (int64_t)h->inter * H);
        if (r == "intermediate.dense.bias") return put(l.ffn1.b, h->inter);
        if (r == "output.dense.weight") return put(l.ffn2.w, (int64_t)h->inter * H);
        if (r == "output.dense.bias") return put(l.ffn2.b, H);
        if (r == "output.LayerNorm.weight") return put(l.ln2_g, H);
        if (r == "output.LayerNorm.bias") return put(l.ln2_b, H);
    }
    return bfail(RSB_ERR_INVALID, "unknown weight name %s", name);
}

static size_t bert_ws_layout(const rsb_bert* h, int T, size_t off[6]) {
    auto al = [](size_t x) { return (x + 1023) / 1024 * 1024; };   // TMA global addresses: 16 B is enough; keep 1 KB
    const size_t Tp = (size_t)((T + 127) / 128 * 128);
    size_t o = 0;
    off[0] = o; o += al(Tp * h->hidden * 2);        // H
    off[1] = o; o += al(Tp * 3 * h->hidden * 2);    // QKV
    off[2] = o; o += al(Tp * h->hidden * 2);        // CTX
    off[3] = o; o += al(Tp * h->hidden * 2);        // TMP (pre-LN sums)
    off[4] = o; o += al(Tp * h->inter * 2);         // FFN intermediate
    off[5] = o;
    return o;
}
extern "C" size_t rsb_bert_workspace_bytes(rsb_bert_t* h, int total_tokens) {
    if (!h) return 0;
    size_t off[6];
    return bert_ws_layout(h, std::max(total_tokens, 1), off);
}

// input_ids / token_type_ids [T] int32 (token_type_ids may be NULL), cu_seqlens [B+1] int32 (all device), out [B, 768] f16
extern "C" int rsb_bert_forward(rsb_bert_t* h, const int32_t* input_ids, const int32_t* token_type_ids,
                                const int32_t* cu_seqlens, int B, int T, int max_seqlen, int pooling, void* out_f16,
                                void* ws, size_t ws_bytes, rsb_stream_t stream) {
    if (!h || !input_ids || !cu_seqlens || !out_f16) return bfail(RSB_ERR_INVALID, "null argument");
    if (B <= 0 || T <= 0) return bfail(RSB_ERR_INVALID, "empty batch");
    if (max_seqlen > ATT_MAXS || max_seqlen > h->max_pos)
        return bfail(RSB_ERR_UNSUPPORTED, "sequence longer than %s%ld tokens", "", (long)std::min(ATT_MAXS, h->max_pos));
    size_t off[6];
    const size_t need = bert_ws_layout(h, T, off);
    if (ws_bytes < need) return bfail(RSB_ERR_OOM, "encoder workspace too small (%s need %ld bytes)", "", (long)need);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* w = static_cast<unsigned char*>(ws);
    __half* Hs = reinterpret_cast<__half*>(w + off[0]);
    __half* QKV = reinterpret_cast<__half*>(w + off[1]);
    __half* CTX = reinterpret_cast<__half*>(w + off[2]);
    __half* TMP = reinterpret_cast<__half*>(w + off[3]);
    __half* FF = reinterpret_cast<__half*>(w + off[4]);
    h->launches = 0;

    const int rows_per_block = 8;   // 256 threads = 8 warps = 8 rows
    const int ln_grid = (T + rows_per_block - 1) / rows_per_block;
    embed_ln_kernel<<<ln_grid, 256, 0, st>>>(input_ids, token_type_ids, cu_seqlens, B, T, h->word, h->pos, h->type,
                                             h->emb_g, h->emb_b, h->eps, h->vocab, h->max_pos, Hs);
    h->launches++;
    if (prepare_attention(h, cu_seqlens, B, max_seqlen, st, &h->launches) != RSB_OK) return bfail(RSB_ERR_OOM, "long-sequence list");
    // RSB_BERT_PROFILE=1 (diagnostic): CUDA events between the kernels of the forward, summed per kernel kind over the
    // layers and printed to stderr after each forward -- per-kernel times INSIDE a back-to-back run (ncu's are isolated,
    // cold-cache and at other clocks).  Synchronises the stream; never set in a timed run.
    static const bool prof = getenv("RSB_BERT_PROFILE") != nullptr;
    enum { P_QKV, P_ATT, P_AO, P_LN1, P_FFN1, P_FFN2, P_LN2, P_KINDS };
    std::vector<cudaEvent_t> pev;
    auto mark = [&]() {
        if (!prof) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        pev.push_back(e);
    };
    mark();
    for (int li = 0; li < h->layers; ++li) {
        Layer& l = h->L[li];
        if (launch_gemm<EPI_BIAS>(Hs, T, l.qkv, QKV, nullptr, st) != RSB_OK) return bfail(RSB_ERR_CUDA, "tensor map encode failed");
        mark();
        launch_attention(h, QKV, cu_seqlens, B, max_seqlen, CTX, st, &h->launches);
        mark();
        if (launch_gemm<EPI_BIAS_RESIDUAL>(CTX, T, l.attn_out, TMP, Hs, st) != RSB_OK) return bfail(RSB_ERR_CUDA, "tensor map encode failed");
        mark();
        launch_layernorm(h, TMP, T, l.ln1_g, l.ln1_b, Hs, st);
        mark();
        if (launch_gemm<EPI_BIAS_GELU>(Hs, T, l.ffn1, FF, nullptr, st) != RSB_OK) return bfail(RSB_ERR_CUDA, "tensor map encode failed");
        mark();
        if (launch_gemm<EPI_BIAS_RESIDUAL>(FF, T, l.ffn2, TMP, Hs, st, true) != RSB_OK) return bfail(RSB_ERR_CUDA, "tensor map encode failed");
        mark();
        launch_layernorm(h, TMP, T, l.ln2_g, l.ln2_b, Hs, st);
        mark();
        h->launches += 6;   // + the attention launch(es), counted in launch_attention
    }
    pool_kernel<<<B, 256, 0, st>>>(Hs, cu_seqlens, pooling, static_cast<__half*>(out_f16));
    h->launches++;
    if (prof) {
        cudaStreamSynchronize(st);
        float sum[P_KINDS] = {};
        for (size_t i = 0; i + 1 < pev.size(); ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, pev[i], pev[i + 1]);
            sum[i % P_KINDS] += ms;
        }
        for (cudaEvent_t e : pev) cudaEventDestroy(e);
        const float L = (float)h->layers * 1e-3f;
        fprintf(stderr, "[rsb_bert profile] T=%d us/layer: qkv %.1f attn %.1f attn_out %.1f ln1 %.1f ffn1 %.1f ffn2 %.1f ln2 %.1f  (sum %.1f)\n", T,
                sum[P_QKV] / L, sum[P_ATT] / L, sum[P_AO] / L, sum[P_LN1] / L, sum[P_FFN1] / L, sum[P_FFN2] / L, sum[P_LN2] / L,
                (sum[0] + sum[1] + sum[2] + sum[3] + sum[4] + sum[5] + sum[6]) / L);
    }
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) return bfail(RSB_ERR_CUDA, "encoder launch failed: %s", cudaGetErrorString(e));
    return RSB_OK;
}

extern "C" int64_t rsb_bert_launches(rsb_bert_t* h) { return h ? h->launches : 0; }

// the forward's attention on its own: qkv [T, 3 x 768] (Q | K | V per token), ctx [T, 768], all fp16
extern "C" int rsb_bert_attention(rsb_bert_t* h, const void* qkv_f16, const int32_t* cu_seqlens, int B, int T, int max_seqlen,
                                  void* ctx_f16, rsb_stream_t stream) {
    if (!h || !qkv_f16 || !cu_seqlens || !ctx_f16) return bfail(RSB_ERR_INVALID, "null argument");
    if (B <= 0 || T <= 0) return bfail(RSB_ERR_INVALID, "empty batch");
    if (max_seqlen > ATT_MAXS) return bfail(RSB_ERR_UNSUPPORTED, "sequence longer than %s%ld tokens", "", (long)ATT_MAXS);
    cudaStream_t st = (cudaStream_t)stream;
    long launches = 0;
    if (prepare_attention(h, cu_seqlens, B, max_seqlen, st, &launches) != RSB_OK) return bfail(RSB_ERR_OOM, "long-sequence list");
    launch_attention(h, static_cast<const __half*>(qkv_f16), cu_seqlens, B, max_seqlen, static_cast<__half*>(ctx_f16), st, &launches);
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) return bfail(RSB_ERR_CUDA, "attention launch failed: %s", cudaGetErrorString(e));
    return RSB_OK;
}

// the forward's LayerNorm on its own (eps of the handle): in / out [T, 768], gamma / beta [768], all fp16
extern "C" int rsb_bert_layernorm(rsb_bert_t* h, const void* in_f16, int T, const void* gamma, const void* beta, void* out_f16,
                                  rsb_stream_t stream) {
    if (!h || !in_f16 || !gamma || !beta || !out_f16) return bfail(RSB_ERR_INVALID, "null argument");
    if (T <= 0) return bfail(RSB_ERR_INVALID, "empty batch");
    launch_layernorm(h, static_cast<const __half*>(in_f16), T, static_cast<const __half*>(gamma), static_cast<const __half*>(beta),
                     static_cast<__half*>(out_f16), (cudaStream_t)stream);
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) return bfail(RSB_ERR_CUDA, "layernorm launch failed: %s", cudaGetErrorString(e));
    return RSB_OK;
}

// plain GEMM entry (tests / roofline of the tensor-core kernel): C[M,N] = A[M,K] W[N,K]^T + bias, epilogue as above;
// RSB_GEMM_ROWS_REVERSED in `epilogue` visits the row tiles last-to-first, as FFN2 does inside the forward
extern "C" int rsb_gemm_f16(const void* A, const void* W, const void* bias, const void* residual, void* C, int M, int N,
                            int K, int epilogue, rsb_stream_t stream) {
    if (!A || !W || !bias || !C) return bfail(RSB_ERR_INVALID, "null argument");
    if (M <= 0 || N % G_BN || K % G_BK || N <= 0 || K <= 0) return bfail(RSB_ERR_INVALID, "need N %% 128 == 0 and K %% 64 == 0");
    const bool m_rev = (epilogue & RSB_GEMM_ROWS_REVERSED) != 0;
    epilogue &= ~RSB_GEMM_ROWS_REVERSED;
    if (epilogue == EPI_BIAS_RESIDUAL && !residual) return bfail(RSB_ERR_INVALID, "residual is NULL");
    Linear lin;
    lin.w = (__half*)W; lin.b = (__half*)bias; lin.N = N; lin.K = K;
    lin.map_ok = make_map(&lin.map, W, N, K, G_BN);      // launch_gemm takes the pair kernel only with a valid map
    if (!lin.map_ok) return bfail(RSB_ERR_CUDA, "tensor map encode failed");
    lin.pair_ok = (N % H_BN == 0) && N <= H_BIAS_MAX;
    cudaStream_t st = (cudaStream_t)stream;
    const __half* Ah = (const __half*)A;
    int rc;
    if (epilogue == EPI_BIAS) rc = launch_gemm<EPI_BIAS>(Ah, M, lin, (__half*)C, nullptr, st, m_rev);
    else if (epilogue == EPI_BIAS_GELU) rc = launch_gemm<EPI_BIAS_GELU>(Ah, M, lin, (__half*)C, nullptr, st, m_rev);
    else if (epilogue == EPI_BIAS_RESIDUAL) rc = launch_gemm<EPI_BIAS_RESIDUAL>(Ah, M, lin, (__half*)C, (const __half*)residual, st, m_rev);
    else return bfail(RSB_ERR_INVALID, "unknown epilogue");
    if (rc != RSB_OK) return bfail(RSB_ERR_CUDA, "tensor map encode failed");
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) return bfail(RSB_ERR_CUDA, "gemm launch failed: %s", cudaGetErrorString(e));
    return RSB_OK;
}
