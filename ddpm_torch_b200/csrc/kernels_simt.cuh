// CUDA-core kernels of the engine: everything that is not a tensor-core contraction
// (GroupNorm, SiLU, dropout, softmax, q_sample / MSE / p_sample tails, layout converters) plus a generic
// tiled conv / wgrad / strided-GEMM used for the geometries the tcgen05 engine does not take
// (Ci=3 / Co=3, stride-2 down-convs, channel counts that are not multiples of 64, tiny token counts).
// All activations are NHWC bf16; statistics, reductions and accumulators are fp32 (fp64 for GroupNorm sums).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ddpm {

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ float silu_f(float y) { return y / (1.f + __expf(-y)); }
__device__ __forceinline__ float silu_grad_f(float y) {
    const float s = 1.f / (1.f + __expf(-y));
    return s * (1.f + y * (1.f - s));
}
// one-MUFU sigmoid for the bandwidth-bound GroupNorm passes (abs error ~5e-4, below bf16 resolution of the outputs)
__device__ __forceinline__ float sigmoid_fast(float y) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * y));
    return fmaf(0.5f, t, 0.5f);
}
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int e = 0; e < 4; ++e) { const float2 t = __bfloat1622float2(h[e]); f[2 * e] = t.x; f[2 * e + 1] = t.y; }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
    uint4 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int e = 0; e < 4; ++e) h[e] = __floats2bfloat162_rn(f[2 * e], f[2 * e + 1]);
    return u;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// counter-based RNG for dropout: Philox4x32-10 keyed by (seed, layer); counter = element index / 4
__device__ __forceinline__ uint4 philox4x32(uint32_t c0, uint32_t c1, uint32_t k0, uint32_t k1) {
    uint32_t c2 = 0, c3 = 0;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
// keep-mask for 8 consecutive elements starting at element index e (multiple of 8): ONE Philox call, 16 random bits per
// element (drop probability quantised to 1/65536)
__device__ __forceinline__ uint32_t dropout_keep8(unsigned long long seed, uint32_t layer, unsigned long long e, float p) {
    const uint32_t thr = (uint32_t)(p * 65536.f);
    const uint4 r = philox4x32((uint32_t)(e >> 3), (uint32_t)(e >> 35), (uint32_t)seed ^ (layer * 0x9E3779B1u), (uint32_t)(seed >> 32));
    uint32_t m = 0;
    m |= ((r.x & 0xffffu) >= thr) << 0; m |= ((r.x >> 16) >= thr) << 1;
    m |= ((r.y & 0xffffu) >= thr) << 2; m |= ((r.y >> 16) >= thr) << 3;
    m |= ((r.z & 0xffffu) >= thr) << 4; m |= ((r.z >> 16) >= thr) << 5;
    m |= ((r.w & 0xffffu) >= thr) << 6; m |= ((r.w >> 16) >= thr) << 7;
    return m;
}

// Sampler epilogue of the final conv (diffusion.py:107-158): when `ps.x` is set the gathered eps never reaches memory - the
// thread that owns pixel (b, y, x) applies the alpha/beta update to its C_out values of x_t in place (same fp32 operation order
// as k_psample_tail / the reference).
struct PsampleEpi { float* x; const float* z; const float* coef; unsigned long long seed; float* pred; /* optional: clipped x0 prediction (p_sample_progressive) */ };
__device__ __forceinline__ float psample_update(float xt, float eps, float zz, float c0, float c1, float c2, float c3, float nzsg, float* pred) {
    float x0 = __fsub_rn(__fmul_rn(c0, xt), __fmul_rn(c1, eps));
    x0 = fminf(fmaxf(x0, -1.f), 1.f);
    if (pred) *pred = x0;
    const float mean = __fadd_rn(__fmul_rn(c2, x0), __fmul_rn(c3, xt));
    return __fadd_rn(mean, __fmul_rn(nzsg, zz));
}
__device__ __forceinline__ float philox_normal(unsigned long long seed, uint32_t step, long long i) {
    const uint4 r = philox4x32((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)seed ^ (step * 0x9E3779B1u), (uint32_t)(seed >> 32));
    const float u1 = ((float)r.x + 1.f) * 2.3283064365386963e-10f, u2 = (float)r.y * 2.3283064365386963e-10f;
    return sqrtf(-2.f * __logf(u1)) * __cosf(6.283185307179586f * u2);
}

// ============================================================================ timestep embedding (functions.py:10-26)
__global__ void k_timestep_embedding(const long long* __restrict__ t, float* __restrict__ out, int B, int dim) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int half = dim / 2;
    if (i >= B * half) return;
    const int b = i / half, j = i % half;
    const float k = logf(10000.f) / (float)(half - 1);
    const float f = expf(-(float)j * k);
    const float a = (float)t[b] * f;
    out[(size_t)b * dim + j] = sinf(a);
    out[(size_t)b * dim + half + j] = cosf(a);
    if ((dim & 1) && j == 0) out[(size_t)b * dim + dim - 1] = 0.f;
}

// ============================================================================ generic strided batched GEMM (CUDA cores)
// C[z][m][n] = alpha * sum_k A(z,m,k) * B(z,k,n) (+ bias[n]) (+ C if accumulate); element strides are arbitrary.
// TA/TB/TC in {float, bf16}.  Optional SiLU on A at load (temb MLP).  64x64x16 tile, 256 threads, 4x4 per thread.
template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ldf<bf16>(const bf16* p) { return __bfloat162float(*p); }
template <typename T> __device__ __forceinline__ void stf(T* p, float v);
template <> __device__ __forceinline__ void stf<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void stf<bf16>(bf16* p, float v) { *p = __float2bfloat16_rn(v); }

struct SgemmParams {
    const void* A; const void* B; void* C; const float* bias;
    int M, N, K;
    long long sa_m, sa_k, sa_z, sb_k, sb_n, sb_z, sc_m, sc_n, sc_z;
    float alpha; int accumulate; int silu_a;      // accumulate: 1 = C += (read-modify-write), 2 = atomicAdd (TC = float only)
    int ksplit;                                   // > 1: blockIdx.z = problem*ksplit + split; K is cut in ksplit ranges, the output
                                                  // (pre-zeroed) is accumulated with atomics and the bias is added by split 0
};

template <typename TC> __device__ __forceinline__ void atomic_addf(TC* p, float v);
template <> __device__ __forceinline__ void atomic_addf<float>(float* p, float v) { atomicAdd(p, v); }
template <> __device__ __forceinline__ void atomic_addf<bf16>(bf16* p, float v) { *p = __float2bfloat16_rn(__bfloat162float(*p) + v); }

template <typename TA, typename TB, typename TC>
__device__ __forceinline__ void sgemm_body(const SgemmParams& p, int bz, int split = 0) {
    __shared__ float As[16][65];
    __shared__ float Bs[16][65];
    const TA* A = reinterpret_cast<const TA*>(p.A) + (long long)bz * p.sa_z;
    const TB* Bm = reinterpret_cast<const TB*>(p.B) + (long long)bz * p.sb_z;
    TC* C = reinterpret_cast<TC*>(p.C) + (long long)bz * p.sc_z;
    const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
    if (m0 >= p.M || n0 >= p.N) return;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[4][4] = {};
    const int ks = p.ksplit > 1 ? p.ksplit : 1;
    const int kper = ((p.K + ks - 1) / ks + 15) / 16 * 16;
    const int kbeg = split * kper;
    int kend = kbeg + kper; if (kend > p.K) kend = p.K;
    for (int k0 = kbeg; k0 < kend; k0 += 16) {
        for (int i = threadIdx.x; i < 1024; i += 256) {
            const int kk = i & 15, r = i >> 4;
            const int m = m0 + r, k = k0 + kk;
            float a = 0.f, b = 0.f;
            if (m < p.M && k < kend) { a = ldf<TA>(A + (long long)m * p.sa_m + (long long)k * p.sa_k); if (p.silu_a) a = silu_f(a); }
            const int n = n0 + r;
            if (n < p.N && k < kend) b = ldf<TB>(Bm + (long long)k * p.sb_k + (long long)n * p.sb_n);
            As[kk][r] = a; Bs[kk][r] = b;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * b[j];
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= p.M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= p.N) continue;
            float v = acc[i][j] * p.alpha;
            if (p.bias && split == 0) v += p.bias[n];
            TC* c = C + (long long)m * p.sc_m + (long long)n * p.sc_n;
            if (p.accumulate == 2 || ks > 1) { atomic_addf<TC>(c, v); continue; }
            if (p.accumulate) v += ldf<TC>(c);
            stf<TC>(c, v);
        }
    }
}
template <typename TA, typename TB, typename TC>
__global__ void __launch_bounds__(256) k_sgemm(const SgemmParams p) {
    pdl_entry();
    const int ks = p.ksplit > 1 ? p.ksplit : 1;
    sgemm_body<TA, TB, TC>(p, blockIdx.z / ks, blockIdx.z % ks);
}
// table-driven: blockIdx.z selects an independent problem (per-ResBlock timestep projections) and its K split
__global__ void __launch_bounds__(256) k_sgemm_table(const SgemmParams* __restrict__ table, int ksplit) {
    pdl_entry();
    const SgemmParams p = table[blockIdx.z / ksplit];
    sgemm_body<float, float, float>(p, 0, blockIdx.z % ksplit);
}
// column sums of an fp32 [M][N] matrix (bias grads of the timestep MLP): out[n] += sum_m A[m][n]
__global__ void k_colsum_f32(const float* __restrict__ A, float* __restrict__ out, int M, int N, long long lda) {
    pdl_entry();
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float s = 0.f;
    for (int m = 0; m < M; ++m) s += A[(long long)m * lda + n];
    atomicAdd(out + n, s);
}
__global__ void k_add_f32(float* __restrict__ dst, const float* __restrict__ a, const float* __restrict__ b, int n) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = a[i] + (b ? b[i] : 0.f);
}

// ============================================================================ GroupNorm (32 groups, eps 1e-6; unet.py:18-20)
// stats: per (b, group) {sum, sumsq} accumulated in fp64 atomics; input = channel-concat of up to two NHWC tensors.
struct GnSrc { const bf16* x0; const bf16* x1; int C0, C1; };   // C = C0 + C1, both multiples of 8

// Launch with blockDim.x = (256/oct)*oct (oct = C/8 <= 256) so that every thread owns ONE channel octet for its whole
// pixel loop: per-channel partial sums stay in registers and are flushed once.
struct GnFin { const float* gamma; const float* beta; float* K; int* ticket; float eps; };   // fused finalize (last block per image)
__global__ void __launch_bounds__(256, 4) k_gn_stats(GnSrc s, double* __restrict__ stats /*[B][32][2]*/, int HW, int pix_per_block, GnFin fin) {
    pdl_entry();
    const int C = s.C0 + s.C1;
    const int oct = C >> 3;                       // 16-byte octets per pixel
    const int cg = C >> 5;                        // channels per group
    const int b = blockIdx.y;
    const int p0 = blockIdx.x * pix_per_block;
    int p1 = p0 + pix_per_block; if (p1 > HW) p1 = HW;
    __shared__ float sh[64];                      // [32][2]
    for (int i = threadIdx.x; i < 64; i += blockDim.x) sh[i] = 0.f;
    __syncthreads();
    const int o = threadIdx.x % oct, lp = threadIdx.x / oct, pstep = blockDim.x / oct;
    const int c = o * 8;
    const bool first = c < s.C0;
    float su[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sq[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const bf16* src = first ? s.x0 + (long long)b * HW * s.C0 + c : s.x1 + (long long)b * HW * s.C1 + (c - s.C0);
    const int sstride = first ? s.C0 : s.C1;
    for (int pp = p0 + lp; pp < p1; pp += 8 * pstep) {
        uint4 u[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int q = pp + k * pstep; u[k] = q < p1 ? __ldg(reinterpret_cast<const uint4*>(src + (long long)q * sstride)) : make_uint4(0, 0, 0, 0); }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            float f[8];
            unpack8(u[k], f);
#pragma unroll
            for (int e = 0; e < 8; ++e) { su[e] += f[e]; sq[e] = fmaf(f[e], f[e], sq[e]); }
        }
    }
    {   // flush: merge elements that share a group before touching shared memory
        int gcur = c / cg; float a1 = 0.f, a2 = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int g = (c + e) / cg;
            if (g != gcur) { atomicAdd(&sh[gcur * 2], a1); atomicAdd(&sh[gcur * 2 + 1], a2); a1 = a2 = 0.f; gcur = g; }
            a1 += su[e]; a2 += sq[e];
        }
        atomicAdd(&sh[gcur * 2], a1); atomicAdd(&sh[gcur * 2 + 1], a2);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 64; i += blockDim.x) atomicAdd(&stats[(long long)b * 64 + i], (double)sh[i]);
    // the block that arrives last for this image turns {sum, sumsq} into the per-channel constants K (saves a launch per norm)
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(fin.ticket + b, 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const double inv_n = 1.0 / ((double)HW * cg);
    float* Kb = fin.K + (long long)b * 4 * C;
    for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
        const int g = ch / cg;
        const double m = __ldcg(&stats[(long long)b * 64 + g * 2]) * inv_n;
        double var = __ldcg(&stats[(long long)b * 64 + g * 2 + 1]) * inv_n - m * m;
        if (var < 0) var = 0;
        const float r = (float)(1.0 / sqrt(var + (double)fin.eps)), mf = (float)m;
        const float scv = r * fin.gamma[ch];
        Kb[ch] = scv; Kb[C + ch] = fin.beta[ch] - mf * scv; Kb[2 * C + ch] = r; Kb[3 * C + ch] = mf * r;
    }
}

// K[b][0..3][C] = { sc = rstd*gamma, sh = beta - mean*sc, r = rstd, mr = mean*rstd }   ->  y = x*sc + sh ; xh = x*r - mr
__device__ __forceinline__ void ld8(const float* p, float (&v)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// y = act(gn(x)) [* dropout] -> bf16 NHWC [B,HW,C] ; grid (pixel blocks, B), blockDim.x = (256/oct)*oct
struct GnApply {
    GnSrc s; const float* K; bf16* y;
    int HW; int silu; float drop_p; unsigned long long seed; uint32_t layer;
    unsigned char* mask;          // [B*HW*C/8] keep bits of the dropout (written when drop_p > 0 and mask != null; read by the backward)
    // statistics delivered by the PRODUCERS of the two sources (conv epilogues, gn_epilogue.cuh): per (image, 4-channel quad)
    // {sum, sum of squares} in fp64, [B][C0/4][2] and [B][C1/4][2].  When qs0 != null the per-channel constants are derived here
    // (every block redoes the few loads of its image - cheaper than a launch) and block 0 of the image publishes them in Kout.
    const double* qs0; const double* qs1; const float* gamma; const float* beta; float eps; float* Kout;
};
// mean / rstd of the group that holds concat-channel ch, from the producers' quad statistics
__device__ __forceinline__ void gn_group_from_quads(const GnApply& a, int b, int ch, int cg, float& mean, float& rstd) {
    const int q0 = (ch / cg) * (cg >> 2), nq = cg >> 2, Q0 = a.s.C0 >> 2, Q1 = a.s.C1 >> 2;
    double S = 0.0, SS = 0.0;
    for (int q = q0; q < q0 + nq; ++q) {
        const double* p = q < Q0 ? a.qs0 + ((long long)b * Q0 + q) * 2 : a.qs1 + ((long long)b * Q1 + (q - Q0)) * 2;
        S += p[0]; SS += p[1];
    }
    const double inv_n = 1.0 / ((double)a.HW * cg);
    const double m = S * inv_n;
    double var = SS * inv_n - m * m;
    if (var < 0) var = 0;
    mean = (float)m; rstd = (float)(1.0 / sqrt(var + (double)a.eps));
}
__global__ void __launch_bounds__(256, 4) k_gn_apply(const GnApply a, int pix_per_block) {
    pdl_entry();
    const int C = a.s.C0 + a.s.C1, oct = C >> 3;
    const int b = blockIdx.y;
    const int p0 = blockIdx.x * pix_per_block;
    int p1 = p0 + pix_per_block; if (p1 > a.HW) p1 = a.HW;
    const int o = threadIdx.x % oct, lp = threadIdx.x / oct, pstep = blockDim.x / oct;
    const int c = o * 8;
    const bool first = c < a.s.C0;
    float sc[8], sh[8];
    if (a.qs0) {
        const int cg = C >> 5;                      // multiple of 4: the thread's 8 channels lie in at most two groups
        float ga[8], be[8], r[2], m[2];
        ld8(a.gamma + c, ga); ld8(a.beta + c, be);
        gn_group_from_quads(a, b, c, cg, m[0], r[0]);
        if ((c + 4) / cg != c / cg) gn_group_from_quads(a, b, c + 4, cg, m[1], r[1]); else { m[1] = m[0]; r[1] = r[0]; }
#pragma unroll
        for (int e = 0; e < 8; ++e) { sc[e] = r[e >> 2] * ga[e]; sh[e] = be[e] - m[e >> 2] * sc[e]; }
        if (a.Kout && blockIdx.x == 0 && lp == 0) {
            float* Kb = a.Kout + (long long)b * 4 * C + c;
#pragma unroll
            for (int e = 0; e < 8; ++e) { Kb[e] = sc[e]; Kb[C + e] = sh[e]; Kb[2 * C + e] = r[e >> 2]; Kb[3 * C + e] = m[e >> 2] * r[e >> 2]; }
        }
    } else {
        ld8(a.K + (long long)b * 4 * C + c, sc); ld8(a.K + (long long)b * 4 * C + C + c, sh);
    }
    const float keep_scale = a.drop_p > 0.f ? 1.f / (1.f - a.drop_p) : 1.f;
    const bf16* src = first ? a.s.x0 + (long long)b * a.HW * a.s.C0 + c : a.s.x1 + (long long)b * a.HW * a.s.C1 + (c - a.s.C0);
    const int sstride = first ? a.s.C0 : a.s.C1;
    bf16* dst = a.y + (long long)b * a.HW * C + c;
    for (int pp = p0 + lp; pp < p1; pp += 4 * pstep) {
        uint4 u[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { const int q = pp + k * pstep; if (q < p1) u[k] = __ldg(reinterpret_cast<const uint4*>(src + (long long)q * sstride)); }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int q = pp + k * pstep;
            if (q >= p1) break;
            float f[8];
            unpack8(u[k], f);
            uint32_t keep = 0xffu;
            if (a.drop_p > 0.f) {
                keep = dropout_keep8(a.seed, a.layer, (unsigned long long)(((long long)b * a.HW + q) * oct + o) * 8, a.drop_p);
                if (a.mask) a.mask[((long long)b * a.HW + q) * oct + o] = (unsigned char)keep;
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float y = fmaf(f[e], sc[e], sh[e]);
                if (a.silu) y *= sigmoid_fast(y);
                f[e] = ((keep >> e) & 1u) ? y * keep_scale : 0.f;
            }
            *reinterpret_cast<uint4*>(dst + (long long)q * C) = pack8(f);
        }
    }
}

// Per-(image, channel) GroupNorm constants K from the producers' quad statistics WITHOUT a pass over the tensor: inference plans
// whose consumer conv applies the norm in its operand path (conv_halo2.cuh, XF).  grid = B, one thread per channel.
__global__ void __launch_bounds__(256) k_gn_prep(const GnApply a) {
    pdl_entry();
    const int C = a.s.C0 + a.s.C1, cg = C >> 5, b = blockIdx.x;
    float* Kb = a.Kout + (long long)b * 4 * C;
    for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
        float m, r;
        gn_group_from_quads(a, b, ch, cg, m, r);
        const float sc = r * __ldg(a.gamma + ch);
        Kb[ch] = sc; Kb[C + ch] = __ldg(a.beta + ch) - m * sc; Kb[2 * C + ch] = r; Kb[3 * C + ch] = m * r;
    }
}

// Small feature maps (H*W <= 64: the 4x4 / 8x8 levels, whose producers are split-K finalizers without a statistics epilogue):
// ONE block per image computes the group statistics and applies the norm in the same launch (the image is 8-32 KB and is
// re-read from L1/L2), instead of a statistics launch + an apply launch.  blockDim.x = (256/oct)*oct as for k_gn_apply.
__global__ void __launch_bounds__(256) k_gn_small(const GnApply a) {
    pdl_entry();
    const int C = a.s.C0 + a.s.C1, oct = C >> 3, cg = C >> 5;
    const int b = blockIdx.x;
    __shared__ float sh[64];                      // [32][2]
    for (int i = threadIdx.x; i < 64; i += blockDim.x) sh[i] = 0.f;
    __syncthreads();
    const int o = threadIdx.x % oct, lp = threadIdx.x / oct, pstep = blockDim.x / oct;
    const int c = o * 8;
    const bool first = c < a.s.C0;
    const bf16* src = first ? a.s.x0 + (long long)b * a.HW * a.s.C0 + c : a.s.x1 + (long long)b * a.HW * a.s.C1 + (c - a.s.C0);
    const int sstride = first ? a.s.C0 : a.s.C1;
    float su[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sq[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int q = lp; q < a.HW; q += pstep) {
        float f[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(src + (long long)q * sstride)), f);
#pragma unroll
        for (int e = 0; e < 8; ++e) { su[e] += f[e]; sq[e] = fmaf(f[e], f[e], sq[e]); }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) { const int g = (c + e) / cg; atomicAdd(&sh[2 * g], su[e]); atomicAdd(&sh[2 * g + 1], sq[e]); }
    __syncthreads();
    const float inv_n = 1.f / ((float)a.HW * (float)cg);
    float sc[8], shf[8];
    float* Kb = a.Kout + (long long)b * 4 * C + c;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int g = (c + e) / cg;
        const float m = sh[2 * g] * inv_n;
        float var = sh[2 * g + 1] * inv_n - m * m; if (var < 0.f) var = 0.f;
        const float r = rsqrtf(var + a.eps);
        sc[e] = r * __ldg(a.gamma + c + e); shf[e] = __ldg(a.beta + c + e) - m * sc[e];
        if (lp == 0) { Kb[e] = sc[e]; Kb[C + e] = shf[e]; Kb[2 * C + e] = r; Kb[3 * C + e] = m * r; }
    }
    const float keep_scale = a.drop_p > 0.f ? 1.f / (1.f - a.drop_p) : 1.f;
    bf16* dst = a.y + (long long)b * a.HW * C + c;
    for (int q = lp; q < a.HW; q += pstep) {
        float f[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(src + (long long)q * sstride)), f);
        uint32_t keep = 0xffu;
        if (a.drop_p > 0.f) {
            keep = dropout_keep8(a.seed, a.layer, (unsigned long long)(((long long)b * a.HW + q) * oct + o) * 8, a.drop_p);
            if (a.mask) a.mask[((long long)b * a.HW + q) * oct + o] = (unsigned char)keep;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float y = fmaf(f[e], sc[e], shf[e]);
            if (a.silu) y *= sigmoid_fast(y);
            f[e] = ((keep >> e) & 1u) ? y * keep_scale : 0.f;
        }
        *reinterpret_cast<uint4*>(dst + (long long)q * C) = pack8(f);
    }
}

// ---- backward of y = act(gn(x))*mask.  With dn = dy * mask * act'(y):
//   pass 1 (reduce):  cs[b][c] = { sum_p dn , sum_p dn*xh }                      (per image, per channel; fp32 atomics)
//   finalize:         S1[b,g] = sum_{c in g} gamma_c cs0 ; S2 = sum gamma_c cs1 ; dgamma_c += sum_b cs1 ; dbeta_c += sum_b cs0
//                     PQ[b][0][c] = rstd^2*S2/n  (=: P) ;  PQ[b][1][c] = rstd*S1/n - P*mean   (=: Q)
//   pass 2 (apply):   dx = sc*dn - P*x - Q  (+ addend) ,  sc = rstd*gamma
struct GnBwd {
    GnSrc s; const bf16* dy; const float* K; const float* gamma;
    float* cs; float* PQ; float* dgamma; float* dbeta;
    bf16* dx0; bf16* dx1; int acc0, acc1;                         // destinations for the two sources (accumulate flags)
    const bf16* addend;                                           // optional [B,HW,C] term added to dx (skip-path gradient)
    int B, HW; int pix_per_block; int silu; float drop_p; unsigned long long seed; uint32_t layer;
    const unsigned char* mask;    // keep bits saved by the forward pass (drop_p > 0)
    int* ticket;                  // [B] arrival counters (zeroed per pass): the last reduce block of an image runs the finalize
    int dn_inplace;               // reduce pass overwrites dy with dn = mask*dy*silu'(y); apply pass reads it back as-is
};
__global__ void __launch_bounds__(256, 2) k_gn_bwd_reduce(const GnBwd a) {
    pdl_entry();   // grid (pixel blocks, B), blockDim.x = (256/oct)*oct
    // cs[b][0][c] = sum_p dn ; cs[b][1][c] = sum_p dn * x   (raw x: the finalize kernel converts to sum dn*xh = r*S - m*r*sum dn)
    // Issue-bound kernel (ncu: issue-active 50% at 16 warps/SM): keep it at <= 64 registers for 4 blocks per SM.
    const int C = a.s.C0 + a.s.C1, oct = C >> 3;
    extern __shared__ float sh2[];                // [2][C]
    for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) sh2[i] = 0.f;
    const int b = blockIdx.y;
    const int p0 = blockIdx.x * a.pix_per_block;
    int p1 = p0 + a.pix_per_block; if (p1 > a.HW) p1 = a.HW;
    const int o = threadIdx.x % oct, lp = threadIdx.x / oct, pstep = blockDim.x / oct;
    const int c = o * 8;
    const bool first = c < a.s.C0;
    const float* Kb = a.K + (long long)b * 4 * C + c;
    float sc[8], sh[8];
    ld8(Kb, sc); ld8(Kb + C, sh);
    const float keep_scale = a.drop_p > 0.f ? 1.f / (1.f - a.drop_p) : 1.f;
    float s0[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s1[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const bf16* src = first ? a.s.x0 + (long long)b * a.HW * a.s.C0 + c : a.s.x1 + (long long)b * a.HW * a.s.C1 + (c - a.s.C0);
    const int sstride = first ? a.s.C0 : a.s.C1;
    const bf16* dyp = a.dy + (long long)b * a.HW * C + c;
    const unsigned char* mk = (a.drop_p > 0.f) ? a.mask + (long long)b * a.HW * oct + o : nullptr;
    for (int pp = p0 + lp; pp < p1; pp += 4 * pstep) {
        uint4 ux[4], ud[4]; uint32_t kp[4] = {0xffu, 0xffu, 0xffu, 0xffu};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int q = pp + k * pstep;
            if (q < p1) {
                ux[k] = __ldg(reinterpret_cast<const uint4*>(src + (long long)q * sstride)); ud[k] = __ldg(reinterpret_cast<const uint4*>(dyp + (long long)q * C));
                if (mk) kp[k] = mk[(long long)q * oct];
            }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int q = pp + k * pstep;
            if (q >= p1) break;
            float x[8], d[8];
            unpack8(ux[k], x); unpack8(ud[k], d);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float dn = ((kp[k] >> e) & 1u) ? d[e] * keep_scale : 0.f;
                if (a.silu) { const float y = fmaf(x[e], sc[e], sh[e]); const float sg = sigmoid_fast(y); dn *= sg * fmaf(y, 1.f - sg, 1.f); }
                s0[e] += dn; s1[e] = fmaf(dn, x[e], s1[e]);
                d[e] = dn;
            }
            // dn (gradient at the normalised pre-activation) replaces dy in place: the apply pass then needs no SiLU / mask math
            if (a.dn_inplace) *reinterpret_cast<uint4*>(const_cast<bf16*>(dyp) + (long long)q * C) = pack8(d);
        }
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < 8; ++e) { atomicAdd(&sh2[c + e], s0[e]); atomicAdd(&sh2[C + c + e], s1[e]); }
    __syncthreads();
    float* csb = a.cs + (long long)b * 2 * C;
    for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) atomicAdd(csb + i, sh2[i]);
    // last block of this image: group sums, dgamma/dbeta, and the per-channel P,Q of the apply pass (was k_gn_bwd_finalize)
    __shared__ int s_last; __shared__ float S[64];
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(a.ticket + b, 1) == (int)gridDim.x - 1);
    if (threadIdx.x < 64) S[threadIdx.x] = 0.f;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int cg = C >> 5;
    const float* Kc = a.K + (long long)b * 4 * C;
    for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
        const float g = __ldg(a.gamma + ch), c0 = __ldcg(csb + ch);
        const float c1 = Kc[2 * C + ch] * __ldcg(csb + C + ch) - Kc[3 * C + ch] * c0;
        atomicAdd(&S[(ch / cg) * 2], g * c0); atomicAdd(&S[(ch / cg) * 2 + 1], g * c1);
        atomicAdd(a.dbeta + ch, c0); atomicAdd(a.dgamma + ch, c1);
    }
    __syncthreads();
    const float inv_n = 1.f / ((float)a.HW * (float)cg);
    float* PQb = a.PQ + (long long)b * 2 * C;
    for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
        const float r = Kc[2 * C + ch], mr = Kc[3 * C + ch];
        const float k2 = r * S[(ch / cg) * 2] * inv_n, k3 = r * S[(ch / cg) * 2 + 1] * inv_n;
        PQb[ch] = k3 * r; PQb[C + ch] = k2 - k3 * mr;
    }
}
// grid (pixel blocks, B), blockDim.x = (256/oct)*oct.  Optionally accumulates per-image / total column sums of dx.
template <bool do_cs>
__global__ void __launch_bounds__(256, 2) k_gn_bwd_apply(const GnBwd a, float* cs_per_img, int cs_ld, float* cs_total, float* cs_total2) {
    pdl_entry();
    const int C = a.s.C0 + a.s.C1, oct = C >> 3;
    extern __shared__ float shc[];                // [C] column sums (only when requested)
    if (do_cs) { for (int i = threadIdx.x; i < C; i += blockDim.x) shc[i] = 0.f; }
    const int b = blockIdx.y;
    const int p0 = blockIdx.x * a.pix_per_block;
    int p1 = p0 + a.pix_per_block; if (p1 > a.HW) p1 = a.HW;
    const int o = threadIdx.x % oct, lp = threadIdx.x / oct, pstep = blockDim.x / oct;
    const int c = o * 8;
    const bool first = c < a.s.C0;
    const float keep_scale = a.drop_p > 0.f ? 1.f / (1.f - a.drop_p) : 1.f;
    const float* Kb = a.K + (long long)b * 4 * C + c;
    const float* PQb = a.PQ + (long long)b * 2 * C + c;
    float sc[8], sh[8], P[8], Q[8];
    ld8(Kb, sc); ld8(Kb + C, sh);
    ld8(PQb, P); ld8(PQb + C, Q);
    const bf16* src = first ? a.s.x0 + (long long)b * a.HW * a.s.C0 + c : a.s.x1 + (long long)b * a.HW * a.s.C1 + (c - a.s.C0);
    const int sstride = first ? a.s.C0 : a.s.C1;
    bf16* dst = first ? a.dx0 + (long long)b * a.HW * a.s.C0 + c : a.dx1 + (long long)b * a.HW * a.s.C1 + (c - a.s.C0);
    const int acc = first ? a.acc0 : a.acc1;
    const bf16* dyp = a.dy + (long long)b * a.HW * C + c;
    const bf16* adp = a.addend ? a.addend + (long long)b * a.HW * C + c : nullptr;
    const unsigned char* mk = (a.drop_p > 0.f) ? a.mask + (long long)b * a.HW * oct + o : nullptr;
    float cs[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int pp = p0 + lp; pp < p1; pp += 2 * pstep) {
        uint4 ux[2], ud[2], ua[2], uo[2]; uint32_t kp[2] = {0xffu, 0xffu};
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int q = pp + k * pstep;
            if (q < p1) {
                ux[k] = __ldg(reinterpret_cast<const uint4*>(src + (long long)q * sstride));
                ud[k] = __ldg(reinterpret_cast<const uint4*>(dyp + (long long)q * C));
                if (adp) ua[k] = __ldg(reinterpret_cast<const uint4*>(adp + (long long)q * C));
                if (acc) uo[k] = *reinterpret_cast<const uint4*>(dst + (long long)q * sstride);
                if (mk && !a.dn_inplace) kp[k] = mk[(long long)q * oct];
            }
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int q = pp + k * pstep;
            if (q >= p1) break;
            float x[8], d[8], ov[8], ad[8];
            unpack8(ux[k], x); unpack8(ud[k], d);
            if (acc) unpack8(uo[k], ov);
            if (adp) unpack8(ua[k], ad);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float dn = d[e];
                if (!a.dn_inplace) {
                    dn = ((kp[k] >> e) & 1u) ? d[e] * keep_scale : 0.f;
                    if (a.silu) { const float y = fmaf(x[e], sc[e], sh[e]); const float sg = sigmoid_fast(y); dn *= sg * fmaf(y, 1.f - sg, 1.f); }
                }
                float v = fmaf(sc[e], dn, -fmaf(P[e], x[e], Q[e]));
                if (adp) v += ad[e];
                if (acc) v += ov[e];
                ov[e] = v; if (do_cs) cs[e] += v;
            }
            *reinterpret_cast<uint4*>(dst + (long long)q * sstride) = pack8(ov);
        }
    }
    if (do_cs) {
        __syncthreads();
#pragma unroll
        for (int e = 0; e < 8; ++e) atomicAdd(&shc[c + e], cs[e]);
        __syncthreads();
        for (int i = threadIdx.x; i < C; i += blockDim.x) {
            const float v = shc[i];
            if (cs_per_img) atomicAdd(cs_per_img + (long long)b * cs_ld + i, v);
            if (cs_total) atomicAdd(cs_total + i, v);
            if (cs_total2) atomicAdd(cs_total2 + i, v);
        }
    }
}

// (Two single-launch variants of this backward were built, verified against the oracle and measured in round 2 - a cluster per
// image with the dy / x slabs staged in shared memory by bulk async copies, and a CTA per (image, group slice) with the pairs
// resident in registers - and removed: both cut HBM traffic to the 3-4 pass minimum but serialise load -> reduce -> apply
// inside a CTA that owns most of an SM, and the training step got slower (9.84-10.1 ms vs 9.20 ms);
// profiles/r02_gn_backward_fused_experiment.txt.)

// ============================================================================ generic conv (CUDA cores)
// out[b,oy,ox,co] = sum_{tap,ci} in[b, iy(oy,ky), ix(ox,kx), ci] * Wp[co][tap*Cin + ci]  (+bias +rowvec[b] +residual)
// map 0: iy = oy*stride + ky - pad ; map 1 (dgrad of the stride-2 conv): iy = (oy-ky)/2 when even ; map 2: nearest-2x
// upsample fused: iy = (oy+ky-1)>>1 on the 2x grid.
enum ConvMap { MAP_NORMAL = 0, MAP_TRANSPOSED2 = 1, MAP_UPSAMPLE2 = 2 };
struct ConvG {
    GnSrc in; const bf16* wp; long long ldw;     // packed weights [Co][ldw]
    const float* bias; const float* rowvec; int rowvec_ld; const bf16* residual;
    void* out; int out_nchw_f32;
    int B, Hi, Wi, Ho, Wo, Co, ksize, stride, pad, map;
    int accumulate;                              // out += (bf16 NHWC only)
};
__device__ __forceinline__ bool conv_map_coord(int map, int o, int k, int stride, int pad, int n_in, int& i) {
    if (map == MAP_NORMAL) { i = o * stride + k - pad; return i >= 0 && i < n_in; }
    if (map == MAP_TRANSPOSED2) { const int d = o - k; i = d >> 1; return d >= 0 && !(d & 1) && i < n_in; }
    const int u = o + k - 1; i = u >> 1; return u >= 0 && i < n_in;
}
__global__ void __launch_bounds__(256) k_conv_generic(const ConvG c) {
    pdl_entry();
    __shared__ float As[16][65];
    __shared__ float Bs[16][65];
    const int Cin = c.in.C0 + c.in.C1;
    const int taps = c.ksize * c.ksize;
    const int P = c.B * c.Ho * c.Wo;
    const int p0 = blockIdx.x * 64, co0 = blockIdx.y * 64;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int lp = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;     // loader: row (pixel / co) and 4-wide k offset
    // loader pixel coordinates
    const int pl = p0 + lp;
    int lb = 0, loy = 0, lox = 0;
    if (pl < P) { lb = pl / (c.Ho * c.Wo); const int r = pl % (c.Ho * c.Wo); loy = r / c.Wo; lox = r % c.Wo; }
    float acc[4][4] = {};
    for (int t = 0; t < taps; ++t) {
        const int ky = c.ksize == 3 ? t / 3 : 0, kx = c.ksize == 3 ? t % 3 : 0;
        int iy = 0, ix = 0;
        bool valid = pl < P;
        if (c.ksize == 3 || c.map != MAP_NORMAL || c.stride != 1) {
            valid = valid && conv_map_coord(c.map, loy, ky, c.stride, c.pad, c.Hi, iy) && conv_map_coord(c.map, lox, kx, c.stride, c.pad, c.Wi, ix);
        } else { iy = loy; ix = lox; }
        const long long ipix = ((long long)lb * c.Hi + iy) * c.Wi + ix;
        for (int k0 = 0; k0 < Cin; k0 += 16) {
            {   // A tile: 64 pixels x 16 channels
                const int ci = k0 + lk;
                float f[4] = {0, 0, 0, 0};
                if (valid && ci < Cin) {
                    const bf16* src = ci < c.in.C0 ? c.in.x0 + ipix * c.in.C0 + ci : c.in.x1 + ipix * c.in.C1 + (ci - c.in.C0);
                    const uint2 u = *reinterpret_cast<const uint2*>(src);
                    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
                    const float2 a0 = __bfloat1622float2(h[0]), a1 = __bfloat1622float2(h[1]);
                    f[0] = a0.x; f[1] = a0.y; f[2] = a1.x; f[3] = a1.y;
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) As[lk + e][lp] = f[e];
            }
            {   // B tile: 64 out-channels x 16 k
                const int co = co0 + lp, ci = k0 + lk;
                float f[4] = {0, 0, 0, 0};
                if (co < c.Co && ci < Cin) {
                    const uint2 u = *reinterpret_cast<const uint2*>(c.wp + (long long)co * c.ldw + (long long)t * Cin + ci);
                    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
                    const float2 a0 = __bfloat1622float2(h[0]), a1 = __bfloat1622float2(h[1]);
                    f[0] = a0.x; f[1] = a0.y; f[2] = a1.x; f[3] = a1.y;
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) Bs[lk + e][lp] = f[e];
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < 16; ++kk) {
                float a[4], b[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * b[j];
            }
            __syncthreads();
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int pp = p0 + ty * 4 + i;
        if (pp >= P) continue;
        const int b = pp / (c.Ho * c.Wo);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int co = co0 + tx * 4 + j;
            if (co >= c.Co) continue;
            float v = acc[i][j];
            if (c.bias) v += c.bias[co];
            if (c.rowvec) v += c.rowvec[(long long)b * c.rowvec_ld + co];
            if (c.residual) v += __bfloat162float(c.residual[(long long)pp * c.Co + co]);
            if (c.out_nchw_f32) {
                const int r = pp % (c.Ho * c.Wo);
                reinterpret_cast<float*>(c.out)[((long long)b * c.Co + co) * (c.Ho * c.Wo) + r] = v;
            } else {
                bf16* o = reinterpret_cast<bf16*>(c.out) + (long long)pp * c.Co + co;
                if (c.accumulate) v += __bfloat162float(*o);
                *o = __float2bfloat16_rn(v);
            }
        }
    }
}

// generic wgrad: dW[co][ci][tap] (strides given) += sum_p dy[p][co] * in[map(p,tap)][ci]   (fp32 atomics, split over pixels)
struct WgradG {
    const bf16* dy; GnSrc in; float* dw; long long s_co, s_ci, s_tap;
    int B, Hi, Wi, Ho, Wo, Co, ksize, stride, pad, map, pix_per_split;
    int Co_valid;                                 // rows of dW actually written (dy may be channel-padded)
};
__global__ void __launch_bounds__(256) k_wgrad_generic(const WgradG c) {
    pdl_entry();
    __shared__ float As[16][65];   // [pixel][co]
    __shared__ float Bs[16][65];   // [pixel][ci]
    const int Cin = c.in.C0 + c.in.C1;
    const int taps = c.ksize * c.ksize;
    const int t = blockIdx.z % taps, split = blockIdx.z / taps;
    const int ky = c.ksize == 3 ? t / 3 : 0, kx = c.ksize == 3 ? t % 3 : 0;
    const int P = c.B * c.Ho * c.Wo;
    const int co0 = blockIdx.y * 64, ci0 = blockIdx.x * 64;
    const int pbeg = split * c.pix_per_split;
    int pend = pbeg + c.pix_per_split; if (pend > P) pend = P;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int lpix = threadIdx.x >> 4, lc = (threadIdx.x & 15) * 4;   // loader: pixel in chunk, 4-wide channel offset
    float acc[4][4] = {};
    for (int pc = pbeg; pc < pend; pc += 16) {
        const int pp = pc + lpix;
        float fa[4] = {0, 0, 0, 0}, fb[4] = {0, 0, 0, 0};
        if (pp < pend) {
            const int b = pp / (c.Ho * c.Wo), r = pp % (c.Ho * c.Wo), oy = r / c.Wo, ox = r % c.Wo;
            const int co = co0 + lc;
#pragma unroll
            for (int e = 0; e < 4; ++e) if (co + e < c.Co) fa[e] = __bfloat162float(c.dy[(long long)pp * c.Co + co + e]);
            int iy, ix;
            bool valid = conv_map_coord(c.map, oy, ky, c.stride, c.pad, c.Hi, iy) && conv_map_coord(c.map, ox, kx, c.stride, c.pad, c.Wi, ix);
            if (c.ksize == 1 && c.map == MAP_NORMAL && c.stride == 1) { iy = oy; ix = ox; valid = true; }
            if (valid) {
                const long long ipix = ((long long)b * c.Hi + iy) * c.Wi + ix;
                const int ci = ci0 + lc;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int cc = ci + e;
                    if (cc < Cin) fb[e] = __bfloat162float(cc < c.in.C0 ? c.in.x0[ipix * c.in.C0 + cc] : c.in.x1[ipix * c.in.C1 + (cc - c.in.C0)]);
                }
            }
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) { As[lpix][lc + e] = fa[e]; Bs[lpix][lc + e] = fb[e]; }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * b[j];
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int co = co0 + ty * 4 + i;
        if (co >= c.Co_valid) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ci = ci0 + tx * 4 + j;
            if (ci >= Cin) continue;
            atomicAdd(c.dw + co * c.s_co + ci * c.s_ci + t * c.s_tap, acc[i][j]);
        }
    }
}

// ============================================================================ in_conv: NCHW fp32 [B,Ci<=4,H,W] -> NHWC bf16 [B,H,W,Co], 3x3 pad 1
// Also used as the data-gradient of the 3-channel out_conv (x := d_eps, w := flipped/transposed weights).
// w layout: [Co][CI*9] fp32 (OIHW), out NHWC bf16.  CI <= 4, Co % 32 == 0.
// lane <-> pixel (two pixels per lane, 64 per warp); output channels are produced 32 at a time with the weights fetched as
// warp-broadcast 16-byte shared-memory reads, so one fetch feeds 64 pixels (the per-octet version was shared-memory bound).
// q_sample prologue (diffusion.py:92-97): with `noise` set, the kernel's input is x_t = sqrt_ab[t_b]*x + sqrt_1mab[t_b]*noise,
// formed while the taps are loaded (same two multiplies + add as the reference); the centre tap also stores x_t to `xt_out`
// (the weight gradient of this conv needs it in the backward pass).
struct QsamplePro { const float* noise; const long long* t; const float* tab_a; const float* tab_s; float* xt_out; };
template <int CI>
__global__ void __launch_bounds__(128) k_in_conv(const float* __restrict__ x, const float* __restrict__ w,
                                                const float* __restrict__ bias, bf16* __restrict__ out,
                                                int B, int H, int W, int Co, double* qstats, const QsamplePro qp) {
    pdl_entry();
    extern __shared__ float sw[];                 // [CI*9][Co] + [Co]
    constexpr int K = CI * 9;
    for (int i = threadIdx.x; i < Co * K; i += blockDim.x) sw[(i % K) * Co + i / K] = w[i];
    for (int i = threadIdx.x; i < Co; i += blockDim.x) sw[Co * K + i] = bias ? bias[i] : 0.f;
    __syncthreads();
    const long long P = (long long)B * H * W;
    const int lane = threadIdx.x & 31;
    const long long warp_id = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long base = warp_id * 64; base < P; base += nwarps * 64) {
        float in[2][K];
        long long pix[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            pix[u] = base + u * 32 + lane;
            const bool pv = pix[u] < P;
            const int b = pv ? (int)(pix[u] / (H * W)) : 0, r = pv ? (int)(pix[u] % (H * W)) : 0, y = r / W, xx = r % W;
            float qa = 1.f, qs_ = 0.f;
            if (qp.noise && pv) { const long long tb = qp.t[b]; qa = __ldg(qp.tab_a + tb); qs_ = __ldg(qp.tab_s + tb); }
#pragma unroll
            for (int ci = 0; ci < CI; ++ci)
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                    const int iy = y + t / 3 - 1, ix = xx + t % 3 - 1;
                    float v = 0.f;
                    if (pv && iy >= 0 && iy < H && ix >= 0 && ix < W) {
                        const long long j = (((long long)b * CI + ci) * H + iy) * W + ix;
                        v = __ldg(x + j);
                        if (qp.noise) {
                            v = __fadd_rn(__fmul_rn(qa, v), __fmul_rn(qs_, __ldg(qp.noise + j)));
                            if (t == 4) qp.xt_out[j] = v;
                        }
                    }
                    in[u][ci * 9 + t] = v;
                }
        }
        for (int c0 = 0; c0 < Co; c0 += 32) {
            float acc[2][32];
#pragma unroll
            for (int j = 0; j < 32; ++j) { const float bv = sw[Co * K + c0 + j]; acc[0][j] = bv; acc[1][j] = bv; }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const float v0 = in[0][k], v1 = in[1][k];
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 wv = *reinterpret_cast<const float4*>(sw + k * Co + c0 + j4 * 4);     // warp-uniform address: broadcast
                    acc[0][j4 * 4] = fmaf(v0, wv.x, acc[0][j4 * 4]); acc[0][j4 * 4 + 1] = fmaf(v0, wv.y, acc[0][j4 * 4 + 1]);
                    acc[0][j4 * 4 + 2] = fmaf(v0, wv.z, acc[0][j4 * 4 + 2]); acc[0][j4 * 4 + 3] = fmaf(v0, wv.w, acc[0][j4 * 4 + 3]);
                    acc[1][j4 * 4] = fmaf(v1, wv.x, acc[1][j4 * 4]); acc[1][j4 * 4 + 1] = fmaf(v1, wv.y, acc[1][j4 * 4 + 1]);
                    acc[1][j4 * 4 + 2] = fmaf(v1, wv.z, acc[1][j4 * 4 + 2]); acc[1][j4 * 4 + 3] = fmaf(v1, wv.w, acc[1][j4 * 4 + 3]);
                }
            }
            if (qstats) {      // GroupNorm statistics of the output (gn_epilogue.cuh): H*W % 32 == 0, so a warp's 32 pixels share an image
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const long long p0w = base + u * 32;                     // warp-uniform
                    if (p0w >= P) continue;
                    const int nimg = (int)(p0w / (H * W));
                    epi_quad_stats(acc[u], pix[u] < P, qstats + ((long long)nimg * (Co >> 2) + (c0 >> 2)) * 2, lane);
                }
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                if (pix[u] >= P) continue;
                uint4* op = reinterpret_cast<uint4*>(out + pix[u] * Co + c0);
#pragma unroll
                for (int j8 = 0; j8 < 4; ++j8) {
                    float f[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) f[e] = acc[u][j8 * 8 + e];
                    op[j8] = pack8(f);
                }
            }
        }
    }
}
// Correlation of a wide NHWC bf16 tensor with a narrow NCHW fp32 tensor (3x3 window):
//   acc[C][ci][t] = sum_p wide[p][C] * narrow[b, ci, y + t/3 - 1, x + t%3 - 1]
// = weight gradient of in_conv (wide = dY, narrow = x_t):   dW[C][ci][t]      -> dw[C*s_c + ci*s_ci + t*s_t]
// = weight gradient of out_conv (wide = a, narrow = d_eps):  dW[ci][C][8 - t]  (flip_t = 1, strides swapped by the caller)
// thread <-> wide channel C (blockDim.x = C <= 256); the narrow 3x3 patches of 32 pixels are staged in shared memory.
template <int CI>
__global__ void __launch_bounds__(256) k_corr3x3(const bf16* __restrict__ wide, const float* __restrict__ narrow, float* __restrict__ dw,
                                                 long long s_c, long long s_ci, long long s_t, int flip_t, float* __restrict__ dbias_wide,
                                                 int B, int H, int W, int C, int pix_per_block) {
    pdl_entry();
    constexpr int K = CI * 9, PB = 32;
    __shared__ float sx[PB][K + 1];
    const int c = threadIdx.x;
    const long long P = (long long)B * H * W;
    const long long p0 = (long long)blockIdx.x * pix_per_block;
    long long p1 = p0 + pix_per_block; if (p1 > P) p1 = P;
    float acc[K]; float accb = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.f;
    for (long long pb = p0; pb < p1; pb += PB) {
        __syncthreads();
        for (int i = threadIdx.x; i < PB * K; i += blockDim.x) {
            const int pp = i / K, k = i % K, ci = k / 9, t = k % 9;
            const long long p = pb + pp;
            float v = 0.f;
            if (p < p1) {
                const int b = (int)(p / (H * W)), r = (int)(p % (H * W)), y = r / W, xx = r % W;
                const int iy = y + t / 3 - 1, ix = xx + t % 3 - 1;
                if (iy >= 0 && iy < H && ix >= 0 && ix < W) v = narrow[(((long long)b * CI + ci) * H + iy) * W + ix];
            }
            sx[pp][k] = v;
        }
        __syncthreads();
        if (c < C) {
            const int n = (int)((p1 - pb) < PB ? (p1 - pb) : PB);
            for (int pp = 0; pp < n; ++pp) {
                const float d = __bfloat162float(wide[(pb + pp) * C + c]);
                accb += d;
#pragma unroll
                for (int k = 0; k < K; ++k) acc[k] += d * sx[pp][k];
            }
        }
    }
    if (c < C) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int ci = k / 9, t = k % 9;
            atomicAdd(dw + c * s_c + ci * s_ci + (flip_t ? 8 - t : t) * s_t, acc[k]);
        }
        if (dbias_wide) atomicAdd(dbias_wide + c, accb);
    }
}
// out_conv forward: NHWC bf16 [B,H,W,C] -> NCHW fp32 [B,Co<=4,H,W], 3x3 pad 1.  4 lanes per pixel (C/4 channels each),
// weights [Co][C][9] (OIHW fp32) staged in shared memory as [9][Co][C].
template <int CO>
__global__ void __launch_bounds__(256) k_out_conv(const bf16* __restrict__ a, const float* __restrict__ w, const float* __restrict__ bias,
                                                 float* __restrict__ out, int B, int H, int W, int C) {
    pdl_entry();
    // 4 lanes per pixel group (C/4 channels each); a lane handles PX consecutive pixels of a row so that every 16-byte
    // weight fetch from shared memory feeds PX pixels (the one-pixel version was bound by shared-memory reads)
    constexpr int PX = 4;
    extern __shared__ float sw[];                 // [9][CO][C]
    for (int i = threadIdx.x; i < CO * C * 9; i += blockDim.x) {
        const int t = i % 9, c = (i / 9) % C, co = i / (9 * C);
        sw[(t * CO + co) * C + c] = w[i];
    }
    __syncthreads();
    const int WG = W / PX;                        // pixel groups per row (W % 4 == 0)
    const long long G = (long long)B * H * WG;
    const int lane4 = threadIdx.x & 3;
    const int cpl = C >> 2;                       // channels per lane (multiple of 8)
    for (long long g = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 2; g < G; g += ((long long)gridDim.x * blockDim.x) >> 2) {
        const int b = (int)(g / (H * WG)), r = (int)(g % (H * WG)), y = r / WG, x0 = (r % WG) * PX;
        float acc[PX][CO];
#pragma unroll
        for (int p = 0; p < PX; ++p)
#pragma unroll
            for (int co = 0; co < CO; ++co) acc[p][co] = 0.f;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            const int iy = y + ky - 1;
            if (iy < 0 || iy >= H) continue;
            const bf16* rowp = a + (((long long)b * H + iy) * W) * C + lane4 * cpl;
            for (int c8 = 0; c8 < cpl; c8 += 8) {
                float f[PX + 2][8];               // input columns x0-1 .. x0+PX
#pragma unroll
                for (int j = 0; j < PX + 2; ++j) {
                    const int ix = x0 + j - 1;
                    if (ix >= 0 && ix < W) unpack8(__ldg(reinterpret_cast<const uint4*>(rowp + (long long)ix * C + c8)), f[j]);
                    else {
#pragma unroll
                        for (int e = 0; e < 8; ++e) f[j][e] = 0.f;
                    }
                }
#pragma unroll
                for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                    for (int co = 0; co < CO; ++co) {
                        const float* wr = sw + ((ky * 3 + kx) * CO + co) * C + lane4 * cpl + c8;
                        const float4 w0 = *reinterpret_cast<const float4*>(wr), w1 = *reinterpret_cast<const float4*>(wr + 4);
#pragma unroll
                        for (int p = 0; p < PX; ++p) {
                            const float* ff = f[p + kx];
                            acc[p][co] += ff[0] * w0.x + ff[1] * w0.y + ff[2] * w0.z + ff[3] * w0.w + ff[4] * w1.x + ff[5] * w1.y + ff[6] * w1.z + ff[7] * w1.w;
                        }
                    }
            }
        }
#pragma unroll
        for (int p = 0; p < PX; ++p)
#pragma unroll
            for (int co = 0; co < CO; ++co) {
                acc[p][co] += __shfl_xor_sync(0xffffffffu, acc[p][co], 1);
                acc[p][co] += __shfl_xor_sync(0xffffffffu, acc[p][co], 2);
            }
        if (lane4 == 0) {
#pragma unroll
            for (int co = 0; co < CO; ++co) {
                float4 o4 = make_float4(acc[0][co] + bias[co], acc[1][co] + bias[co], acc[2][co] + bias[co], acc[3][co] + bias[co]);
                *reinterpret_cast<float4*>(out + ((long long)b * CO + co) * (H * W) + y * W + x0) = o4;
            }
        }
    }
}
// w'[c][co*9 + t'] = w[co][c][8 - t']  : the 3->C "in_conv" whose forward is the data-gradient of out_conv
__global__ void k_flip_transpose_w(const float* __restrict__ w, float* __restrict__ wt, int Co, int C) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Co * C * 9) return;
    const int t = i % 9, c = (i / 9) % C, co = i / (9 * C);
    wt[(c * Co + co) * 9 + (8 - t)] = w[i];
}
// sum over pixels of a narrow NCHW fp32 tensor: out[c] += sum_{b,p} x[b][c][p]   (bias gradient of out_conv)
__global__ void __launch_bounds__(256) k_chansum_nchw(const float* __restrict__ x, float* __restrict__ out, int B, int C, int HW) {
    pdl_entry();
    const int c = blockIdx.y;
    float s = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)B * HW; i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / HW), r = (int)(i % HW);
        s += x[((long long)b * C + c) * HW + r];
    }
    s = warp_sum(s);
    __shared__ float sh[8];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { float t = 0.f; for (int k = 0; k < 8; ++k) t += sh[k]; atomicAdd(out + c, t); }
}
// ============================================================================ column sums: per image and total
// dy [B][HW][C] bf16 -> per_img[b][ld] (+=, fp32 atomics, optional) and total[c] (+=)
__global__ void __launch_bounds__(256) k_colsum(const bf16* __restrict__ dy, float* per_img, int ld, float* total, float* total2,
                                               int HW, int C, int C_valid, int pix_per_block) {
    pdl_entry();
    // blockDim.x = (256/oct)*oct: one channel octet per thread; partials are merged in shared memory so that each block
    // issues ONE atomic per channel (the first version issued one per thread and spent 14 ms/step in contention)
    extern __shared__ float sh[];                 // [C]
    const int b = blockIdx.y;
    const int p0 = blockIdx.x * pix_per_block;
    int p1 = p0 + pix_per_block; if (p1 > HW) p1 = HW;
    const int oct = C >> 3;
    for (int i = threadIdx.x; i < C; i += blockDim.x) sh[i] = 0.f;
    __syncthreads();
    const int o = threadIdx.x % oct, lp = threadIdx.x / oct, pstep = blockDim.x / oct;
    float s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int p = p0 + lp; p < p1; p += pstep) {
        float f[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(dy + ((long long)b * HW + p) * C + o * 8)), f);
#pragma unroll
        for (int e = 0; e < 8; ++e) s[e] += f[e];
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) atomicAdd(&sh[o * 8 + e], s[e]);
    __syncthreads();
    for (int i = threadIdx.x; i < C_valid; i += blockDim.x) {
        const float v = sh[i];
        if (per_img) atomicAdd(per_img + (long long)b * ld + i, v);
        if (total) atomicAdd(total + i, v);
        if (total2) atomicAdd(total2 + i, v);
    }
}

// ============================================================================ softmax over rows of S fp32 [rows][T] -> P bf16
__global__ void __launch_bounds__(256) k_softmax_rows(const float* __restrict__ S, bf16* __restrict__ P, long long rows, int T) {
    pdl_entry();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * 8 + warp;
    if (row >= rows) return;
    const float* s = S + row * T;
    float mx = -3.0e38f;
    for (int j = lane; j < T; j += 32) mx = fmaxf(mx, s[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int j = lane; j < T; j += 32) sum += __expf(s[j] - mx);
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    for (int j = lane; j < T; j += 32) P[row * T + j] = __float2bfloat16_rn(__expf(s[j] - mx) * inv);
}
// dS = P * (dP - rowsum(dP*P)) * scale  -> bf16
__global__ void __launch_bounds__(256) k_softmax_bwd(const bf16* __restrict__ P, const float* __restrict__ dP, bf16* __restrict__ dS,
                                                    long long rows, int T, float scale) {
    pdl_entry();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * 8 + warp;
    if (row >= rows) return;
    float dot = 0.f;
    for (int j = lane; j < T; j += 32) dot += __bfloat162float(P[row * T + j]) * dP[row * T + j];
    dot = warp_sum(dot);
    for (int j = lane; j < T; j += 32)
        dS[row * T + j] = __float2bfloat16_rn(__bfloat162float(P[row * T + j]) * (dP[row * T + j] - dot) * scale);
}

// ============================================================================ whole attention for T = 16 tokens (4x4 level)
// unet.py:37-60 at the 4x4 resolution: softmax(Q K^T / sqrt(C)) V is 2 x 16x16xC products per image - far below one MMA tile,
// so the three launches of the generic route (SIMT GEMM, softmax, SIMT GEMM; five more in backward) are pure latency.  One CTA
// per image keeps the image's [16][3C] q|k|v rows in shared memory and does scores, softmax and P.V (backward: dP, dS, dQ, dK,
// dV) in one launch.  Rows are padded by 8 elements so the 16 K rows of a score column land in different banks.
__device__ __forceinline__ float dot8_bf16(const uint4 a, const uint4 b) {
    const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
    const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) { const float2 x = __bfloat1622float2(pa[i]), y = __bfloat1622float2(pb[i]); acc = fmaf(x.x, y.x, fmaf(x.y, y.y, acc)); }
    return acc;
}
constexpr int ATTN16_T = 16;
inline size_t attn16_smem(int C, bool bwd) {
    return (size_t)ATTN16_T * (3 * C + 8) * 2 + (bwd ? (size_t)ATTN16_T * (C + 8) * 2 : 0) + 2 * ATTN16_T * ATTN16_T * 4;
}
inline bool attn16_eligible(int T, int C) { return T == ATTN16_T && (C == 128 || C == 256 || C == 512); }

__global__ void __launch_bounds__(256) k_attn16_fwd(const bf16* __restrict__ qkv, bf16* __restrict__ O, bf16* __restrict__ Pm, int C, float scale) {
    pdl_entry();
    constexpr int T = ATTN16_T;
    extern __shared__ __align__(16) unsigned char sm_raw[];
    const int ld = 3 * C + 8;
    bf16* s = reinterpret_cast<bf16*>(sm_raw);
    float* P = reinterpret_cast<float*>(sm_raw + (size_t)T * ld * 2);
    const int n = blockIdx.x, tid = threadIdx.x;
    const bf16* src = qkv + (long long)n * T * 3 * C;
    const int oct = 3 * C / 8;
    for (int i = tid; i < T * oct; i += 256) { const int r = i / oct, o = i % oct; *reinterpret_cast<uint4*>(s + r * ld + o * 8) = __ldg(reinterpret_cast<const uint4*>(src + (long long)r * 3 * C) + o); }
    __syncthreads();
    {   // thread = one (query i, key j) pair; the 16 keys of a query sit in one half-warp
        const int i = tid / T, j = tid % T;
        const bf16* qi = s + i * ld; const bf16* kj = s + j * ld + C;
        float acc = 0.f;
        for (int c = 0; c < C; c += 8) acc += dot8_bf16(*reinterpret_cast<const uint4*>(qi + c), *reinterpret_cast<const uint4*>(kj + c));
        acc *= scale;
        float mx = acc;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float e = __expf(acc - mx);
        float sum = e;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        const bf16 pb = __float2bfloat16_rn(e / sum);      // the probabilities the backward pass reads are the ones applied here
        P[tid] = __bfloat162float(pb);
        if (Pm) Pm[(long long)n * T * T + tid] = pb;
    }
    __syncthreads();
    const int npair = C / 2, groups = 256 / npair, rows = T / groups;
    const int cp = tid % npair, r0 = (tid / npair) * rows;
    float2 v[T];
#pragma unroll
    for (int j = 0; j < T; ++j) v[j] = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(s + j * ld + 2 * C + 2 * cp));
    for (int i = r0; i < r0 + rows; ++i) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int j = 0; j < T; ++j) { const float p = P[i * T + j]; a0 = fmaf(p, v[j].x, a0); a1 = fmaf(p, v[j].y, a1); }
        *reinterpret_cast<__nv_bfloat162*>(O + ((long long)n * T + i) * C + 2 * cp) = __floats2bfloat162_rn(a0, a1);
    }
}

// dqkv[n][t][0:C | C:2C | 2C:3C] = dQ | dK | dV  from dO, the saved probabilities and q|k|v
__global__ void __launch_bounds__(256) k_attn16_bwd(const bf16* __restrict__ qkv, const bf16* __restrict__ dO, const bf16* __restrict__ Pm,
                                                   bf16* __restrict__ dqkv, int C, float scale) {
    pdl_entry();
    constexpr int T = ATTN16_T;
    extern __shared__ __align__(16) unsigned char sm_raw[];
    const int ld = 3 * C + 8, ldo = C + 8;
    bf16* s = reinterpret_cast<bf16*>(sm_raw);
    bf16* sdo = s + (size_t)T * ld;
    float* P = reinterpret_cast<float*>(sm_raw + (size_t)T * ld * 2 + (size_t)T * ldo * 2);
    float* dS = P + T * T;
    const int n = blockIdx.x, tid = threadIdx.x;
    const bf16* src = qkv + (long long)n * T * 3 * C;
    const bf16* gsrc = dO + (long long)n * T * C;
    const int oct = 3 * C / 8, octo = C / 8;
    for (int i = tid; i < T * oct; i += 256) { const int r = i / oct, o = i % oct; *reinterpret_cast<uint4*>(s + r * ld + o * 8) = __ldg(reinterpret_cast<const uint4*>(src + (long long)r * 3 * C) + o); }
    for (int i = tid; i < T * octo; i += 256) { const int r = i / octo, o = i % octo; *reinterpret_cast<uint4*>(sdo + r * ldo + o * 8) = __ldg(reinterpret_cast<const uint4*>(gsrc + (long long)r * C) + o); }
    {
        const int i = tid / T, j = tid % T;
        const float p = __bfloat162float(Pm[(long long)n * T * T + tid]);
        P[tid] = p;
        __syncthreads();
        const bf16* gi = sdo + i * ldo; const bf16* vj = s + j * ld + 2 * C;
        float dp = 0.f;
        for (int c = 0; c < C; c += 8) dp += dot8_bf16(*reinterpret_cast<const uint4*>(gi + c), *reinterpret_cast<const uint4*>(vj + c));
        float dot = p * dp;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        dS[tid] = __bfloat162float(__float2bfloat16_rn(p * (dp - dot) * scale));
    }
    __syncthreads();
    const int npair = C / 2, groups = 256 / npair, rows = T / groups;
    const int cp = tid % npair, r0 = (tid / npair) * rows;
    bf16* dst = dqkv + (long long)n * T * 3 * C + 2 * cp;
    float2 x[T];
    // dQ[i] = sum_j dS[i][j] k[j]
#pragma unroll
    for (int j = 0; j < T; ++j) x[j] = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(s + j * ld + C + 2 * cp));
    for (int i = r0; i < r0 + rows; ++i) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int j = 0; j < T; ++j) { const float w = dS[i * T + j]; a0 = fmaf(w, x[j].x, a0); a1 = fmaf(w, x[j].y, a1); }
        *reinterpret_cast<__nv_bfloat162*>(dst + (long long)i * 3 * C) = __floats2bfloat162_rn(a0, a1);
    }
    // dK[j] = sum_i dS[i][j] q[i]
#pragma unroll
    for (int i = 0; i < T; ++i) x[i] = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(s + i * ld + 2 * cp));
    for (int j = r0; j < r0 + rows; ++j) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int i = 0; i < T; ++i) { const float w = dS[i * T + j]; a0 = fmaf(w, x[i].x, a0); a1 = fmaf(w, x[i].y, a1); }
        *reinterpret_cast<__nv_bfloat162*>(dst + (long long)j * 3 * C + C) = __floats2bfloat162_rn(a0, a1);
    }
    // dV[j] = sum_i P[i][j] dO[i]
#pragma unroll
    for (int i = 0; i < T; ++i) x[i] = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(sdo + i * ldo + 2 * cp));
    for (int j = r0; j < r0 + rows; ++j) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int i = 0; i < T; ++i) { const float w = P[i * T + j]; a0 = fmaf(w, x[i].x, a0); a1 = fmaf(w, x[i].y, a1); }
        *reinterpret_cast<__nv_bfloat162*>(dst + (long long)j * 3 * C + 2 * C) = __floats2bfloat162_rn(a0, a1);
    }
}

// ============================================================================ nearest 2x upsample (unet.py:199) and its adjoint
__global__ void k_upsample2x(const bf16* __restrict__ in, bf16* __restrict__ out, int B, int H, int W, int C) {
    pdl_entry();
    const int oct = C >> 3;
    const long long total = (long long)B * 4 * H * W * oct;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long pix = i / oct; const int o = (int)(i % oct);
        const int b = (int)(pix / (4 * H * W)), r = (int)(pix % (4 * H * W)), y = r / (2 * W), x = r % (2 * W);
        reinterpret_cast<uint4*>(out)[i] = __ldg(reinterpret_cast<const uint4*>(in) + (((long long)b * H + (y >> 1)) * W + (x >> 1)) * oct + o);
    }
}
__global__ void k_upsample2x_bwd(const bf16* __restrict__ dout, bf16* __restrict__ din, int B, int H, int W, int C, int accumulate) {
    pdl_entry();
    const int oct = C >> 3;
    const long long total = (long long)B * H * W * oct;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long pix = i / oct; const int o = (int)(i % oct);
        const int b = (int)(pix / (H * W)), r = (int)(pix % (H * W)), y = r / W, x = r % W;
        float s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float f[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(dout) + (((long long)b * 2 * H + 2 * y + (q >> 1)) * 2 * W + 2 * x + (q & 1)) * oct + o), f);
#pragma unroll
            for (int e = 0; e < 8; ++e) s[e] += f[e];
        }
        if (accumulate) {
            float f[8];
            unpack8(reinterpret_cast<const uint4*>(din)[i], f);
#pragma unroll
            for (int e = 0; e < 8; ++e) s[e] += f[e];
        }
        reinterpret_cast<uint4*>(din)[i] = pack8(s);
    }
}
// dst (+)= src  (bf16, 8 at a time)
__global__ void k_add_bf16(bf16* __restrict__ dst, const bf16* __restrict__ src, long long n_oct, int accumulate) {
    pdl_entry();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_oct; i += (long long)gridDim.x * blockDim.x) {
        if (!accumulate) { reinterpret_cast<uint4*>(dst)[i] = __ldg(reinterpret_cast<const uint4*>(src) + i); continue; }
        float a[8], b[8];
        unpack8(reinterpret_cast<const uint4*>(dst)[i], a);
        unpack8(__ldg(reinterpret_cast<const uint4*>(src) + i), b);
#pragma unroll
        for (int e = 0; e < 8; ++e) a[e] += b[e];
        reinterpret_cast<uint4*>(dst)[i] = pack8(a);
    }
}

// ============================================================================ diffusion tails
// q_sample (diffusion.py:92-97): x_t = sqrt_ab[t]*x0 + sqrt_1m_ab[t]*noise, fp32 NCHW, same op order as the reference
__global__ void k_qsample(const float* __restrict__ x0, const float* __restrict__ noise, const long long* __restrict__ t,
                          const float* __restrict__ tab_a, const float* __restrict__ tab_s, float* __restrict__ xt, int per_img, long long total) {
    pdl_entry();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / per_img);
        const float a = tab_a[t[b]], s = tab_s[t[b]];
        xt[i] = __fadd_rn(__fmul_rn(a, x0[i]), __fmul_rn(s, noise[i]));
    }
}
// per-sample MSE (diffusion.py:239, functions.py:99-101) and d(loss)/d(eps) = gscale[b] * 2*(eps-target)/per_img as NHWC bf16
__global__ void __launch_bounds__(256) k_mse(const float* __restrict__ eps, const float* __restrict__ target, float* __restrict__ losses, int per_img) {
    pdl_entry();
    const int b = blockIdx.x;
    float s = 0.f;
    for (int i = threadIdx.x; i < per_img; i += blockDim.x) {
        const float d = target[(long long)b * per_img + i] - eps[(long long)b * per_img + i];
        s += d * d;
    }
    __shared__ float sh[8];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { float tsum = 0.f; for (int w = 0; w < 8; ++w) tsum += sh[w]; losses[b] = tsum / (float)per_img; }
}
// gradient of the per-sample MSE w.r.t. eps (fp32 NCHW): d_eps = gscale[b] * 2*(eps-target)/per_img
__global__ void k_mse_grad(const float* __restrict__ eps, const float* __restrict__ target, const float* __restrict__ gscale,
                           float* __restrict__ d_eps, int per_img, long long total) {
    pdl_entry();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / per_img);
        d_eps[i] = gscale[b] * 2.f * (eps[i] - target[i]) / (float)per_img;
    }
}
__global__ void k_nchw_f32_to_nhwc_bf16(const float* __restrict__ src, bf16* __restrict__ dst, int B, int C, int HW, int Cp) {
    pdl_entry();
    const long long total = (long long)B * HW * Cp;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % Cp); const long long pix = i / Cp; const int b = (int)(pix / HW), r = (int)(pix % HW);
        dst[i] = __float2bfloat16_rn(c < C ? src[((long long)b * C + c) * HW + r] : 0.f);
    }
}
// p_sample_step tail (diffusion.py:107-158, eps-prediction, fixed variance, clip_denoised):
//   x0 = clamp(c0*x_t - c1*eps, -1, 1) ; mean = c2*x0 + c3*x_t ; x = mean + nz*sigma*z        coef = {c0,c1,c2,c3,sigma}
//   coef[5] = nonzero flag (t>0) as float, coef[6] = step index (for the built-in noise stream)
//   z == nullptr and seed != 0: the noise is drawn in-kernel (Philox4x32-10 + Box-Muller; NOT torch's stream)
__global__ void k_psample_tail(const float* __restrict__ eps, float* __restrict__ x /*in: x_t, out: x_{t-1}*/, const float* __restrict__ z,
                               const float* __restrict__ coef, unsigned long long seed, long long total, float* pred) {
    pdl_entry();
    const float c0 = coef[0], c1 = coef[1], c2 = coef[2], c3 = coef[3], nzsg = __fmul_rn(coef[5], coef[4]);
    const uint32_t step = (uint32_t)coef[6];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        float zz = 0.f;
        if (z) zz = z[i];
        else if (seed) zz = philox_normal(seed, step, i);
        x[i] = psample_update(x[i], eps[i], zz, c0, c1, c2, c3, nzsg, pred ? pred + i : nullptr);
    }
}
// generate.py:129  (x * 127.5 + 127.5).round().clamp(0, 255).to(uint8).permute(0, 2, 3, 1): NCHW fp32 -> NHWC uint8.
// Bit-exact with the reference expression: separate fp32 multiply and add (no FMA contraction), round-half-to-even.
template <int C>
__global__ void k_to_uint8_nhwc(const float* __restrict__ x, unsigned char* __restrict__ out, long long npix /*B*H*W*/, int HW) {
    pdl_entry();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / HW; const int p = (int)(i - b * HW);
        const float* src = x + b * C * (long long)HW + p;
        unsigned char v[C];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            float f = __fadd_rn(__fmul_rn(__ldg(src + (long long)c * HW), 127.5f), 127.5f);
            f = fminf(fmaxf(rintf(f), 0.f), 255.f);
            v[c] = (unsigned char)f;
        }
        unsigned char* o = out + i * C;
        if (C == 4) *reinterpret_cast<uchar4*>(o) = make_uchar4(v[0], v[1], v[2], v[3]);
        else {
#pragma unroll
            for (int c = 0; c < C; ++c) o[c] = v[c];
        }
    }
}
// Widths of the narrow convolutions' tensor-core operands (in_conv / out_conv.2, 1..16 image channels):
//   im2col_width(c): row length KP of a 3x3 patch matrix over c channels, 9*c columns zero padded to whole 64-wide K slabs
//   tap_width(c):    row length TW of out_conv's tap outputs, 32 for c <= 3 (one half-slab N tile), else im2col_width(c)
__host__ __device__ constexpr int im2col_width(int c) { return (9 * c + 63) / 64 * 64; }
__host__ __device__ constexpr int tap_width(int c) { return c <= 3 ? 32 : im2col_width(c); }
// out_conv on the tensor cores (unet.py:138-142): the 3x3 conv C -> CO is computed as a 1x1 GEMM to 9*CO "tap outputs"
// per pixel, T[p][t*CO + co] = sum_c a[p][c] * w[co][c][t] (fp32, [P][TW], TW = tap_width(CO)), followed by this gather:
// out[b][co][y][x] = bias[co] + sum_t T[(b, y + t/3 - 1, x + t%3 - 1)][t*CO + co]  (zero outside the image).
// k_pack_tapco builds the GEMM's B operand: rows r = t*CO + co of [TW][C] bf16 (rows >= 9*CO stay zero).
__global__ void k_pack_tapco(const float* __restrict__ w /*[CO][C][9]*/, bf16* __restrict__ out /*[TW][C]*/, int CO, int C) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= CO * C * 9) return;
    const int t = i % 9, c = (i / 9) % C, co = i / (9 * C);
    out[(long long)(t * CO + co) * C + c] = __float2bfloat16_rn(w[i]);
}
// transposed pack for the data gradient: out[c][t*CO + co] = w[co][c][t]   ([C][ld] bf16, ld = im2col_width(CO), columns >= 9*CO stay zero)
__global__ void k_pack_tapco_t(const float* __restrict__ w, bf16* __restrict__ out, int CO, int C, int ld) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= CO * C * 9) return;
    const int t = i % 9, c = (i / 9) % C, co = i / (9 * C);
    out[(long long)c * ld + t * CO + co] = __float2bfloat16_rn(w[i]);
}
// 3x3 im2col of a narrow NCHW fp32 image (CI <= 16 channels) into NHWC bf16 rows of KP = im2col_width(CI):
// dst[p][t*CI + ci] = src[ci][p + sign*o_t], o_t = (t/3 - 1, t%3 - 1), zero outside the image and for columns >= 9*CI.
// sign = +1: the conv's input patches (in_conv forward and weight gradient); sign = -1: the patches the transposed conv sees
// (data and weight gradients of out_conv over d_eps).  A row leaves in 16-byte pieces of 8 columns, so only one piece is held
// in registers (a 192-wide row would not fit).
// With qp.noise set the source is x_t = q_sample(x0, t, noise) formed on the fly (same arithmetic as k_in_conv); the centre tap
// also stores x_t to qp.xt_out.
template <int CI>
__global__ void __launch_bounds__(256) k_im2col3(const float* __restrict__ src, bf16* __restrict__ dst, int B, int H, int W, int sign, const QsamplePro qp) {
    pdl_entry();
    constexpr int KP = im2col_width(CI);
    const long long P = (long long)B * H * W;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (long long)gridDim.x * blockDim.x) {
        const int x = (int)(i % W), y = (int)((i / W) % H); const long long b = i / ((long long)W * H);
        float qa = 1.f, qs_ = 0.f;
        if (qp.noise) { const long long tb = qp.t[b]; qa = __ldg(qp.tab_a + tb); qs_ = __ldg(qp.tab_s + tb); }
        uint4* o = reinterpret_cast<uint4*>(dst + i * KP);
#pragma unroll
        for (int pc = 0; pc < KP / 8; ++pc) {
            __align__(16) bf16 piece[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int k = pc * 8 + e, t = k / CI, ci = k % CI;
                float v = 0.f;
                const int yy = y + sign * (t / 3 - 1), xx = x + sign * (t % 3 - 1);
                if (k < 9 * CI && yy >= 0 && yy < H && xx >= 0 && xx < W) {
                    const long long j = ((b * CI + ci) * H + yy) * W + xx;
                    v = __ldg(src + j);
                    if (qp.noise) {
                        v = __fadd_rn(__fmul_rn(qa, v), __fmul_rn(qs_, __ldg(qp.noise + j)));
                        if (t == 4) qp.xt_out[j] = v;
                    }
                }
                piece[e] = __float2bfloat16_rn(v);
            }
            o[pc] = *reinterpret_cast<const uint4*>(piece);
        }
    }
}
// in_conv weights OIHW fp32 [Co][CI][3][3] -> bf16 [Co][KP], column t*CI + ci (the patch order of k_im2col3), zero padded
__global__ void k_pack_in(const float* __restrict__ w, bf16* __restrict__ wp, int Co, int CI, int KP) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Co * KP) return;
    const int co = i / KP, k = i % KP, t = k / CI, ci = k % CI;
    wp[i] = __float2bfloat16_rn(k < 9 * CI ? w[(co * CI + ci) * 9 + t] : 0.f);
}
// tap-major GEMM results back to OIHW fp32 gradients:
//   mode 0 (out_conv):  gw[(co*C + c)*9 + t]  = S[(t*CO + co)*C + c]      S = [ld][C]
//   mode 1 (in_conv):   gw[(co*CI + ci)*9 + t] = S[co*ld + t*CI + ci]     S = [C][ld]      (ld = im2col_width of the image channels)
__global__ void k_unpack_tap(const float* __restrict__ S, float* __restrict__ gw, int CO, int CI, int mode, int ld) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= CO * CI * 9) return;
    const int t = i % 9, ci = (i / 9) % CI, co = i / (9 * CI);
    gw[i] = mode == 0 ? S[(long long)(t * CO + co) * CI + ci] : S[(long long)co * ld + t * CI + ci];
}
template <int CO>
__global__ void __launch_bounds__(256) k_out_gather(const float* __restrict__ T /*[P][TW]*/, const float* __restrict__ bias, float* __restrict__ out /*NCHW*/,
                                                   int B, int H, int W, const PsampleEpi ps) {
    pdl_entry();
    constexpr int TW = tap_width(CO);
    const long long P = (long long)B * H * W;
    float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f, nzsg = 0.f; uint32_t step = 0;
    if (ps.x) { c0 = ps.coef[0]; c1 = ps.coef[1]; c2 = ps.coef[2]; c3 = ps.coef[3]; nzsg = __fmul_rn(ps.coef[5], ps.coef[4]); step = (uint32_t)ps.coef[6]; }
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (long long)gridDim.x * blockDim.x) {
        const int x = (int)(i % W), y = (int)((i / W) % H); const long long b = i / ((long long)W * H);
        float acc[CO];
#pragma unroll
        for (int co = 0; co < CO; ++co) acc[co] = bias ? __ldg(bias + co) : 0.f;
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
            if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
            const float* r = T + ((b * H + yy) * W + xx) * TW + t * CO;
#pragma unroll
            for (int co = 0; co < CO; ++co) acc[co] += __ldg(r + co);
        }
        if (ps.x) {
#pragma unroll
            for (int co = 0; co < CO; ++co) {
                const long long j = ((b * CO + co) * H + y) * W + x;
                float zz = 0.f;
                if (ps.z) zz = ps.z[j];
                else if (ps.seed) zz = philox_normal(ps.seed, step, j);
                ps.x[j] = psample_update(ps.x[j], acc[co], zz, c0, c1, c2, c3, nzsg, ps.pred ? ps.pred + j : nullptr);
            }
            continue;
        }
#pragma unroll
        for (int co = 0; co < CO; ++co) out[((b * CO + co) * H + y) * W + x] = acc[co];
    }
}
// ---- timestep-embedding projections on the tensor cores (unet.py:77,86: 22 x Linear(512 -> Cout) share one input):
// the per-block fc weights are concatenated into Wcat [tp_ld][E] (bf16, K-major; padding rows zero), its transpose
// WcatT [E][tp_ld] (for the data gradient) and bias_cat [tp_ld]; the weight gradient lands in a [tp_ld][E] scratch and is
// scattered back to the per-block OIHW gradients.
struct FcEnt { const float* w; const float* b; float* gw; int cout; int off; };
// grid (E/32, maxc/32, nblocks), block (32, 8): 32x32 tiles through shared memory so both layouts are written coalesced
__global__ void k_pack_fc(const FcEnt* __restrict__ tab, bf16* __restrict__ Wcat, bf16* __restrict__ WcatT, float* __restrict__ bias_cat, int E, int tp_ld) {
    pdl_entry();
    const FcEnt e = tab[blockIdx.z];
    const int o0 = blockIdx.y * 32, e0 = blockIdx.x * 32;
    if (o0 >= e.cout) return;
    __shared__ float tile[32][33];
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int o = o0 + j;
        const float v = (o < e.cout) ? e.w[(long long)o * E + e0 + threadIdx.x] : 0.f;
        tile[j][threadIdx.x] = v;
        if (o < e.cout) Wcat[(long long)(e.off + o) * E + e0 + threadIdx.x] = __float2bfloat16_rn(v);
    }
    __syncthreads();
    if (WcatT)
        for (int j = threadIdx.y; j < 32; j += 8) {
            const int o = o0 + threadIdx.x;
            if (o < e.cout) WcatT[(long long)(e0 + j) * tp_ld + e.off + o] = __float2bfloat16_rn(tile[threadIdx.x][j]);
        }
    if (blockIdx.x == 0 && threadIdx.y == 0 && o0 + threadIdx.x < e.cout) bias_cat[e.off + o0 + threadIdx.x] = e.b[o0 + threadIdx.x];
}
// grid (ceil(maxc*E/4/256), nblocks): gw[o][e] = Sw[off + o][e]
__global__ void k_scatter_fc_grad(const FcEnt* __restrict__ tab, const float4* __restrict__ Sw, int E) {
    pdl_entry();
    const FcEnt e = tab[blockIdx.y];
    const long long n4 = (long long)e.cout * E / 4, i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n4) reinterpret_cast<float4*>(e.gw)[i] = Sw[(long long)e.off * E / 4 + i];
}
__global__ void k_cast_bf16(const float* __restrict__ x, bf16* __restrict__ y, long long n, int silu) {
    pdl_entry();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float v = x[i];
        if (silu) v = v / (1.f + __expf(-v));
        y[i] = __float2bfloat16_rn(v);
    }
}
// rows 1..B-1 of a [B][row4] float4 matrix <- row 0
__global__ void k_bcast_rows(float4* __restrict__ m, long long row4, long long tot4) {
    pdl_entry();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < tot4) m[row4 + i] = m[i % row4];
}
// one block: fetch step i = *counter, broadcast t_model[i] to t_buf[B], copy the coefficient row, then advance the counter
__global__ void k_sampler_prep(int* __restrict__ counter, const long long* __restrict__ t_model, const float* __restrict__ coef_table /*[S][6]*/,
                               long long* __restrict__ t_buf, float* __restrict__ coef_cur /*[7]*/, int B) {
    pdl_entry();
    const int i = *counter;
    for (int b = threadIdx.x; b < B; b += blockDim.x) t_buf[b] = t_model[i];
    if (threadIdx.x < 6) coef_cur[threadIdx.x] = coef_table[i * 6 + threadIdx.x];
    if (threadIdx.x == 6) coef_cur[6] = (float)i;
    __syncthreads();
    if (threadIdx.x == 0) *counter = i - 1;
}

// ============================================================================ weight (re)packing
// OIHW fp32 -> fwd pack [Co][ld_f] at column k_off + tap*Ci + ci (bf16)   and   dgrad pack [Ci][ld_d] at tap'*Co + co,
// tap' = flip ? 8 - tap : tap   (flip for stride-1 3x3; no flip for the stride-2 gather form and 1x1)
__global__ void k_pack_conv_w(const float* __restrict__ w, bf16* fwd, long long ld_f, int k_off, bf16* dgr, long long ld_d, int flip,
                              int Co, int Ci, int taps) {
    pdl_entry();
    const long long total = (long long)Co * Ci * taps;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(i % taps); const long long r = i / taps; const int ci = (int)(r % Ci), co = (int)(r / Ci);
        const bf16 v = __float2bfloat16_rn(w[i]);
        if (fwd) fwd[(long long)co * ld_f + k_off + (long long)t * Ci + ci] = v;
        if (dgr) dgr[(long long)ci * ld_d + (long long)(flip ? taps - 1 - t : t) * Co + co] = v;
    }
}
// dgrad pack with a padded Co (out_conv: Co=3 -> 8): dgr[ci][tap'*Cop + co]
__global__ void k_pack_conv_w_padded(const float* __restrict__ w, bf16* dgr, long long ld_d, int flip, int Co, int Cop, int Ci, int taps) {
    pdl_entry();
    const long long total = (long long)Co * Ci * taps;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(i % taps); const long long r = i / taps; const int ci = (int)(r % Ci), co = (int)(r / Ci);
        dgr[(long long)ci * ld_d + (long long)(flip ? taps - 1 - t : t) * Cop + co] = __float2bfloat16_rn(w[i]);
    }
}

// data-gradient pack of a stride-2 3x3 conv: [Ci][9*Co] bf16 in four output-parity blocks
// {(py,px)=(0,0): 4 taps @0, (0,1): 2 taps @4Co, (1,0): 2 taps @6Co, (1,1): 1 tap @8Co}; taps ordered (ky asc, kx asc).
__global__ void k_pack_conv_w_s2dgrad(const float* __restrict__ w, bf16* __restrict__ dgr, long long ld_d, int Co, int Ci) {
    pdl_entry();
    const long long total = (long long)Co * Ci * 9;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(i % 9); const long long r = i / 9; const int ci = (int)(r % Ci), co = (int)(r / Ci);
        const int ky = t / 3, kx = t % 3, py = ky & 1, px = kx & 1;
        const int base = (py == 0 ? (px == 0 ? 0 : 4) : (px == 0 ? 6 : 8)) * Co;
        const int j = (py ? 0 : ky / 2) * (px ? 1 : 2) + (px ? 0 : kx / 2);
        dgr[(long long)ci * ld_d + base + (long long)j * Co + co] = __float2bfloat16_rn(w[i]);
    }
}
// ---- table-driven weight maintenance: ONE launch re-packs every conv weight (grid.y = table entry)
enum PackKind { PK_CONV = 0, PK_BIAS_ADD = 1, PK_FLIP_T = 2, PK_UNPACK_GRAD = 3, PK_UPFOLD = 4, PK_IDENTITY = 5 };
struct PackEntry {
    int kind; int Co, Ci, taps; int k_off; int dkind;   // dkind: 0 none, 1 dgrad, 2 dgrad flipped taps, 3 stride-2 parity dgrad
    const float* w; const float* w2; bf16* fwd; long long ld_f; bf16* dgr; long long ld_d; float* fout; float* scratch;
};
__device__ __forceinline__ int pack_dcol(const PackEntry& e, int t) {     // column block of tap t in the dgrad pack
    if (e.dkind == 1) return t * e.Co;
    if (e.dkind == 2) return (e.taps - 1 - t) * e.Co;
    const int ky = t / 3, kx = t % 3, py = ky & 1, px = kx & 1;
    return (py == 0 ? (px == 0 ? 0 : 4) : (px == 0 ? 6 : 8)) * e.Co + ((py ? 0 : ky / 2) * (px ? 1 : 2) + (px ? 0 : kx / 2)) * e.Co;
}
// grid (tiles, entries).  Conv weights / gradient unpacks go through an 8(co) x 64(ci) x taps shared-memory tile so that both
// the fp32 side and the packed side are accessed in 16-byte-or-larger contiguous pieces (the element-wise first version spent
// 0.6 ms/step on 2-byte scattered writes).
__global__ void __launch_bounds__(256) k_pack_table(const PackEntry* __restrict__ table) {
    pdl_entry();
    const PackEntry e = table[blockIdx.y];
    if (e.kind == PK_BIAS_ADD) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e.Co; i += gridDim.x * blockDim.x) e.fout[i] = e.w[i] + (e.w2 ? e.w2[i] : 0.f);
        return;
    }
    if (e.kind == PK_FLIP_T) {
        const long long total = (long long)e.Co * e.Ci * e.taps;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
            const int t = (int)(i % e.taps); const long long r = i / e.taps; const int ci = (int)(r % e.Ci), co = (int)(r / e.Ci);
            e.fout[((long long)ci * e.Co + co) * 9 + (8 - t)] = e.w[i];
        }
        return;
    }
    if (e.kind == PK_IDENTITY) {     // fwd[co][k_off + ci] = (co == ci): the residual of a ResidualBlock as extra K chunks of its conv2
        const long long total = (long long)e.Co * (e.Ci / 8);
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
            const int o = (int)(i % (e.Ci / 8)), co = (int)(i / (e.Ci / 8));
            float f[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) f[u] = (o * 8 + u == co) ? 1.f : 0.f;
            *reinterpret_cast<uint4*>(e.fwd + (long long)co * e.ld_f + e.k_off + o * 8) = pack8(f);
        }
        return;
    }
    if (e.kind == PK_UPFOLD) {
        // nearest-2x upsample folded into the 3x3 conv that follows it (unet.py:199-202): output pixel (2y+py, 2x+px) sees a 2x2
        // neighbourhood of the LOW-resolution input, with the 3x3 taps that land on the same input pixel summed:
        //   rows  py=0: {ky=0} -> y-1, {ky=1,2} -> y      py=1: {ky=0,1} -> y, {ky=2} -> y+1      (columns alike)
        // fwd[co][(q*4 + a*2 + b)*Ci + ci], q = py*2+px, (a, b) = the 2x2 tap in (row, column) order
        const long long total = (long long)e.Co * 16 * (e.Ci / 8);
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
            const int o = (int)(i % (e.Ci / 8)); const int tq = (int)((i / (e.Ci / 8)) % 16); const int co = (int)(i / ((long long)16 * (e.Ci / 8)));
            const int q = tq >> 2, a = (tq >> 1) & 1, b = tq & 1, py = q >> 1, px = q & 1;
            const int ky0 = py == 0 ? (a == 0 ? 0 : 1) : (a == 0 ? 0 : 2), ky1 = py == 0 ? (a == 0 ? 0 : 2) : (a == 0 ? 1 : 2);
            const int kx0 = px == 0 ? (b == 0 ? 0 : 1) : (b == 0 ? 0 : 2), kx1 = px == 0 ? (b == 0 ? 0 : 2) : (b == 0 ? 1 : 2);
            float f[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const float* wp = e.w + ((long long)co * e.Ci + o * 8 + u) * 9;
                float acc = 0.f;
                for (int ky = ky0; ky <= ky1; ++ky) for (int kx = kx0; kx <= kx1; ++kx) acc += wp[ky * 3 + kx];
                f[u] = acc;
            }
            *reinterpret_cast<uint4*>(e.fwd + (long long)co * e.ld_f + (long long)tq * e.Ci + o * 8) = pack8(f);
        }
        return;
    }
    __shared__ float sm[8][64 * 9 + 1];
    const int T = e.taps;
    const int tiles_ci = (e.Ci + 63) / 64, tiles = (e.Co / 8) * tiles_ci;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int co0 = (tile / tiles_ci) * 8, ci0 = (tile % tiles_ci) * 64;
        const int nci = (e.Ci - ci0) < 64 ? (e.Ci - ci0) : 64;
        const int row = nci * T;
        __syncthreads();
        if (e.kind == PK_CONV) {
            for (int idx = threadIdx.x; idx < 8 * row; idx += blockDim.x) {
                const int r = idx / row, j = idx % row;
                sm[r][j] = e.w[((long long)(co0 + r) * e.Ci + ci0) * T + j];                 // sm[r][ci*T + t]
            }
        } else {   // PK_UNPACK_GRAD: scratch [t][Co][Ci] fp32 -> tile, cleared behind the read
            for (int idx = threadIdx.x; idx < 8 * row; idx += blockDim.x) {
                const int ci = idx % nci, r = (idx / nci) % 8, t = idx / (nci * 8);
                float* sp = e.scratch + ((long long)t * e.Co + co0 + r) * e.Ci + ci0 + ci;
                sm[r][ci * T + t] = *sp; *sp = 0.f;
            }
        }
        __syncthreads();
        if (e.kind == PK_UNPACK_GRAD) {
            for (int idx = threadIdx.x; idx < 8 * row; idx += blockDim.x) {
                const int r = idx / row, j = idx % row;
                e.fout[((long long)(co0 + r) * e.Ci + ci0) * T + j] = sm[r][j];
            }
            continue;
        }
        if (e.fwd) {
            const int octs = nci / 8;
            for (int idx = threadIdx.x; idx < 8 * T * octs; idx += blockDim.x) {
                const int o = idx % octs, t = (idx / octs) % T, r = idx / (octs * T);
                float f[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) f[q] = sm[r][(o * 8 + q) * T + t];
                *reinterpret_cast<uint4*>(e.fwd + (long long)(co0 + r) * e.ld_f + e.k_off + (long long)t * e.Ci + ci0 + o * 8) = pack8(f);
            }
        }
        if (e.dkind) {
            for (int idx = threadIdx.x; idx < row; idx += blockDim.x) {
                const int ci = idx / T, t = idx % T;
                float f[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) f[q] = sm[q][ci * T + t];
                *reinterpret_cast<uint4*>(e.dgr + (long long)(ci0 + ci) * e.ld_d + pack_dcol(e, t) + co0) = pack8(f);
            }
        }
    }
}
// split-K finalize: out(bf16) = scratch(fp32) + bias + rowvec[b] + residual ; scratch is cleared behind the read
__global__ void __launch_bounds__(256) k_splitk_finalize(float* __restrict__ scratch, const float* __restrict__ bias, const float* __restrict__ rowvec,
                                                        int rowvec_ld, int rows_per_vec, const bf16* __restrict__ residual, bf16* __restrict__ out,
                                                        long long M, int N) {
    pdl_entry();
    const long long total = M * (N / 8);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / (N / 8); const int c = (int)(i % (N / 8)) * 8;
        float4* sp = reinterpret_cast<float4*>(scratch + row * N + c);
        const float4 a = sp[0], b = sp[1];
        sp[0] = make_float4(0, 0, 0, 0); sp[1] = make_float4(0, 0, 0, 0);
        float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        if (bias) { for (int e = 0; e < 8; ++e) f[e] += __ldg(bias + c + e); }
        if (rowvec) { const float* rv = rowvec + (row / rows_per_vec) * rowvec_ld + c; for (int e = 0; e < 8; ++e) f[e] += __ldg(rv + e); }
        if (residual) { float r8[8]; unpack8(__ldg(reinterpret_cast<const uint4*>(residual + row * N + c)), r8); for (int e = 0; e < 8; ++e) f[e] += r8[e]; }
        *reinterpret_cast<uint4*>(out + row * N + c) = pack8(f);
    }
}
// packed grad [tap][Co][Ci] fp32 -> OIHW fp32 (=)
// (the scratch is cleared behind the read so the next backward starts from zeros without a memset)
__global__ void k_unpack_conv_grad(float* __restrict__ packed, float* __restrict__ g, int Co, int Ci, int taps) {
    pdl_entry();
    const long long total = (long long)Co * Ci * taps;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(i % taps); const long long r = i / taps; const int ci = (int)(r % Ci), co = (int)(r / Ci);
        const long long j = ((long long)t * Co + co) * Ci + ci;
        g[i] = packed[j];
        packed[j] = 0.f;
    }
}
__global__ void k_fill_f32(float* p, float v, long long n) {
    pdl_entry();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = v;
}
// small fp32 elementwise helpers for the timestep-embedding MLP backward: dx = dy * silu'(x)
__global__ void k_silu_bwd_f32(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx, long long n) {
    pdl_entry();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) dx[i] = dy[i] * silu_grad_f(x[i]);
}

}  // namespace ddpm
