// Row-wise softmax cross-entropy for large vocabularies (V = 151936 for Qwen3), forward and gradient.
//
// Replaces the arithmetic of eager_cross_entropy / fixed_cross_entropy
// (veomni/ops/kernels/cross_entropy/eager.py:23-38) and of the liger fused-linear-cross-entropy element kernel
// (veomni/ops/kernels/cross_entropy/liger.py) on the logits of one row chunk:
//     loss_row = logsumexp(x) - x[label]                 (0 when label == ignore_index)
//     grad     = (softmax(x) - onehot(label)) * scale    (0 for ignored rows)
//
// HBM-bound. One CTA of 1024 threads owns a row: pass 1 streams the row once and keeps a per-thread online
// (max, sum) pair — one exp2 per element plus one per 8-element vector for the running rescale; pass 2 re-reads
// the row and writes the gradient over it (in place when grad == logits). With 2 CTAs per SM, 296 rows of 304 KB
// (bf16) are in flight = 90 MB, which the 126 MB L2 holds, so the second read is an L2 hit and DRAM sees the
// algorithmic minimum: one read and one write of the chunk. fp32 rows (608 KB) spill L2 and pay a second DRAM read.
#include <cstdio>

#include "common.cuh"

namespace vb {

constexpr int CE_THREADS = 1024;
constexpr float kLog2eCe = 1.4426950408889634f;
constexpr float kLn2Ce = 0.6931471805599453f;

template <typename T>
struct CeVec;
template <>
struct CeVec<__nv_bfloat16> {
    static constexpr int N = 8;
    __device__ static void load(const __nv_bfloat16* p, float (&v)[8]) {
        const uint4 u = *reinterpret_cast<const uint4*>(p);
        float2 a = bf2_to_f2(u.x), b = bf2_to_f2(u.y), c = bf2_to_f2(u.z), d = bf2_to_f2(u.w);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
    }
    __device__ static void store(__nv_bfloat16* p, const float (&v)[8]) {
        uint4 u;
        u.x = f2_to_bf2(v[0], v[1]); u.y = f2_to_bf2(v[2], v[3]); u.z = f2_to_bf2(v[4], v[5]); u.w = f2_to_bf2(v[6], v[7]);
        *reinterpret_cast<uint4*>(p) = u;
    }
};
template <>
struct CeVec<float> {
    static constexpr int N = 4;
    __device__ static void load(const float* p, float (&v)[4]) {
        const float4 u = *reinterpret_cast<const float4*>(p);
        v[0] = u.x; v[1] = u.y; v[2] = u.z; v[3] = u.w;
    }
    __device__ static void store(float* p, const float (&v)[4]) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
};

__device__ __forceinline__ float ce_to_float(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float ce_to_float(float x) { return x; }
__device__ __forceinline__ void ce_from_float(__nv_bfloat16* p, float x) { *p = __float2bfloat16_rn(x); }
__device__ __forceinline__ void ce_from_float(float* p, float x) { *p = x; }

// x: [rows, vocab] with row stride `stride` (elements). `lse` is an output when lse_given == 0 and an input
// otherwise (backward-only call). `grad` may be null (forward only) or alias `x`.
template <typename T>
__global__ void __launch_bounds__(CE_THREADS, 2)
cross_entropy_kernel(const T* __restrict__ x, int64_t stride, int64_t vocab, const int64_t* __restrict__ labels,
                     int64_t ignore_index, float* __restrict__ loss_rows, float* __restrict__ lse, int lse_given,
                     T* grad, int64_t grad_stride, float scale_host, const float* __restrict__ scale_dev,
                     const float* __restrict__ upstream) {
    constexpr int N = CeVec<T>::N;
    __shared__ float red_m[32], red_s[32];
    __shared__ float row_lse2;
    const int64_t row = blockIdx.x;
    const T* xr = x + row * stride;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t label = labels[row];
    const bool ignored = label == ignore_index;
    const bool in_range = label >= 0 && label < vocab;  // anything else (and not ignore_index) yields a NaN loss
    // rows need not be 16-byte aligned relative to the vector width if stride % N != 0: peel a scalar head
    const int64_t mis = (reinterpret_cast<uintptr_t>(xr) & 15) / sizeof(T);
    const int64_t head = mis ? ((vocab < (int64_t)(N - mis)) ? vocab : (int64_t)(N - mis)) : 0;  // N == 16 / sizeof(T)
    const int64_t nvec = (vocab - head) / N;
    const int64_t tail0 = head + nvec * N;

    float lse2;  // log2-domain logsumexp: lse2 = log2(sum exp(x)) = max*log2e + log2(sum exp2((x - max)*log2e))
    if (!lse_given) {
        float m = -INFINITY, s = 0.f;  // running max (already multiplied by log2e) and sum of exp2(x*log2e - m)
        auto fold = [&](float v) {
            const float y = v * kLog2eCe;
            if (y == -INFINITY) return;
            if (y > m) {
                s = s * exp2f(m - y) + 1.f;
                m = y;
            } else {
                s += exp2f(y - m);
            }
        };
        for (int64_t i = tid; i < head; i += CE_THREADS) fold(ce_to_float(xr[i]));
        for (int64_t i = tail0 + tid; i < vocab; i += CE_THREADS) fold(ce_to_float(xr[i]));
        auto fold_vec = [&](const float (&v)[N]) {
            float vm = v[0];
#pragma unroll
            for (int e = 1; e < N; ++e) vm = fmaxf(vm, v[e]);
            vm *= kLog2eCe;
            if (vm > m) {  // one rescale per vector instead of per element
                s *= exp2f(m - vm);
                m = vm;
            }
            if (m != -INFINITY) {
#pragma unroll
                for (int e = 0; e < N; ++e) s += exp2f(fmaf(v[e], kLog2eCe, -m));
            }
        };
        int64_t j = tid;
        for (; j + CE_THREADS < nvec; j += 2 * CE_THREADS) {  // two 16-byte loads in flight per thread
            float v0[N], v1[N];
            CeVec<T>::load(xr + head + j * N, v0);
            CeVec<T>::load(xr + head + (j + CE_THREADS) * N, v1);
            fold_vec(v0);
            fold_vec(v1);
        }
        if (j < nvec) {
            float v0[N];
            CeVec<T>::load(xr + head + j * N, v0);
            fold_vec(v0);
        }
        // block reduction of (m, s) pairs, fixed order -> deterministic
        float wm = warp_max(m);
        float ws = (m == -INFINITY) ? 0.f : s * exp2f(m - wm);
        ws = warp_sum(ws);
        if (lane == 0) {
            red_m[warp] = wm;
            red_s[warp] = ws;
        }
        __syncthreads();
        if (warp == 0) {
            const float pm = red_m[lane], ps = red_s[lane];  // CE_THREADS / 32 == 32 warps
            const float bm = warp_max(pm);
            float bs = (pm == -INFINITY) ? 0.f : ps * exp2f(pm - bm);
            bs = warp_sum(bs);
            if (lane == 0) {
                const float l2 = bm + log2f(bs);
                row_lse2 = l2;
                const float l = l2 * kLn2Ce;
                if (lse) lse[row] = l;
                if (loss_rows) loss_rows[row] = ignored ? 0.f : (in_range ? l - ce_to_float(xr[label]) : NAN);
            }
        }
        __syncthreads();
        lse2 = row_lse2;
    } else {
        lse2 = lse[row] * kLog2eCe;
    }
    if (grad == nullptr) return;

    float scale = scale_host;
    if (scale_dev) scale *= *scale_dev;
    if (upstream) scale *= *upstream;
    T* gr = grad + row * grad_stride;
    if (ignored) {
        float z[N];
#pragma unroll
        for (int e = 0; e < N; ++e) z[e] = 0.f;
        for (int64_t i = tid; i < head; i += CE_THREADS) ce_from_float(gr + i, 0.f);
        for (int64_t i = tail0 + tid; i < vocab; i += CE_THREADS) ce_from_float(gr + i, 0.f);
        for (int64_t j = tid; j < nvec; j += CE_THREADS) CeVec<T>::store(gr + head + j * N, z);
        return;
    }
    for (int64_t i = tid; i < head; i += CE_THREADS) {
        const float p = exp2f(fmaf(ce_to_float(xr[i]), kLog2eCe, -lse2));
        ce_from_float(gr + i, (p - (i == label ? 1.f : 0.f)) * scale);
    }
    for (int64_t i = tail0 + tid; i < vocab; i += CE_THREADS) {
        const float p = exp2f(fmaf(ce_to_float(xr[i]), kLog2eCe, -lse2));
        ce_from_float(gr + i, (p - (i == label ? 1.f : 0.f)) * scale);
    }
    const int64_t lj = (in_range && label >= head && label < tail0) ? (label - head) / N : -1;
    const int le = (int)((label - head) % N);
    auto grad_vec = [&](int64_t j, float (&v)[N]) {
#pragma unroll
        for (int e = 0; e < N; ++e) v[e] = exp2f(fmaf(v[e], kLog2eCe, -lse2));
        if (j == lj) {
#pragma unroll
            for (int e = 0; e < N; ++e)
                if (e == le) v[e] -= 1.f;
        }
#pragma unroll
        for (int e = 0; e < N; ++e) v[e] *= scale;
        CeVec<T>::store(gr + head + j * N, v);
    };
    int64_t j = tid;
    for (; j + CE_THREADS < nvec; j += 2 * CE_THREADS) {
        float v0[N], v1[N];
        CeVec<T>::load(xr + head + j * N, v0);
        CeVec<T>::load(xr + head + (j + CE_THREADS) * N, v1);
        grad_vec(j, v0);
        grad_vec(j + CE_THREADS, v1);
    }
    if (j < nvec) {
        float v0[N];
        CeVec<T>::load(xr + head + j * N, v0);
        grad_vec(j, v0);
    }
}

// 1 / count(labels != ignore_index) as a device scalar (0 valid labels -> 0, so every gradient is 0 and the
// loss sum times it is 0, matching "mean over nothing" being masked out by the callers' token weighting).
__global__ void ce_valid_recip_kernel(const int64_t* __restrict__ labels, int64_t n, int64_t ignore_index,
                                      float* __restrict__ out) {
    __shared__ int red[32];
    int c = 0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) c += labels[i] != ignore_index;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x < 32) {
        c = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (threadIdx.x == 0) {
            out[0] = c > 0 ? 1.f / (float)c : 0.f;
            out[1] = (float)c;
        }
    }
}

// ---- per-token log-probs, entropy and top-k forward-KL distillation -------------------------------------------
// Replaces the arithmetic of _ChunkedLinearLogProbs and _ChunkedLinearTopkDistill
// (veomni/ops/kernels/cross_entropy/chunk_logprobs.py:126-268, chunk_topk_distill.py:79-326) on one logits chunk.
// The reference divides the logits by the temperature in their own dtype and then upcasts
// (chunk_logprobs.py:173-176), so both kernels work on x = round_T(x_in / temperature) in fp32:
//     lse = logsumexp(x),  logp = x[label] - lse,  entropy = lse - sum(softmax(x) * x)          (0 at ignored rows)
//     top-k (K > 0): slp_k = x[id_k] - lse, student_mass = sum_k exp(slp_k), teacher_mass = sum_k exp(tlp_k),
//                    distill = sum_k exp(tlp'_k) * (tlp'_k - slp'_k), ' = clamp_min(clamp) when a clamp is given
// Same streaming structure as cross_entropy_kernel: one 1024-thread CTA per row, the forward keeps an online
// (max, sum e, sum e*x) triple per thread and reduces it in a fixed order; the backward re-reads the row once and
// writes dlogits over it. The top-k ids are read after the row reduction, when the row is in L2.

constexpr int TL_MAX_K = CE_THREADS;  // one top-k entry per thread
constexpr int TL_HIT_WORDS = 512;     // 16384-bit filter over vector indices: a set bit means "scan the top-k list"

template <typename T>
__device__ __forceinline__ float tl_round(float v);
template <>
__device__ __forceinline__ float tl_round<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
template <>
__device__ __forceinline__ float tl_round<float>(float v) { return v; }

// x_in / temperature rounded to the logits dtype, as the reference's division in that dtype; __fdiv_rn because the
// library builds with --use_fast_math, whose '/' is not correctly rounded
template <typename T>
__device__ __forceinline__ float tl_temper(float v, float temperature) {
    return temperature == 1.f ? v : tl_round<T>(__fdiv_rn(v, temperature));
}

__device__ __forceinline__ float tl_load_tlp(const void* tlp, int tlp_dtype, int64_t i) {
    return tlp_dtype == 0 ? __bfloat162float(static_cast<const __nv_bfloat16*>(tlp)[i]) : static_cast<const float*>(tlp)[i];
}

// 16-byte vector loads kept packed until use: two in flight per thread cost 8 registers instead of 2 * N
template <typename T>
__device__ __forceinline__ uint4 tl_load_raw(const T* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void tl_unpack(const uint4& u, float (&v)[8]) { unpack8(u, v); }
__device__ __forceinline__ void tl_unpack(const uint4& u, float (&v)[4]) {
    v[0] = __uint_as_float(u.x); v[1] = __uint_as_float(u.y); v[2] = __uint_as_float(u.z); v[3] = __uint_as_float(u.w);
}

// clamp_min that keeps NaN, as torch.clamp_min does
__device__ __forceinline__ float tl_clamp(float v, int has_clamp, float lo) { return (has_clamp && v < lo) ? lo : v; }

template <typename T>
__global__ void __launch_bounds__(CE_THREADS, 2)
token_stats_kernel(const T* __restrict__ x, int64_t stride, int64_t vocab, const int64_t* __restrict__ labels,
                   int64_t ignore_index, float temperature, float* __restrict__ lse, float* __restrict__ logp,
                   float* __restrict__ entropy, int k, const int64_t* __restrict__ ids, const void* __restrict__ tlp,
                   int tlp_dtype, int has_clamp, float clamp, float* __restrict__ distill,
                   float* __restrict__ student_mass, float* __restrict__ teacher_mass) {
    constexpr int N = CeVec<T>::N;
    __shared__ float red_a[32], red_b[32], red_c[32];
    __shared__ float row_lse;
    const int64_t row = blockIdx.x;
    const T* xr = x + row * stride;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t label = labels[row];
    const bool ignored = label == ignore_index;
    const bool in_range = label >= 0 && label < vocab;
    const int64_t mis = (reinterpret_cast<uintptr_t>(xr) & 15) / sizeof(T);
    const int64_t head = mis ? ((vocab < (int64_t)(N - mis)) ? vocab : (int64_t)(N - mis)) : 0;
    const int64_t nvec = (vocab - head) / N;
    const int64_t tail0 = head + nvec * N;

    // m: running max times log2e; s = sum exp2(x*log2e - m); t = sum exp2(x*log2e - m) * x
    float m = -INFINITY, s = 0.f, t = 0.f;
    auto fold = [&](float v) {
        v = tl_temper<T>(v, temperature);
        const float y = v * kLog2eCe;
        if (y == -INFINITY) return;
        if (y > m) {
            const float c = exp2f(m - y);
            s = s * c + 1.f;
            t = fmaf(t, c, v);
            m = y;
        } else {
            const float e = exp2f(y - m);
            s += e;
            t = fmaf(e, v, t);
        }
    };
    for (int64_t i = tid; i < head; i += CE_THREADS) fold(ce_to_float(xr[i]));
    for (int64_t i = tail0 + tid; i < vocab; i += CE_THREADS) fold(ce_to_float(xr[i]));
    auto fold_vec = [&](float (&v)[N]) {
        if (temperature != 1.f) {
#pragma unroll
            for (int e = 0; e < N; ++e) v[e] = tl_temper<T>(v[e], temperature);
        }
        float vm = v[0];
#pragma unroll
        for (int e = 1; e < N; ++e) vm = fmaxf(vm, v[e]);
        vm *= kLog2eCe;
        if (vm > m) {
            const float c = exp2f(m - vm);
            s *= c;
            t *= c;
            m = vm;
        }
        if (m != -INFINITY) {
#pragma unroll
            for (int e = 0; e < N; ++e) {
                const float p = exp2f(fmaf(v[e], kLog2eCe, -m));
                s += p;
                t = fmaf(p, v[e], t);
            }
        }
    };
    const uint4* xv = reinterpret_cast<const uint4*>(xr + head);
    const int nv = (int)nvec;  // vocab < 2^31 (checked at the ABI): 32-bit vector indices keep the loop in registers
    int j = tid;
    for (; j + CE_THREADS < nv; j += 2 * CE_THREADS) {
        const uint4 r0 = xv[j], r1 = xv[j + CE_THREADS];
        float v[N];
        tl_unpack(r0, v);
        fold_vec(v);
        tl_unpack(r1, v);
        fold_vec(v);
    }
    if (j < nv) {
        float v[N];
        tl_unpack(xv[j], v);
        fold_vec(v);
    }
    // block reduction of the triples, fixed order -> deterministic
    const float wm = warp_max(m);
    const float wc = (m == -INFINITY) ? 0.f : exp2f(m - wm);
    const float ws = warp_sum(s * wc), wt = warp_sum(t * wc);
    if (lane == 0) {
        red_a[warp] = wm;
        red_b[warp] = ws;
        red_c[warp] = wt;
    }
    __syncthreads();
    if (warp == 0) {
        const float pm = red_a[lane];
        const float bm = warp_max(pm);
        const float pc = (pm == -INFINITY) ? 0.f : exp2f(pm - bm);
        const float bs = warp_sum(red_b[lane] * pc), bt = warp_sum(red_c[lane] * pc);
        if (lane == 0) {
            const float l = (bm + log2f(bs)) * kLn2Ce;
            row_lse = l;
            if (lse) lse[row] = l;
            logp[row] = ignored ? 0.f : (in_range ? tl_temper<T>(ce_to_float(xr[label]), temperature) - l : NAN);
            entropy[row] = ignored ? 0.f : l - __fdiv_rn(bt, bs);
        }
    }
    if (k == 0) return;
    if (ignored) {
        if (tid == 0) distill[row] = student_mass[row] = teacher_mass[row] = 0.f;
        return;
    }
    __syncthreads();  // row_lse visible; warp 0 is done reading red_*
    float sm = 0.f, tm = 0.f, d = 0.f;
    if (tid < k) {
        const int64_t id = ids[row * k + tid];
        const float tl = tl_load_tlp(tlp, tlp_dtype, row * k + tid);
        const float sl = (id >= 0 && id < vocab) ? tl_temper<T>(ce_to_float(xr[id]), temperature) - row_lse : NAN;
        sm = expf(sl);  // both masses before the clamp (chunk_topk_distill.py:170-171)
        tm = expf(tl);
        const float tlc = tl_clamp(tl, has_clamp, clamp), slc = tl_clamp(sl, has_clamp, clamp);
        d = expf(tlc) * (tlc - slc);
    }
    sm = warp_sum(sm);
    tm = warp_sum(tm);
    d = warp_sum(d);
    if (lane == 0) {
        red_a[warp] = sm;
        red_b[warp] = tm;
        red_c[warp] = d;
    }
    __syncthreads();
    if (warp == 0) {
        sm = warp_sum(red_a[lane]);
        tm = warp_sum(red_b[lane]);
        d = warp_sum(red_c[lane]);
        if (lane == 0) {
            student_mass[row] = sm;
            teacher_mass[row] = tm;
            distill[row] = d;
        }
    }
}

// dlogits of  sum_r dlogp_r * logp_r + dent_r * entropy_r + ddist_r * distill_r  (each upstream optional = 0):
//     g_v = dlp (d(v=y) - p_v) - dent p_v (x_v - lse + H) + ddist (teacher_mass_eff p_v - pt_sparse[v])
// (chunk_logprobs.py:230-249, chunk_topk_distill.py:266-306), pt_sparse[v] = sum over k with id_k == v of
// exp(tlp'_k), each k gated by slp_k >= clamp when a clamp is given; teacher_mass_eff = sum of the same terms.
// Output rounding as chunk_logprobs.py:251-258: g to the logits dtype, then / temperature in that dtype.
// The top-k (id, coefficient) pairs sit in shared memory with a bit filter over the vectors they fall in, so only
// vectors whose bit is set scan the list; the sparse term is added in fp32 before the single rounding.
template <typename T>
__global__ void __launch_bounds__(CE_THREADS, 2)
token_grad_kernel(const T* x, int64_t stride, int64_t vocab, const int64_t* __restrict__ labels, int64_t ignore_index,
                  float temperature, const float* __restrict__ lse, const float* __restrict__ entropy,
                  const float* __restrict__ dlogp, const float* __restrict__ dent, const float* __restrict__ ddist,
                  int k, const int64_t* __restrict__ ids, const void* __restrict__ tlp, int tlp_dtype, int has_clamp,
                  float clamp, T* grad, int64_t grad_stride) {
    constexpr int N = CeVec<T>::N;
    __shared__ int s_id[TL_MAX_K];
    __shared__ float s_coef[TL_MAX_K];
    __shared__ uint32_t s_hit[TL_HIT_WORDS];
    __shared__ float red[33];
    __shared__ float s_alp, s_akl;  // only the label's vector and the filtered vectors need these: kept out of registers
    __shared__ int s_k;
    const int64_t row = blockIdx.x;
    const T* xr = x + row * stride;
    T* gr = grad + row * grad_stride;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t label = labels[row];
    const bool ignored = label == ignore_index;
    const bool in_range = label >= 0 && label < vocab;
    const int64_t mis = (reinterpret_cast<uintptr_t>(xr) & 15) / sizeof(T);
    const int64_t head = mis ? ((vocab < (int64_t)(N - mis)) ? vocab : (int64_t)(N - mis)) : 0;
    const int64_t nvec = (vocab - head) / N;
    const int64_t tail0 = head + nvec * N;
    if (ignored) {
        float z[N];
#pragma unroll
        for (int e = 0; e < N; ++e) z[e] = 0.f;
        for (int64_t i = tid; i < head; i += CE_THREADS) ce_from_float(gr + i, 0.f);
        for (int64_t i = tail0 + tid; i < vocab; i += CE_THREADS) ce_from_float(gr + i, 0.f);
        for (int64_t jj = tid; jj < nvec; jj += CE_THREADS) CeVec<T>::store(gr + head + jj * N, z);
        return;
    }
    const float a_lp = dlogp ? dlogp[row] : 0.f;
    const float a_ent = dent ? dent[row] : 0.f;
    const float a_kl = (ddist && k > 0) ? ddist[row] : 0.f;
    const float l = lse[row];
    const float lse2 = l * kLog2eCe;
    const float hl = a_ent != 0.f ? entropy[row] - l : 0.f;  // x + hl = log p + H
    const bool topk = a_kl != 0.f;                           // row-uniform
    float tmass = 0.f;
    if (topk) {
        for (int i = tid; i < TL_HIT_WORDS; i += CE_THREADS) s_hit[i] = 0u;
        float coef = 0.f;
        int64_t id = -1;
        if (tid < k) {
            id = ids[row * k + tid];
            if (id >= 0 && id < vocab) {
                coef = expf(tl_clamp(tl_load_tlp(tlp, tlp_dtype, row * k + tid), has_clamp, clamp));
                if (has_clamp && !(tl_temper<T>(ce_to_float(xr[id]), temperature) - l >= clamp)) coef = 0.f;
            } else {
                id = -1;  // outside the vocabulary: no gradient (the forward reports NaN for the row)
            }
            s_id[tid] = id >= 0 ? (int)(id - head) : INT_MIN;  // relative to the first vector, as the filter
            s_coef[tid] = coef;
        }
        __syncthreads();  // s_hit cleared; every read of the row above precedes the first write below
        if (id >= head && id < tail0) {  // scalar head / tail elements always scan the list
            const int64_t jv = (id - head) / N;
            atomicOr(&s_hit[(jv >> 5) & (TL_HIT_WORDS - 1)], 1u << (jv & 31));
        }
        const float wsum = warp_sum(coef);
        if (lane == 0) red[warp] = wsum;
        __syncthreads();
        if (warp == 0) {
            const float b = warp_sum(red[lane]);
            if (lane == 0) red[32] = b;
        }
        __syncthreads();
        tmass = red[32];
    }
    if (tid == 0) {
        s_alp = a_lp;
        s_akl = a_kl;
        s_k = k;
    }
    __syncthreads();
    auto sparse = [&](int rel) {  // pt_sparse at vocabulary index head + rel; duplicate ids add up in k order
        float acc = 0.f;
        const int kk = s_k;
        for (int i = 0; i < kk; ++i)
            if (s_id[i] == rel) acc += s_coef[i];
        return acc;
    };
    const float c1 = fmaf(-a_ent, hl, fmaf(a_kl, tmass, -a_lp));  // g_v = p_v (c1 - dent x_v) + sparse and label terms
    auto finish = [&](float g) {
        const float r = tl_round<T>(g);
        return temperature == 1.f ? r : __fdiv_rn(r, temperature);
    };
    const int ll = (in_range && label >= head && label < tail0) ? (int)(label - head) : -1;
    // g_v before the final rounding; e is the element's position in its vector, le the label's (any value if absent)
    auto elem = [&](float xin, int e, int le) {
        const float xv = tl_temper<T>(xin, temperature);
        const float p = exp2f(fmaf(xv, kLog2eCe, -lse2));
        float g = p * fmaf(-a_ent, xv, c1);
        if (e == le) g += s_alp;
        return g;
    };
    for (int64_t i = tid; i < head; i += CE_THREADS)  // scalar head and tail: the label test is i == label
        ce_from_float(gr + i, finish(elem(ce_to_float(xr[i]), 0, i == label ? 0 : 1) - (topk ? a_kl * sparse((int)(i - head)) : 0.f)));
    for (int64_t i = tail0 + tid; i < vocab; i += CE_THREADS)
        ce_from_float(gr + i, finish(elem(ce_to_float(xr[i]), 0, i == label ? 0 : 1) - (topk ? a_kl * sparse((int)(i - head)) : 0.f)));
    // one 16-byte vector of logits -> its gradient, unpacked and repacked element by element so that two vectors in
    // flight per thread fit the 32 registers of 2 CTAs per SM
    auto grad_raw = [&](const uint4& r, int jv) {
        const int le = ll - jv * N;
        uint4 o;
        if constexpr (N == 8) {
            float2 f = bf2_to_f2(r.x);
            o.x = f2_to_bf2(finish(elem(f.x, 0, le)), finish(elem(f.y, 1, le)));
            f = bf2_to_f2(r.y);
            o.y = f2_to_bf2(finish(elem(f.x, 2, le)), finish(elem(f.y, 3, le)));
            f = bf2_to_f2(r.z);
            o.z = f2_to_bf2(finish(elem(f.x, 4, le)), finish(elem(f.y, 5, le)));
            f = bf2_to_f2(r.w);
            o.w = f2_to_bf2(finish(elem(f.x, 6, le)), finish(elem(f.y, 7, le)));
        } else {
            o.x = __float_as_uint(finish(elem(__uint_as_float(r.x), 0, le)));
            o.y = __float_as_uint(finish(elem(__uint_as_float(r.y), 1, le)));
            o.z = __float_as_uint(finish(elem(__uint_as_float(r.z), 2, le)));
            o.w = __float_as_uint(finish(elem(__uint_as_float(r.w), 3, le)));
        }
        return o;
    };
    auto filtered = [&](int jv) { return topk && ((s_hit[(jv >> 5) & (TL_HIT_WORDS - 1)] >> (jv & 31)) & 1u); };
    // vectors the filter marks are left for the second loop, which adds the sparse term; the list scan stays out of
    // the streaming loop
    const uint4* xv = reinterpret_cast<const uint4*>(xr + head);
    uint4* gv = reinterpret_cast<uint4*>(gr + head);
    const int nv = (int)nvec;
    int j = tid;
    for (; j + CE_THREADS < nv; j += 2 * CE_THREADS) {
        const uint4 r0 = xv[j], r1 = xv[j + CE_THREADS];
        if (!filtered(j)) gv[j] = grad_raw(r0, j);
        if (!filtered(j + CE_THREADS)) gv[j + CE_THREADS] = grad_raw(r1, j + CE_THREADS);
    }
    if (j < nv && !filtered(j)) gv[j] = grad_raw(xv[j], j);
    if (!topk) return;
    const float ak = s_akl;
    for (j = tid; j < nv; j += CE_THREADS) {  // this thread's own vectors: their logits are still unwritten
        if (!filtered(j)) continue;
        float v[N];
        tl_unpack(xv[j], v);
        const int le = ll - j * N;
#pragma unroll
        for (int e = 0; e < N; ++e) v[e] = finish(elem(v[e], e, le) - ak * sparse(j * N + e));
        CeVec<T>::store(reinterpret_cast<T*>(gv + j), v);
    }
}

}  // namespace vb

using namespace vb;

extern "C" int vb200_cross_entropy(const void* logits, int32_t dtype, int64_t rows, int64_t vocab, int64_t row_stride,
                                   const int64_t* labels, int64_t ignore_index, float* loss_rows, float* lse,
                                   int32_t lse_given, void* grad, int64_t grad_stride, float scale,
                                   const float* scale_dev, const float* upstream, void* stream) {
    if (rows == 0) return VB200_OK;
    if (rows < 0 || vocab <= 0 || !logits || !labels) return vb200_set_error(VB200_EINVAL, "cross_entropy: bad arguments");
    if (dtype != 0 && dtype != 1) return vb200_set_error(VB200_EINVAL, "cross_entropy: dtype must be 0 (bf16) or 1 (f32)");
    if (lse_given && !lse) return vb200_set_error(VB200_EINVAL, "cross_entropy: lse_given without lse");
    if (!lse_given && !grad && !loss_rows && !lse) return vb200_set_error(VB200_EINVAL, "cross_entropy: nothing to compute");
    const size_t esz = dtype == 0 ? 2 : 4;
    // the gradient row must share the logits row's 16-byte phase so both use the same head/vector split
    if (grad && (((uintptr_t)grad ^ (uintptr_t)logits) & 15) != 0)
        return vb200_set_error(VB200_EINVAL, "cross_entropy: grad and logits must have the same 16-byte alignment phase");
    if (grad && ((grad_stride - row_stride) * (int64_t)esz) % 16 != 0)
        return vb200_set_error(VB200_EINVAL, "cross_entropy: grad/logits row strides must differ by a multiple of 16 bytes");
    if (rows > 0x7fffffffLL) return vb200_set_error(VB200_EINVAL, "cross_entropy: too many rows");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == 0)
        cross_entropy_kernel<__nv_bfloat16><<<(unsigned)rows, CE_THREADS, 0, s>>>(
            (const __nv_bfloat16*)logits, row_stride, vocab, labels, ignore_index, loss_rows, lse, lse_given,
            (__nv_bfloat16*)grad, grad_stride, scale, scale_dev, upstream);
    else
        cross_entropy_kernel<float><<<(unsigned)rows, CE_THREADS, 0, s>>>(
            (const float*)logits, row_stride, vocab, labels, ignore_index, loss_rows, lse, lse_given, (float*)grad,
            grad_stride, scale, scale_dev, upstream);
    vb200_count_launch(1);
    VB_HOST_CHECK_LAUNCH();
    return VB200_OK;
}

// argument checks shared by the two token-statistics entry points
static int tl_check(const char* what, const void* logits, int32_t dtype, int64_t rows, int64_t vocab,
                    const int64_t* labels, float temperature, int32_t k, const int64_t* ids, const void* tlp,
                    int32_t tlp_dtype) {
    char msg[160];
    if (rows < 0 || vocab <= 0 || !logits || !labels) {
        snprintf(msg, sizeof msg, "%s: bad arguments", what);
        return vb200_set_error(VB200_EINVAL, msg);
    }
    if (dtype != 0 && dtype != 1) {
        snprintf(msg, sizeof msg, "%s: dtype must be 0 (bf16) or 1 (f32)", what);
        return vb200_set_error(VB200_EINVAL, msg);
    }
    if (!(temperature > 0.f) || isinf(temperature)) {
        snprintf(msg, sizeof msg, "%s: temperature must be a positive finite number", what);
        return vb200_set_error(VB200_EINVAL, msg);
    }
    if (k < 0 || k > TL_MAX_K) {
        snprintf(msg, sizeof msg, "%s: top-k width K = %d is outside [0, %d]", what, (int)k, TL_MAX_K);
        return vb200_set_error(VB200_EINVAL, msg);
    }
    if (k > 0 && (!ids || !tlp || (tlp_dtype != 0 && tlp_dtype != 1))) {
        snprintf(msg, sizeof msg, "%s: top-k needs ids and bf16/f32 teacher log-probs", what);
        return vb200_set_error(VB200_EINVAL, msg);
    }
    if (rows > 0x7fffffffLL || vocab > 0x7fffffffLL) {
        snprintf(msg, sizeof msg, "%s: rows and vocab must be below 2^31", what);
        return vb200_set_error(VB200_EINVAL, msg);
    }
    return VB200_OK;
}

extern "C" int vb200_token_logprobs(const void* logits, int32_t dtype, int64_t rows, int64_t vocab, int64_t row_stride,
                                    const int64_t* labels, int64_t ignore_index, float temperature, float* lse,
                                    float* logp, float* entropy, int32_t k, const int64_t* topk_ids,
                                    const void* topk_logp, int32_t topk_dtype, int32_t has_clamp, float clamp,
                                    float* distill, float* student_mass, float* teacher_mass, void* stream) {
    if (rows == 0) return VB200_OK;
    int rc = tl_check("token_logprobs", logits, dtype, rows, vocab, labels, temperature, k, topk_ids, topk_logp, topk_dtype);
    if (rc != VB200_OK) return rc;
    if (!logp || !entropy) return vb200_set_error(VB200_EINVAL, "token_logprobs: logp and entropy are required");
    if (k > 0 && (!distill || !student_mass || !teacher_mass))
        return vb200_set_error(VB200_EINVAL, "token_logprobs: top-k needs distill, student_mass and teacher_mass");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == 0)
        token_stats_kernel<__nv_bfloat16><<<(unsigned)rows, CE_THREADS, 0, s>>>(
            (const __nv_bfloat16*)logits, row_stride, vocab, labels, ignore_index, temperature, lse, logp, entropy, k,
            topk_ids, topk_logp, topk_dtype, has_clamp, clamp, distill, student_mass, teacher_mass);
    else
        token_stats_kernel<float><<<(unsigned)rows, CE_THREADS, 0, s>>>(
            (const float*)logits, row_stride, vocab, labels, ignore_index, temperature, lse, logp, entropy, k,
            topk_ids, topk_logp, topk_dtype, has_clamp, clamp, distill, student_mass, teacher_mass);
    vb200_count_launch(1);
    VB_HOST_CHECK_LAUNCH();
    return VB200_OK;
}

extern "C" int vb200_token_logprobs_bwd(const void* logits, int32_t dtype, int64_t rows, int64_t vocab,
                                        int64_t row_stride, const int64_t* labels, int64_t ignore_index,
                                        float temperature, const float* lse, const float* entropy, const float* dlogp,
                                        const float* dentropy, const float* ddistill, int32_t k, const int64_t* topk_ids,
                                        const void* topk_logp, int32_t topk_dtype, int32_t has_clamp, float clamp,
                                        void* grad, int64_t grad_stride, void* stream) {
    if (rows == 0) return VB200_OK;
    int rc = tl_check("token_logprobs_bwd", logits, dtype, rows, vocab, labels, temperature, k, topk_ids, topk_logp,
                      topk_dtype);
    if (rc != VB200_OK) return rc;
    if (!lse || !grad) return vb200_set_error(VB200_EINVAL, "token_logprobs_bwd: lse and grad are required");
    if (dentropy && !entropy) return vb200_set_error(VB200_EINVAL, "token_logprobs_bwd: dentropy needs the saved entropy");
    const size_t esz = dtype == 0 ? 2 : 4;
    if ((((uintptr_t)grad ^ (uintptr_t)logits) & 15) != 0)
        return vb200_set_error(VB200_EINVAL, "token_logprobs_bwd: grad and logits must have the same 16-byte alignment phase");
    if (((grad_stride - row_stride) * (int64_t)esz) % 16 != 0)
        return vb200_set_error(VB200_EINVAL, "token_logprobs_bwd: grad/logits row strides must differ by a multiple of 16 bytes");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == 0)
        token_grad_kernel<__nv_bfloat16><<<(unsigned)rows, CE_THREADS, 0, s>>>(
            (const __nv_bfloat16*)logits, row_stride, vocab, labels, ignore_index, temperature, lse, entropy, dlogp,
            dentropy, ddistill, k, topk_ids, topk_logp, topk_dtype, has_clamp, clamp, (__nv_bfloat16*)grad, grad_stride);
    else
        token_grad_kernel<float><<<(unsigned)rows, CE_THREADS, 0, s>>>(
            (const float*)logits, row_stride, vocab, labels, ignore_index, temperature, lse, entropy, dlogp, dentropy,
            ddistill, k, topk_ids, topk_logp, topk_dtype, has_clamp, clamp, (float*)grad, grad_stride);
    vb200_count_launch(1);
    VB_HOST_CHECK_LAUNCH();
    return VB200_OK;
}

extern "C" int vb200_count_valid_labels(const int64_t* labels, int64_t n, int64_t ignore_index, float* out2,
                                        void* stream) {
    if (!labels || !out2 || n < 0) return vb200_set_error(VB200_EINVAL, "count_valid_labels: bad arguments");
    ce_valid_recip_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(labels, n, ignore_index, out2);
    vb200_count_launch(1);
    VB_HOST_CHECK_LAUNCH();
    return VB200_OK;
}
